// encrypt.cu -- batched fresh encryptions on the GPU (SURVEY.md 8f rank 2: the step before the
// hot path).  The reference encrypts one bit at a time on the host, O(N*D) per bit, drawing
// from glibc rand() (src/SecretKey.cpp:35-80); this kernel builds n fresh blocks at once with
// the same construction and a counter-based generator:
//
//   Enc(1): ones at the secret positions, random bits elsewhere;
//   Enc(0): a random secret position h; random bits everywhere else; the bit at h is forced to 0
//           if every other secret position came out 1, otherwise it stays random.
//
// Randomness is Philox-4x32-10 keyed by the caller's seed with counter (block, unit), so a block's
// words do not depend on how the batch is split over launches or GPUs (oracle/csgn_oracle.c holds
// the CPU restatement the tests compare against, bit for bit).  Three forms: short even blocks
// (a warp builds 32 blocks, coalesced), long blocks (a warp builds one block), and a lane-per-block
// form for odd L.  The work is ten Philox rounds per 16 bytes.
//
// Each form reads its plaintext bits from one of two sources: a byte per block (csgn_encrypt_batch), or the bit planes
// of n integers laid one after another (csgn_encrypt_uint: block i encrypts bit i / n of values[i % n]).
#include "kernels.cuh"
#include "launch.cuh"

#include <algorithm>

namespace csgn {
namespace {

__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                               uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

constexpr uint32_t kTag = 0x43534731u;

// Bit i of the planes of n integers: plane j = i / n (LSB first), element k = i - j*n.  The quotient comes from the
// host's magic = floor((2^64 - 1) / n): umulhi(i, magic) is floor(i / n) or one less, and one step corrects it.
__device__ __forceinline__ bool plane_bit(const UIntPlanes &p, uint64_t i) {
    uint64_t j = __umul64hi(i, p.magic), k = i - j * p.n;
    if (k >= p.n) {
        ++j;
        k -= p.n;
    }
    return (__ldg(p.values + k) >> j) & 1u;
}

template <bool PLANES>
__global__ void __launch_bounds__(256)
encrypt_batch_kernel(const uint8_t *__restrict__ bits, const uint64_t n, const uint64_t first_block,
                     const uint32_t L, const uint64_t pad_mask, const uint64_t *__restrict__ mask,
                     const uint64_t *__restrict__ positions, const uint32_t D, const uint32_t k0, const uint32_t k1,
                     uint64_t *__restrict__ out, const UIntPlanes planes) {
    pdl_enter();
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint64_t b = first_block + i;
        const uint32_t b_lo = (uint32_t)b, b_hi = (uint32_t)(b >> 32);
        const bool one = PLANES ? plane_bit(planes, i) : (__ldg(bits + i) & 1u);
        uint64_t hole = 0, hbit = 0, hole_word = 0;
        if (!one) {
            const uint4 r = philox4x32_10(b_lo, b_hi, 0xffffffffu, kTag, k0, k1);
            hole = __ldg(positions + (r.x % D));
            hbit = 1ull << (63u - (uint32_t)(hole & 63u));
        }
        const uint32_t hw = (uint32_t)(hole >> 6);
        uint64_t *blk = out + i * L;
        bool others = true;
        for (uint32_t u = 0; 2 * u < L; ++u) {
            const uint4 r = philox4x32_10(b_lo, b_hi, u, kTag, k0, k1);
            uint64_t w[2] = {(uint64_t)r.x | ((uint64_t)r.y << 32), (uint64_t)r.z | ((uint64_t)r.w << 32)};
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const uint32_t wi = 2 * u + h;
                if (wi >= L) break;
                if (wi == L - 1) w[h] &= pad_mask;
                const uint64_t m = __ldg(mask + wi);
                if (one) {
                    w[h] |= m;
                } else {
                    const uint64_t mo = (wi == hw) ? (m & ~hbit) : m;
                    others = others && ((w[h] & mo) == mo);
                    if (wi == hw) hole_word = w[h];
                }
                blk[wi] = w[h];
            }
        }
        if (!one && others) blk[hw] = hole_word & ~hbit;
    }
}

// Short even blocks (L4 = L/2 <= 32 units, e.g. N=1247): a warp builds 32 consecutive blocks and
// walks their 32*L4 units in L4 fully coalesced steps, one Philox call and one 16-byte store per
// lane and step.  "Every other secret bit is 1" is a per-block AND across lanes: as in the decrypt
// kernel, each step's ballot goes into a per-warp fail string and lane b reads block b's bits; the
// lane then patches the hole word of its block.
template <int L4C, bool PLANES>
__global__ void __launch_bounds__(256)
encrypt_batch_units_kernel(const uint8_t *__restrict__ bits, const uint64_t n, const uint64_t first_block,
                           const uint32_t L4rt, const uint64_t pad_mask, const uint64_t *__restrict__ mask,
                           const uint64_t *__restrict__ positions, const uint32_t D, const uint32_t k0,
                           const uint32_t k1, uint64_t *__restrict__ out, const UIntPlanes planes) {
    constexpr int kWarps = 8;
    __shared__ uint64_t sMask[64];               // 2*L4 <= 64 words
    __shared__ uint32_t sFail[kWarps][32];       // L4 <= 32 ballot words per warp
    __shared__ uint32_t sHole[kWarps][32];       // per block of the chunk: hole position, or ~0u for Enc(1)
    const uint32_t L4 = L4C ? (uint32_t)L4C : L4rt;
    const uint32_t L = 2 * L4;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    pdl_enter();
    if (threadIdx.x < L) sMask[threadIdx.x] = mask[threadIdx.x];
    __syncthreads();
    uint4 *out4 = reinterpret_cast<uint4 *>(out);
    const uint64_t n_chunks = (n + 31) >> 5;
    for (uint64_t chunk = (uint64_t)blockIdx.x * kWarps + warp; chunk < n_chunks; chunk += (uint64_t)gridDim.x * kWarps) {
        // lane b prepares block b of the chunk: its bit and, for Enc(0), its hole
        const uint64_t my_i = chunk * 32u + lane;
        uint32_t my_hole = 0xffffffffu;
        if (my_i < n && !(PLANES ? plane_bit(planes, my_i) : (__ldg(bits + my_i) & 1u))) {
            const uint64_t b = first_block + my_i;
            const uint4 r = philox4x32_10((uint32_t)b, (uint32_t)(b >> 32), 0xffffffffu, kTag, k0, k1);
            my_hole = (uint32_t)__ldg(positions + (r.x % D));
        }
        sHole[warp][lane] = my_hole;
        __syncwarp();
        for (uint32_t r = 0; r < L4; ++r) {
            const uint32_t q = 32u * r + lane;            // unit within the chunk
            const uint32_t bl = q / L4, u = q - bl * L4;  // block within the chunk, unit within the block
            const uint64_t i = chunk * 32u + bl;
            bool fail = false;
            if (i < n) {
                const uint64_t b = first_block + i;
                const uint4 x = philox4x32_10((uint32_t)b, (uint32_t)(b >> 32), u, kTag, k0, k1);
                uint64_t w0 = (uint64_t)x.x | ((uint64_t)x.y << 32), w1 = (uint64_t)x.z | ((uint64_t)x.w << 32);
                if (u == L4 - 1) w1 &= pad_mask;
                const uint64_t m0 = sMask[2 * u], m1 = sMask[2 * u + 1];
                const uint32_t hole = sHole[warp][bl];
                if (hole == 0xffffffffu) {
                    w0 |= m0;
                    w1 |= m1;
                } else {
                    const uint64_t hbit = 1ull << (63u - (hole & 63u));
                    const uint32_t hw = hole >> 6;
                    const uint64_t mo0 = (hw == 2 * u) ? (m0 & ~hbit) : m0, mo1 = (hw == 2 * u + 1) ? (m1 & ~hbit) : m1;
                    fail = ((w0 & mo0) != mo0) || ((w1 & mo1) != mo1);
                }
                out4[i * L4 + u] = make_uint4((uint32_t)w0, (uint32_t)(w0 >> 32), (uint32_t)w1, (uint32_t)(w1 >> 32));
            }
            const uint32_t bal = __ballot_sync(0xffffffffu, fail);
            if (lane == 0) sFail[warp][r] = bal;
        }
        __syncwarp();   // orders the stores above before the patch below, within the warp
        if (my_hole != 0xffffffffu) {
            const uint32_t lo = lane * L4, hi = lo + L4;
            uint32_t any = 0;
            for (uint32_t w = lo >> 5; w <= (hi - 1) >> 5; ++w) {
                const uint32_t first = max(lo, w << 5) - (w << 5), last = min(hi, (w + 1) << 5) - (w << 5);
                const uint32_t m = (last - first == 32u) ? 0xffffffffu : (((1u << (last - first)) - 1u) << first);
                any |= sFail[warp][w] & m;
            }
            if (any == 0u) out[my_i * L + (my_hole >> 6)] &= ~(1ull << (63u - (my_hole & 63u)));
        }
        __syncwarp();
    }
}

// Long blocks (L >= 64 words, e.g. N=16383): one WARP builds one block, lanes striding over the
// 16-byte units -- coalesced 512-byte stores per step; the "other secret bits" flag is a warp vote.
template <bool PLANES>
__global__ void __launch_bounds__(256)
encrypt_batch_warp_kernel(const uint8_t *__restrict__ bits, const uint64_t n, const uint64_t first_block,
                          const uint32_t L, const uint64_t pad_mask, const uint64_t *__restrict__ mask,
                          const uint64_t *__restrict__ positions, const uint32_t D, const uint32_t k0,
                          const uint32_t k1, uint64_t *__restrict__ out, const UIntPlanes planes) {
    pdl_enter();
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warp_global = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint32_t n_units = (L + 1) / 2;
    for (uint64_t i = warp_global; i < n; i += n_warps) {
        const uint64_t b = first_block + i;
        const uint32_t b_lo = (uint32_t)b, b_hi = (uint32_t)(b >> 32);
        const bool one = PLANES ? plane_bit(planes, i) : (__ldg(bits + i) & 1u);
        uint64_t hole = 0, hbit = 0;
        if (!one) {
            const uint4 r = philox4x32_10(b_lo, b_hi, 0xffffffffu, kTag, k0, k1);   // same value on every lane
            hole = __ldg(positions + (r.x % D));
            hbit = 1ull << (63u - (uint32_t)(hole & 63u));
        }
        const uint32_t hw = (uint32_t)(hole >> 6);
        uint64_t *blk = out + i * L;
        bool others = true;
        for (uint32_t u = lane; u < n_units; u += 32) {
            const uint4 r = philox4x32_10(b_lo, b_hi, u, kTag, k0, k1);
            uint64_t w[2] = {(uint64_t)r.x | ((uint64_t)r.y << 32), (uint64_t)r.z | ((uint64_t)r.w << 32)};
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const uint32_t wi = 2 * u + h;
                if (wi >= L) break;
                if (wi == L - 1) w[h] &= pad_mask;
                const uint64_t m = __ldg(mask + wi);
                if (one) {
                    w[h] |= m;
                } else {
                    const uint64_t mo = (wi == hw) ? (m & ~hbit) : m;
                    others = others && ((w[h] & mo) == mo);
                }
                blk[wi] = w[h];
            }
        }
        const bool all_others = __all_sync(0xffffffffu, others);
        __syncwarp();
        if (!one && all_others && lane == ((hw >> 1) & 31u)) blk[hw] &= ~hbit;   // the lane that wrote word hw
    }
}

}  // namespace

namespace {

template <bool PLANES>
cudaError_t launch_encrypt(const uint8_t *bits, const UIntPlanes &planes, uint64_t n, uint64_t first_block, uint32_t L,
                           uint64_t pad_mask, const uint64_t *mask, const uint64_t *positions, uint32_t D, uint64_t seed,
                           uint64_t *out, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    count_launch();
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    if (L >= 64) {
        const uint32_t wgrid = (uint32_t)std::max<uint64_t>(
            1, std::min<uint64_t>((n + 7) / 8, (uint64_t)device_props().sm_count * 8));
        return launch_kernel(encrypt_batch_warp_kernel<PLANES>, wgrid, 256, 0, stream, bits, n, first_block, L, pad_mask,
                             mask, positions, D, k0, k1, out, planes);
    }
    const bool aligned = (reinterpret_cast<uintptr_t>(out) & 15u) == 0;
    if (!(L & 1u) && L <= 64 && aligned && !env_long("CSGN_ENC_LANE", 0)) {
        const uint64_t n_chunks = (n + 31) / 32;
        const uint32_t ugrid = (uint32_t)std::max<uint64_t>(
            1, std::min<uint64_t>((n_chunks + 7) / 8, (uint64_t)device_props().sm_count * 8));
        if (L == 20)
            return launch_kernel(encrypt_batch_units_kernel<10, PLANES>, ugrid, 256, 0, stream, bits, n, first_block,
                                 L / 2, pad_mask, mask, positions, D, k0, k1, out, planes);
        return launch_kernel(encrypt_batch_units_kernel<0, PLANES>, ugrid, 256, 0, stream, bits, n, first_block, L / 2,
                             pad_mask, mask, positions, D, k0, k1, out, planes);
    }
    const uint32_t grid = (uint32_t)std::max<uint64_t>(
        1, std::min<uint64_t>((n + 255) / 256, (uint64_t)device_props().sm_count * 8));
    return launch_kernel(encrypt_batch_kernel<PLANES>, grid, 256, 0, stream, bits, n, first_block, L, pad_mask, mask,
                         positions, D, k0, k1, out, planes);
}

}  // namespace

cudaError_t launch_encrypt_batch(const uint8_t *bits, uint64_t n, uint64_t first_block, uint32_t L, uint64_t pad_mask,
                                 const uint64_t *mask, const uint64_t *positions, uint32_t D, uint64_t seed,
                                 uint64_t *out, cudaStream_t stream) {
    return launch_encrypt<false>(bits, UIntPlanes{}, n, first_block, L, pad_mask, mask, positions, D, seed, out, stream);
}

cudaError_t launch_encrypt_uint(const uint64_t *values, uint64_t n, uint32_t width, uint64_t first_block, uint32_t L,
                                uint64_t pad_mask, const uint64_t *mask, const uint64_t *positions, uint32_t D,
                                uint64_t seed, uint64_t *out, cudaStream_t stream) {
    const UIntPlanes planes = {values, n, n ? UINT64_MAX / n : 0};
    return launch_encrypt<true>(nullptr, planes, (uint64_t)width * n, first_block, L, pad_mask, mask, positions, D,
                                seed, out, stream);
}

}  // namespace csgn
