// misc.cu -- K2 (ciphertext add = block concatenation), the piece-table copy of ciphertext arrays, and the device
// checksum.
//
// K2: out = a || b            (reference src/Ciphertext.cpp:107-122, :215-223)
// Roofline: HBM copy bandwidth, 16*L bytes per block moved (8*L read + 8*L written).
// operator+= appends in place (out == a): only b moves.
#include "kernels.cuh"
#include "launch.cuh"

#include <algorithm>

namespace csgn {
namespace {

constexpr int kCopyThreads = 256;
constexpr int kCopyUnroll = 4;

// The streaming copy loop shared by every copy kernel: CTA tiles of kCopyThreads * kCopyUnroll units over the
// destination, grid-stride, kCopyUnroll loads in flight per thread before the stores.  `src.tile(first, end)` is
// called once per tile (uniform over the CTA), `src.load(i)` returns destination unit i.
template <typename VecT, typename Src>
__device__ __forceinline__ void stream_copy(Src &src, const uint64_t total, VecT *__restrict__ out) {
    const uint64_t span = (uint64_t)blockDim.x * kCopyUnroll;
    const uint64_t stride = (uint64_t)gridDim.x * span;
    for (uint64_t tile = (uint64_t)blockIdx.x * span; tile < total; tile += stride) {
        src.tile(tile, tile + span < total ? tile + span : total);
        VecT v[kCopyUnroll];
        bool live[kCopyUnroll];
#pragma unroll
        for (int u = 0; u < kCopyUnroll; ++u) {
            const uint64_t i = tile + threadIdx.x + (uint64_t)u * blockDim.x;
            live[u] = i < total;
            if (live[u]) v[u] = src.load(i);
        }
#pragma unroll
        for (int u = 0; u < kCopyUnroll; ++u) {
            const uint64_t i = tile + threadIdx.x + (uint64_t)u * blockDim.x;
            if (live[u]) __stcs(out + i, v[u]);
        }
    }
}

template <typename VecT>
struct TwoSources {
    const VecT *__restrict__ a;
    uint64_t na;
    const VecT *__restrict__ b;
    __device__ __forceinline__ void tile(uint64_t, uint64_t) {}
    __device__ __forceinline__ VecT load(uint64_t i) const { return (i < na) ? __ldcs(a + i) : __ldcs(b + (i - na)); }
};

// Two-source streaming copy.  VecT = uint4 when every pointer and both lengths are
// 16-byte granular, else uint64_t.
template <typename VecT>
__global__ void __launch_bounds__(kCopyThreads)
concat_kernel(const VecT *__restrict__ a, const uint64_t na, const VecT *__restrict__ b, const uint64_t nb,
              VecT *__restrict__ out) {
    TwoSources<VecT> src{a, na, b};
    pdl_enter();
    stream_copy(src, na + nb, out);
}

// Piece table (ciphertext arrays, segments.cu): destination units [dst[p], dst[p+1]) come from src[p].  The pieces
// that a tile touches are found once per tile; a unit then searches only among those.
template <typename VecT>
struct PieceSources {
    const VecT *const *__restrict__ src;
    const uint64_t *__restrict__ dst;      // n + 1 unit offsets, dst[0] = 0, dst[n] = total
    uint32_t n;
    uint32_t lo, hi;                       // pieces of the current tile
    // last p in [l, h] with dst[p] <= i
    __device__ __forceinline__ uint32_t find(uint64_t i, uint32_t l, uint32_t h) const {
        while (l < h) {
            const uint32_t m = (l + h + 1) >> 1;
            if (__ldg(dst + m) <= i) l = m;
            else h = m - 1;
        }
        return l;
    }
    __device__ __forceinline__ void tile(uint64_t first, uint64_t end) {
        lo = find(first, 0, n - 1);
        hi = find(end - 1, lo, n - 1);
    }
    __device__ __forceinline__ VecT load(uint64_t i) const {
        const uint32_t p = find(i, lo, hi);
        return __ldcs(src[p] + (i - __ldg(dst + p)));
    }
};

template <typename VecT>
__global__ void __launch_bounds__(kCopyThreads)
piece_copy_kernel(const VecT *const *__restrict__ src, const uint64_t *__restrict__ dst, const uint32_t n,
                  VecT *__restrict__ out) {
    PieceSources<VecT> s{src, dst, n, 0, 0};
    pdl_enter();
    stream_copy(s, dst[n], out);
}

uint32_t copy_grid(uint64_t units) {
    const uint64_t per_cta = (uint64_t)kCopyThreads * kCopyUnroll;
    return (uint32_t)std::max<uint64_t>(
        1, std::min<uint64_t>((units + per_cta - 1) / per_cta, (uint64_t)device_props().sm_count * 16));
}

__global__ void __launch_bounds__(256)
checksum_kernel(const uint64_t *__restrict__ v, const uint64_t n_words, uint64_t *acc) {
    uint64_t x = 0, s = 0, h = 0;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    pdl_enter();
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += stride) {
        const uint64_t w = __ldcs(v + i);
        x ^= w;
        s += w;
        h += w * (2ull * i + 1ull);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        x ^= __shfl_xor_sync(0xffffffffu, x, off);
        s += __shfl_xor_sync(0xffffffffu, s, off);
        h += __shfl_xor_sync(0xffffffffu, h, off);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicXor(reinterpret_cast<unsigned long long *>(acc), (unsigned long long)x);
        atomicAdd(reinterpret_cast<unsigned long long *>(acc + 1), (unsigned long long)s);
        atomicAdd(reinterpret_cast<unsigned long long *>(acc + 2), (unsigned long long)h);
    }
}

// out[0] = in[0] + ... + in[n-1]   (the partial counts of a ciphertext held as several segments)
__global__ void __launch_bounds__(32)
sum_words_kernel(const uint64_t *__restrict__ in, const uint32_t n, uint64_t *out) {
    pdl_enter();
    uint64_t s = 0;
    for (uint32_t i = threadIdx.x; i < n; i += 32) s += in[i];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if (threadIdx.x == 0) *out = s;
}

}  // namespace

cudaError_t launch_sum_words(const uint64_t *in, uint32_t n, uint64_t *out, cudaStream_t stream) {
    count_launch();
    return launch_kernel(sum_words_kernel, 1, 32, 0, stream, in, n, out);
}

cudaError_t launch_concat(const uint64_t *a, uint64_t n_words_a, const uint64_t *b, uint64_t n_words_b,
                          uint64_t *out, cudaStream_t stream) {
    if (a == out) {  // append in place: only b moves
        out += n_words_a;
        a = nullptr;
        n_words_a = 0;
    }
    if (n_words_a + n_words_b == 0) return cudaSuccess;
    const bool vec = (((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) |
                        reinterpret_cast<uintptr_t>(out)) & 15u) == 0) &&
                     (n_words_a % 2 == 0) && (n_words_b % 2 == 0);
    const uint64_t units = vec ? (n_words_a + n_words_b) / 2 : (n_words_a + n_words_b);
    const uint32_t grid = copy_grid(units);
    count_launch();
    if (vec)
        return launch_kernel(concat_kernel<uint4>, grid, kCopyThreads, 0, stream, reinterpret_cast<const uint4 *>(a),
                             n_words_a / 2, reinterpret_cast<const uint4 *>(b), n_words_b / 2,
                             reinterpret_cast<uint4 *>(out));
    return launch_kernel(concat_kernel<uint64_t>, grid, kCopyThreads, 0, stream, a, n_words_a, b, n_words_b, out);
}

cudaError_t launch_piece_copy(const void *const *src, const uint64_t *dst, uint32_t n_pieces, uint64_t total_units,
                              bool units16, void *out, cudaStream_t stream) {
    if (n_pieces == 0 || total_units == 0) return cudaSuccess;
    count_launch();
    if (units16)
        return launch_kernel(piece_copy_kernel<uint4>, copy_grid(total_units), kCopyThreads, 0, stream,
                             reinterpret_cast<const uint4 *const *>(src), dst, n_pieces, static_cast<uint4 *>(out));
    return launch_kernel(piece_copy_kernel<uint64_t>, copy_grid(total_units), kCopyThreads, 0, stream,
                         reinterpret_cast<const uint64_t *const *>(src), dst, n_pieces, static_cast<uint64_t *>(out));
}

cudaError_t launch_checksum(const uint64_t *v, uint64_t n_words, uint64_t *acc, cudaStream_t stream) {
    if (n_words == 0) return cudaSuccess;
    const DeviceProps &dp = device_props();
    const uint32_t grid = (uint32_t)std::max<uint64_t>(
        1, std::min<uint64_t>((n_words + 255) / 256, (uint64_t)dp.sm_count * 8));
    count_launch();
    return launch_kernel(checksum_kernel, grid, 256, 0, stream, v, n_words, acc);
}

}  // namespace csgn
