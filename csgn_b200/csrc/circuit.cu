// circuit.cu -- a whole gate circuit over every lane of a set of ciphertext arrays in one launch (csgn_seg_circuit).
//
// Lanes are independent, so a persistent grid runs one warp per lane and the warps take lanes from a device counter.
// A lane's gate wires live in its slice of a scratch arena (cap blocks); its wire table (address, blocks, live) sits in
// a per-warp table in global memory.  Input wires point straight into the input buffers and are never copied.
//
// A gate is evaluated in the output order of csgn_seg_mul_sum (its products i-major, then its terms; a term is a
// product with the all-ones block) with the lane layout of segments.cu's seg_mul_kernel: for U < 32 units a warp step
// covers 32/U blocks, lane l holding unit l % U of block l / U, and a block's popcount comes from a shuffle scan and
// its rank from a ballot of the group leaders; for U >= 32 the lanes walk one block in steps of 32 units and a warp
// reduction gives its popcount.  Survivors are written contiguously at the arena's top.  Every warp vote runs on the
// full mask.
//
// Cancellation runs in place on the gate's output, with the rule of csgn_seg_cancel: the first occurrence of every block
// value that occurs an odd number of times.  Each warp has a hash table of kCancelSlots slots in shared memory; a slot
// holds (the lowest index + 1) of the blocks of its value (atomicCAS takes it, atomicMin lowers it), and a parity bit.
//
// Wires die at their last use (the host stages that list).  When a gate's uncompacted bound does not fit above the
// arena's top, the live wires slide down to the bottom of the slice; when it still does not fit, or a gate's output
// exceeds kCircuitCancelBlocks and must be cancelled, the lane is flagged and abandoned: the host evaluates it gate by
// gate.  Wires written by the kernel are read back with plain loads (never the read-only path).
#include "kernels.cuh"
#include "launch.cuh"
#include "seg_device.cuh"

#include <algorithm>

namespace csgn {
namespace {

constexpr int kCircThreads = 256;
constexpr uint32_t kCircWarpsPerCta = kCircThreads / 32;
constexpr uint32_t kCancelSlots = 2 * kCircuitCancelBlocks;   // a power of two: load factor at most 1/2
// per warp: the slots (uint32), their parity bits, the slot of every block (uint16)
constexpr size_t kCancelSmemPerWarp = kCancelSlots * 4 + kCancelSlots / 8 + kCircuitCancelBlocks * 2;
static_assert(kCancelSmemPerWarp % 16 == 0, "per-warp cancel scratch keeps 16-byte alignment");

struct Wire {
    uint64_t p;      // device address of the wire's first block
    uint32_t len;    // blocks
    uint32_t arena;  // 1: a live wire in the lane's arena slice
};
static_assert(sizeof(Wire) == kCircuitWireBytes, "wire table entry");

template <typename VT>
__device__ __forceinline__ VT all_ones();
template <>
__device__ __forceinline__ uint2 all_ones<uint2>() { return make_uint2(~0u, ~0u); }
template <>
__device__ __forceinline__ uint4 all_ones<uint4>() { return make_uint4(~0u, ~0u, ~0u, ~0u); }

// The gate with operands at `ops` (p pairs, then q terms) into out[0, ...): returns the blocks written.
template <typename VT>
__device__ uint32_t gate_eval(const uint32_t *ops, uint32_t p, uint32_t q, const Wire *wires, VT *out, uint32_t U,
                              uint32_t min_bits) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t G = U >= 32u ? 1u : 32u / U;                // blocks per warp step
    const uint32_t w0 = U >= 32u ? lane : lane % U;
    const uint32_t j0 = U >= 32u ? 0u : lane / U;
    const uint32_t gl = j0 * U, glast = min(gl + U - 1u, 31u);
    const uint32_t below = (1u << gl) - 1u;                   // leaders of the groups before this one
    uint32_t running = 0;
    for (uint32_t i = 0; i < p + q; ++i) {
        const bool term = i >= p;
        const Wire y = wires[__ldg(ops + (term ? p + i : 2 * i + 1))];
        const Wire x = term ? y : wires[__ldg(ops + 2 * i)];
        const uint32_t t1 = term ? 1u : x.len, t2 = y.len;
        if (t1 == 0 || t2 == 0) continue;
        const VT *a = reinterpret_cast<const VT *>(x.p), *b = reinterpret_cast<const VT *>(y.p);
        for (uint32_t r = 0; r < t1; ++r) {
            const VT *arow = a + (uint64_t)r * U;
            if (U < 32u) {
                VT xa = {};
                if (j0 < G) xa = term ? all_ones<VT>() : arow[w0];
                for (uint32_t js = 0; js < t2; js += G) {
                    const uint32_t j = js + j0;
                    const bool has = j0 < G && j < t2;
                    VT v = {};
                    if (has) v = vand(xa, b[(uint64_t)j * U + w0]);
                    bool alive = has;
                    if (min_bits) {                            // inclusive scan; a group's total is a difference
                        uint32_t s = vpopc(v);
#pragma unroll
                        for (uint32_t d = 1; d < 32u; d <<= 1) {
                            const uint32_t z = __shfl_up_sync(0xffffffffu, s, d);
                            if (lane >= d) s += z;
                        }
                        const uint32_t hi = __shfl_sync(0xffffffffu, s, glast);
                        const uint32_t lo = __shfl_sync(0xffffffffu, s, gl ? gl - 1u : 0u);
                        alive = has && hi - (gl ? lo : 0u) >= min_bits;
                    }
                    const uint32_t vote = __ballot_sync(0xffffffffu, alive && w0 == 0u);
                    if (alive) out[((uint64_t)running + __popc(vote & below)) * U + w0] = v;
                    running += __popc(vote);
                }
            } else {
                // the block goes to position `running` at once; a block that does not survive is overwritten
                for (uint32_t j = 0; j < t2; ++j) {
                    const VT *brow = b + (uint64_t)j * U;
                    VT *o = out + (uint64_t)running * U;
                    uint32_t s = 0;
                    for (uint32_t w = lane; w < U; w += 32u) {
                        const VT v = term ? brow[w] : vand(arow[w], brow[w]);
                        o[w] = v;
                        s += vpopc(v);
                    }
                    if (min_bits == 0u || __reduce_add_sync(0xffffffffu, s) >= min_bits) ++running;
                }
            }
        }
    }
    __syncwarp();
    return running;
}

// v[0, T) reduced in place to the first occurrence of every value that occurs an odd number of times (T <=
// kCircuitCancelBlocks).  Groups of G lanes (the power of two >= U, up to 32) take one block each per warp step, as in
// segments.cu's cancellation.  Returns the surviving blocks.
template <typename VT>
__device__ uint32_t cancel_in_place(VT *v, uint32_t T, uint32_t U, uint32_t *occ, uint32_t *par, uint16_t *slot_of) {
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t log2g = 0;
    while (log2g < 5 && (1u << log2g) < U) ++log2g;
    const uint32_t G = 1u << log2g, sub = lane & (G - 1u), grp = lane >> log2g, B = 32u >> log2g;
    constexpr uint32_t mask = kCancelSlots - 1u;
    for (uint32_t s = lane; s < kCancelSlots; s += 32u) occ[s] = 0u;
    for (uint32_t s = lane; s < kCancelSlots / 32u; s += 32u) par[s] = 0u;
    __syncwarp();
    for (uint32_t i0 = 0; i0 < T; i0 += B) {
        const uint32_t i = i0 + grp;
        const bool live = i < T;
        const VT *p = v + (uint64_t)i * U;
        uint64_t h = 0;
        if (live)
            for (uint32_t w = sub; w < U; w += G) h += unit_hash(p[w], w);
#pragma unroll
        for (uint32_t d = 1; d < 32u; d <<= 1) {
            const uint64_t y = __shfl_xor_sync(0xffffffffu, h, d);
            if (d < G) h += y;
        }
        uint32_t slot = (uint32_t)mix64(h) & mask;
        if (G < 32u) {                                         // the group leader probes alone
            if (live && sub == 0u) {
                for (;;) {
                    const uint32_t o = atomicCAS(occ + slot, 0u, i + 1u);
                    if (o == 0u) break;
                    const VT *q = v + (uint64_t)(o - 1u) * U;
                    bool eq = true;
                    for (uint32_t w = 0; w < U && eq; ++w) eq = veq(p[w], q[w]);
                    if (eq) {
                        atomicMin(occ + slot, i + 1u);
                        break;
                    }
                    slot = (slot + 1u) & mask;
                }
                atomicXor(par + (slot >> 5), 1u << (slot & 31u));
                slot_of[i] = (uint16_t)slot;
            }
        } else {                                               // one block per step: the whole warp probes
            for (;;) {
                uint32_t o = 0;
                if (lane == 0u) o = atomicCAS(occ + slot, 0u, i + 1u);
                o = __shfl_sync(0xffffffffu, o, 0);
                if (o == 0u) break;
                const VT *q = v + (uint64_t)(o - 1u) * U;
                bool eq = true;
                for (uint32_t w = lane; w < U; w += 32u) eq &= veq(p[w], q[w]);
                if (__all_sync(0xffffffffu, eq)) {
                    if (lane == 0u) atomicMin(occ + slot, i + 1u);
                    break;
                }
                slot = (slot + 1u) & mask;
            }
            if (lane == 0u) {
                atomicXor(par + (slot >> 5), 1u << (slot & 31u));
                slot_of[i] = (uint16_t)slot;
            }
        }
    }
    __syncwarp();
    // Survivors move down in order.  A block's destination d <= its index; with G < 32 it may be a block of the same
    // step that another group has not read yet, hence the read, sync, write.  With G = 32 every lane copies the units
    // it alone reads and writes.
    const uint32_t below = (1u << (grp * G)) - 1u;             // lanes of the groups before this one
    uint32_t running = 0;
    for (uint32_t i0 = 0; i0 < T; i0 += B) {
        const uint32_t i = i0 + grp;
        bool keep = false;
        if (i < T) {
            const uint32_t s = slot_of[i];
            keep = occ[s] == i + 1u && ((par[s >> 5] >> (s & 31u)) & 1u);
        }
        const uint32_t vote = __ballot_sync(0xffffffffu, keep && sub == 0u);
        const uint32_t d = running + __popc(vote & below);
        if (G < 32u) {
            const bool mine = keep && sub < U && d != i;
            VT x = {};
            if (mine) x = v[(uint64_t)i * U + sub];
            __syncwarp();
            if (mine) v[(uint64_t)d * U + sub] = x;
            __syncwarp();
        } else if (keep && d != i) {
            for (uint32_t w = lane; w < U; w += 32u) v[(uint64_t)d * U + w] = v[(uint64_t)i * U + w];
        }
        running += __popc(vote);
    }
    __syncwarp();
    return running;
}

// The live arena wires among [first, end) moved down, in order, to the bottom of the slice; returns the new top.
template <typename VT>
__device__ uint64_t slide_down(Wire *wires, uint32_t first, uint32_t end, VT *base, uint32_t U) {
    const uint32_t lane = threadIdx.x & 31u;
    uint64_t dst = 0;
    for (uint32_t w = first; w < end; ++w) {
        const Wire x = wires[w];
        if (!x.arena) continue;
        const VT *src = reinterpret_cast<const VT *>(x.p);
        VT *d = base + dst * U;
        if (src != d) {                                        // d < src: chunks move in increasing order
            const uint64_t units = (uint64_t)x.len * U;
            for (uint64_t u0 = 0; u0 < units; u0 += 32u) {
                const uint64_t u = u0 + lane;
                VT y = {};
                if (u < units) y = src[u];
                __syncwarp();
                if (u < units) d[u] = y;
                __syncwarp();
            }
            if (lane == 0u) wires[w].p = reinterpret_cast<uint64_t>(d);
            __syncwarp();
        }
        dst += x.len;
    }
    return dst;
}

// Every gate over lane k; false when the lane does not fit (it is then abandoned).
template <typename VT>
__device__ bool run_lane(const CircuitArgs &a, uint32_t U, uint64_t k, Wire *wires, uint32_t *smem) {
    const uint32_t lane = threadIdx.x & 31u;
    VT *base = reinterpret_cast<VT *>(a.arena) + k * a.cap * U;
    bool big = false;
    for (uint32_t i = lane; i < a.n_inputs; i += 32u) {
        const uint64_t *o = a.in_off + (uint64_t)i * (a.n + 1) + k;
        const uint64_t o0 = __ldg(o), t = __ldg(o + 1) - o0;
        big |= t > 0xffffffffull;                              // wire lengths are 32-bit
        wires[i] = {__ldg(a.in_base + i) + o0 * U * sizeof(VT), (uint32_t)t, 0u};
    }
    if (__any_sync(0xffffffffu, big)) return false;
    __syncwarp();
    uint32_t *occ = smem, *par = occ + kCancelSlots;
    uint16_t *slot_of = reinterpret_cast<uint16_t *>(par + kCancelSlots / 32);
    uint64_t top = 0;                                          // blocks in use at the bottom of the slice
    for (uint32_t g = 0; g < a.n_gates; ++g) {
        const uint32_t *gp = a.gates + __ldg(a.gate_at + g);
        const uint32_t p = __ldg(gp), q = __ldg(gp + 1);
        const uint32_t *ops = gp + 2;
        uint64_t bound = 0;                                    // the uncompacted output, or more than cap
        for (uint32_t i = 0; i < p + q && bound <= a.cap; ++i)
            bound += i < p ? (uint64_t)wires[__ldg(ops + 2 * i)].len * wires[__ldg(ops + 2 * i + 1)].len
                           : wires[__ldg(ops + p + i)].len;
        if (bound > a.cap - top) {
            top = slide_down(wires, a.n_inputs, a.n_inputs + g, base, U);
            if (bound > a.cap - top) return false;
        }
        VT *out = base + top * U;
        uint32_t t = gate_eval(ops, p, q, wires, out, U, a.min_bits);
        if (a.cancel && t > 1u) {
            if (t > kCircuitCancelBlocks) return false;
            t = cancel_in_place(out, t, U, occ, par, slot_of);
        }
        if (lane == 0u) wires[a.n_inputs + g] = {reinterpret_cast<uint64_t>(out), t, 1u};
        top += t;
        __syncwarp();
        const uint32_t f1 = __ldg(a.free_at + g + 1);
        for (uint32_t f = __ldg(a.free_at + g) + lane; f < f1; f += 32u) wires[__ldg(a.frees + f)].arena = 0u;
        __syncwarp();
    }
    for (uint32_t j = lane; j < a.n_outputs; j += 32u) {
        const uint32_t w = __ldg(a.outputs + j);
        if (w < a.n_inputs) continue;
        const Wire x = wires[w];
        uint64_t *r = a.res + 2 * (k * a.n_outputs + j);
        r[0] = (x.p - reinterpret_cast<uint64_t>(base)) / (U * sizeof(VT));
        r[1] = x.len;
    }
    return true;
}

template <typename VT>
__global__ void __launch_bounds__(kCircThreads, 2) circuit_kernel(const CircuitArgs a, const uint32_t U) {
    extern __shared__ __align__(16) uint32_t circuit_smem[];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    Wire *wires = reinterpret_cast<Wire *>(a.wires) +
                  (uint64_t)(blockIdx.x * kCircWarpsPerCta + warp) * (a.n_inputs + a.n_gates);
    uint32_t *smem = circuit_smem + (a.cancel ? warp * (uint32_t)(kCancelSmemPerWarp / 4) : 0u);
    pdl_enter();
    for (;;) {
        unsigned long long k = 0;
        if (lane == 0u) k = atomicAdd(a.next, 1ull);
        k = __shfl_sync(0xffffffffu, k, 0);
        if (k >= a.n) break;
        const bool ok = run_lane<VT>(a, U, k, wires, smem);
        if (lane == 0u) a.fallback[k] = ok ? 0u : 1u;
        __syncwarp();
    }
}

size_t smem_bytes(bool cancel) { return cancel ? kCancelSmemPerWarp * kCircWarpsPerCta : 0; }

// The persistent grid: as many CTAs as are resident at once, and no more than the lanes need.
template <typename VT>
uint32_t circuit_grid(uint64_t n, bool cancel) {
    static bool attr = false;
    if (!attr) {
        cudaFuncSetAttribute(circuit_kernel<VT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes(true));
        attr = true;
    }
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, circuit_kernel<VT>, kCircThreads, smem_bytes(cancel)) !=
            cudaSuccess ||
        per_sm < 1)
        per_sm = 1;
    const uint64_t want = (n + kCircWarpsPerCta - 1) / kCircWarpsPerCta;
    return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(want, (uint64_t)device_props().sm_count * per_sm));
}

}  // namespace

uint32_t circuit_warps(uint64_t n, bool units16, bool cancel) {
    return (units16 ? circuit_grid<uint4>(n, cancel) : circuit_grid<uint2>(n, cancel)) * kCircWarpsPerCta;
}

cudaError_t launch_circuit(const CircuitArgs &a, uint32_t L, bool units16, cudaStream_t stream) {
    if (a.n == 0) return cudaSuccess;
    count_launch();
    const bool cancel = a.cancel != 0;
    if (units16)
        return launch_kernel(circuit_kernel<uint4>, circuit_grid<uint4>(a.n, cancel), kCircThreads,
                             smem_bytes(cancel), stream, a, L / 2);
    return launch_kernel(circuit_kernel<uint2>, circuit_grid<uint2>(a.n, cancel), kCircThreads, smem_bytes(cancel),
                         stream, a, L);
}

}  // namespace csgn
