// segments.cu -- kernels of ciphertext arrays: many independent small ciphertexts held in ONE buffer, element k being
// blocks [off[k], off[k+1]) (include/csgn.h, "ciphertext arrays").  Each kernel serves any number of elements in one
// launch; the host (capi_seg.cu) builds the work tables from the offsets, so no kernel searches or divides per unit.
//
//   grouped multiply   element k = a_k * b_k, all-pairs AND, i-major      (reference src/Ciphertext.cpp:153-163),
//                      or a sum of products and plain terms a0_k*b0_k || ... || c0_k || ... (operands in any buffers;
//                      a term is a product with one all-ones block)
//   segmented decrypt  counts[k] = satisfied blocks of element k           (reference src/SecretKey.cpp:126-140),
//                      or over the bit planes of encrypted integers: bit j of values[k] = parity of element k of plane j
//   cancellation       element k = the first occurrence, in order, of every block value that occurs an odd number of
//                      times in element k (insert into a hash table per element, count, write)
//
// (the element-wise concat / gather / pack copy is misc.cu's streaming copy over a piece table.)
//
// Units are 16 bytes (uint4) when L is even and the storage is 16-byte aligned, 8 bytes otherwise.  A warp handles a
// block of U units with min(U, 32) lanes: for U < 32 one warp step covers 32/U (multiply) or 32/G (decrypt, G the
// power of two >= U) whole blocks, for U >= 32 the lanes walk the block in steps of 32 units.
#include "kernels.cuh"
#include "launch.cuh"
#include "fold.cuh"
#include "seg_device.cuh"

#include <algorithm>

namespace csgn {
namespace {

constexpr int kSegThreads = 256;
constexpr int kSegCtasPerSm = 8;

// Modes of the grouped multiply: kSegPlain writes every block at its item's `out`; kSegCount writes, per item, the
// number of its blocks with at least min_bits set bits (live[it]); kSegWriteLive writes only those blocks, in order,
// from block base[it] on.
enum SegMode { kSegPlain, kSegCount, kSegWriteLive };

// ---------------------------------------------------------------------------------------
// grouped multiply: a warp task is a run of items; an item is the `rows` blocks at address a (rows of one element's
// left operand, or the all-ones block of a plain term) times the t2 blocks at address b, written to block `out` on.
// Lane l holds unit w = l % U of block j = l / U of each warp step (U < 32), or units l, l+32, ... of one block
// (U >= 32).
// The counting modes walk an item's blocks in warp steps that every lane takes (no early return, no per-lane loop
// bound), because each step votes with the full mask: a lane with no block (past t2, or beyond the last whole block of
// a step) counts 0 set bits and is not live.
// The counting modes ask for 3 resident CTAs per SM: left to its own register target, ptxas spills in them.
// ---------------------------------------------------------------------------------------
template <typename VT, SegMode MODE>
__global__ void __launch_bounds__(kSegThreads, MODE == kSegPlain ? 0 : 3)
seg_mul_kernel(VT *__restrict__ out, const uint32_t U, const SegMulItem *__restrict__ items,
               const uint32_t *__restrict__ tasks, const uint32_t n_tasks, const uint32_t min_bits,
               uint32_t *__restrict__ live, const uint64_t *__restrict__ base) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t G = U >= 32u ? 1u : 32u / U;                // blocks per warp step
    const uint32_t w0 = U >= 32u ? lane : lane % U;
    const uint32_t j0 = U >= 32u ? 0u : lane / U;
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    pdl_enter();
    if constexpr (MODE != kSegPlain) {
        // group of this lane (U < 32): lanes [gl, gl + U); the scan just before gl and at its last lane give its total
        const uint32_t gl = j0 * U, glast = min(gl + U - 1u, 31u);
        const uint32_t below = (1u << gl) - 1u;                // leaders of the groups before this one
        for (uint32_t t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < n_tasks; t += warps) {
            const uint32_t it_end = __ldg(tasks + t + 1);
            for (uint32_t it = __ldg(tasks + t); it < it_end; ++it) {
                const SegMulItem m = items[it];
                const VT *a = reinterpret_cast<const VT *>(m.a), *b = reinterpret_cast<const VT *>(m.b);
                uint64_t pos = MODE == kSegWriteLive ? __ldg(base + it) : 0;   // next surviving block of this item
                uint32_t running = 0;
                for (uint32_t r = 0; r < m.rows; ++r) {
                    const VT *arow = a + (uint64_t)r * U;
                    if (U < 32u) {
                        VT x = {};
                        if (j0 < G) x = __ldg(arow + w0);
                        for (uint32_t js = 0; js < m.t2; js += G) {
                            const uint32_t j = js + j0;
                            const bool has = j0 < G && j < m.t2;
                            VT v = {};
                            if (has) v = vand(x, __ldg(b + (uint64_t)j * U + w0));
                            // inclusive scan of the lanes' set bits; a group's total is a difference of two scans
                            uint32_t s = vpopc(v);
#pragma unroll
                            for (uint32_t d = 1; d < 32u; d <<= 1) {
                                const uint32_t y = __shfl_up_sync(0xffffffffu, s, d);
                                if (lane >= d) s += y;
                            }
                            const uint32_t hi = __shfl_sync(0xffffffffu, s, glast);
                            const uint32_t lo = __shfl_sync(0xffffffffu, s, gl ? gl - 1u : 0u);
                            const bool alive = has && hi - (gl ? lo : 0u) >= min_bits;
                            const uint32_t vote = __ballot_sync(0xffffffffu, alive && w0 == 0u);
                            if (MODE == kSegWriteLive && alive)
                                __stcs(out + (pos + running + __popc(vote & below)) * U + w0, v);
                            running += __popc(vote);
                        }
                    } else {
                        for (uint32_t j = 0; j < m.t2; ++j) {
                            const VT *brow = b + (uint64_t)j * U;
                            uint32_t s = 0;
                            for (uint32_t w = w0; w < U; w += 32u) s += vpopc(vand(__ldg(arow + w), __ldg(brow + w)));
                            if (__reduce_add_sync(0xffffffffu, s) >= min_bits) {   // the same verdict on every lane
                                if (MODE == kSegWriteLive) {                     // read again (L1 / L2), then store
                                    VT *o = out + (pos + running) * U;
#pragma unroll 4
                                    for (uint32_t w = w0; w < U; w += 32u)
                                        __stcs(o + w, vand(__ldg(arow + w), __ldg(brow + w)));
                                }
                                ++running;
                            }
                        }
                    }
                }
                if (MODE == kSegCount && lane == 0u) live[it] = running;
            }
        }
        return;
    }
    if (j0 >= G) return;                                       // lanes beyond the last whole block of a step
    for (uint32_t t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < n_tasks; t += warps) {
        const uint32_t it_end = __ldg(tasks + t + 1);
        for (uint32_t it = __ldg(tasks + t); it < it_end; ++it) {
            const SegMulItem m = items[it];
            const VT *a = reinterpret_cast<const VT *>(m.a), *b = reinterpret_cast<const VT *>(m.b);
            for (uint32_t r = 0; r < m.rows; ++r) {
                const VT *arow = a + (uint64_t)r * U;
                VT *orow = out + (m.out + (uint64_t)r * m.t2) * U;
                if (U < 32u) {
                    const VT x = __ldg(arow + w0);
#pragma unroll 4
                    for (uint32_t j = j0; j < m.t2; j += G)
                        __stcs(orow + (uint64_t)j * U + w0, vand(x, __ldg(b + (uint64_t)j * U + w0)));
                } else {
                    for (uint32_t j = 0; j < m.t2; ++j) {
                        const VT *brow = b + (uint64_t)j * U;
                        VT *o = orow + (uint64_t)j * U;
#pragma unroll 4
                        for (uint32_t w = w0; w < U; w += 32u) __stcs(o + w, vand(__ldg(arow + w), __ldg(brow + w)));
                    }
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// segmented decrypt: groups of G lanes (G a power of two, >= U up to 32) evaluate one block each per warp step; the
// group's verdict is one ballot.  Group leaders that hold the same element find each other with match.any and add
// their verdicts with one more ballot: one atomic per (warp step, element), not one per block.
// With PLANES the tasks walk the bit planes of encrypted integers: task t reads plane task_plane[t], whose storage and
// offsets come from planes[], and XORs its elements' parities into bit j of counts[e] instead of adding the counts.
// ---------------------------------------------------------------------------------------
// The plane form holds the plane's addresses in registers: 6 resident CTAs per SM keep ptxas from spilling them.
template <typename VT, bool PLANES>
__global__ void __launch_bounds__(kSegThreads, PLANES ? 6 : 0)
seg_decrypt_kernel(const VT *__restrict__ v, const uint32_t U, const uint32_t log2g, const VT *__restrict__ mask,
                   const uint64_t *__restrict__ off, const SegDecTask *__restrict__ tasks, const uint32_t n_tasks,
                   uint64_t *counts, const SegPlane *__restrict__ planes, const uint32_t *__restrict__ task_plane) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t G = 1u << log2g, sub = lane & (G - 1u), grp = lane >> log2g, B = 32u >> log2g;
    const uint32_t gmask = G == 32u ? 0xffffffffu : ((1u << G) - 1u) << (grp * G);
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    pdl_enter();
    for (uint32_t t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < n_tasks; t += warps) {
        const SegDecTask task = tasks[t];
        uint32_t plane = 0;
        if constexpr (PLANES) {
            plane = __ldg(task_plane + t);
            v = reinterpret_cast<const VT *>(planes[plane].v);
            off = planes[plane].off;
        }
        uint64_t e = task.elem;                                // element of this lane's block: never decreases
        for (uint64_t blk0 = task.first; blk0 < task.end; blk0 += B) {
            const uint64_t blk = blk0 + grp;
            const bool live = blk < task.end;
            bool fails = false;
            if (live) {
                const VT *p = v + blk * U;
                for (uint32_t w = sub; w < U; w += G) fails |= unit_fails(__ldcs(p + w), __ldg(mask + w));
            }
            // the vote is taken by every lane (a `live && ballot` would skip it on lanes past the task's end)
            const uint32_t vote = __ballot_sync(0xffffffffu, fails);
            const bool sat = live && (vote & gmask) == 0u;
            const bool leader = live && sub == 0u;
            if (leader) {                                      // last e in [e, elem_last] with off[e] <= blk
                uint64_t lo = e, hi = task.elem_last;
                while (lo < hi) {
                    const uint64_t mid = lo + ((hi - lo + 1) >> 1);
                    if (__ldg(off + mid) <= blk) lo = mid;
                    else hi = mid - 1;
                }
                e = lo;
            }
            // Every lane executes both warp-wide votes with the full mask; a group's sum is the popcount of the
            // satisfied leaders among its peers (verdicts are 0 / 1), so no reduction runs over a partial mask.
            const uint64_t key = leader ? e : ~0ull;
            const uint32_t peers = __match_any_sync(0xffffffffu, key);
            const uint32_t sum = __popc(peers & __ballot_sync(0xffffffffu, leader && sat));
            if constexpr (PLANES) {
                if (leader && (sum & 1u) && lane == (uint32_t)(__ffs(peers) - 1))
                    atomicXor(reinterpret_cast<unsigned long long *>(counts + e), 1ull << plane);
            } else {
                if (leader && sum && lane == (uint32_t)(__ffs(peers) - 1))
                    atomicAdd(reinterpret_cast<unsigned long long *>(counts + e), (unsigned long long)sum);
            }
        }
    }
}

// The parities of the plane elements that were counted on their own (launch_decrypt_count): entry i XORs bit
// entries[2i + 1] of values[entries[2i]] with counts[i] & 1.  Several entries may name one value.
__global__ void __launch_bounds__(kSegThreads)
seg_uint_pack_kernel(const uint64_t *__restrict__ counts, const uint64_t *__restrict__ entries, const uint32_t n,
                     uint64_t *values) {
    pdl_enter();
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        if (__ldg(counts + i) & 1u)
            atomicXor(reinterpret_cast<unsigned long long *>(values + __ldg(entries + 2 * i)),
                      1ull << __ldg(entries + 2 * i + 1));
}

// ---------------------------------------------------------------------------------------
// cancellation: groups of G lanes (G the power of two >= U, up to 32) take one block each per warp step, as in the
// segmented decrypt.  A block's hash is the splitmix64 finaliser of the sum of its words' finalised values (each word
// offset by its position), so the lanes of a group add their parts in any order; the hash only chooses the first slot
// to probe.  Linear probing from there: an empty slot is taken by atomicCAS; a taken slot's occupant is compared word
// for word, and an equal occupant is the representative.  Equal blocks walk the same slots, and a slot is taken once,
// so every value of an element has exactly one representative whatever the order of the warps.  With G < 32 the group
// leader probes alone and compares serially (groups probe different numbers of slots, so no warp vote runs there);
// with G = 32 (WARP_BLOCK) the warp holds one block, every lane takes every probe, and lane 0's atomicCAS is broadcast.
// The insert pass asks for 4 resident CTAs per SM: left to its own register target, ptxas spills in the probe loops.
// (The hash and the unit helpers are in seg_device.cuh, shared with the circuit kernel.)
// ---------------------------------------------------------------------------------------

// Block b (of the whole array) survives when it is the first of its value's blocks and the value occurs an odd number
// of times in its element.
__device__ __forceinline__ bool cancel_survives(const uint64_t b, const SegCancelScratch &s) {
    const int32_t d = __ldg(s.rep + b);
    const uint64_t r = b - (uint64_t)(int64_t)d;
    return __ldg(s.first + r) == d && ((__ldg(s.parity + (r >> 5)) >> (r & 31u)) & 1u);
}

template <typename VT, bool WARP_BLOCK>
__global__ void __launch_bounds__(kSegThreads, 4)
seg_cancel_insert_kernel(const VT *__restrict__ v, const uint32_t U, const uint32_t log2g,
                         const SegCancelTask *__restrict__ tasks, const uint32_t n_tasks, const SegCancelScratch s) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t G = 1u << log2g, sub = lane & (G - 1u), grp = lane >> log2g, B = 32u >> log2g;
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    pdl_enter();
    for (uint32_t t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < n_tasks; t += warps) {
        const SegCancelTask task = tasks[t];
        const VT *ev = v + task.elem * U;                      // the element's first block
        uint32_t *slots = s.slots + task.slot;
        for (uint32_t i0 = task.first; i0 < task.end; i0 += B) {
            const uint32_t i = i0 + grp;                       // element-relative block of this lane's group
            const bool live = i < task.end;
            const VT *p = ev + (uint64_t)i * U;
            uint64_t h = 0;
            if (live)
                for (uint32_t w = sub; w < U; w += G) h += unit_hash(__ldg(p + w), w);
            // the group's sum on each of its lanes; every lane takes every step with the full mask
#pragma unroll
            for (uint32_t d = 1; d < 32u; d <<= 1) {
                const uint64_t y = __shfl_xor_sync(0xffffffffu, h, d);
                if (d < G) h += y;
            }
            h = mix64(h);
            uint32_t slot = (uint32_t)h & task.slot_mask, r = 0;
            bool records;                                      // the lane that records the block's representative
            if (!WARP_BLOCK) {
                records = live && sub == 0u;
                while (records) {
                    const uint32_t occ = atomicCAS(slots + slot, 0u, i + 1u);
                    if (occ == 0u) {
                        r = i;
                        break;
                    }
                    const VT *q = ev + (uint64_t)(occ - 1u) * U;
                    bool eq = true;
                    for (uint32_t w = 0; w < U && eq; ++w) eq = veq(__ldg(p + w), __ldg(q + w));
                    if (eq) {
                        r = occ - 1u;
                        break;
                    }
                    slot = (slot + 1u) & task.slot_mask;
                }
            } else {                                           // one block per warp step: the whole warp probes
                for (;;) {
                    uint32_t occ = 0;
                    if (lane == 0u) occ = atomicCAS(slots + slot, 0u, i + 1u);
                    occ = __shfl_sync(0xffffffffu, occ, 0);
                    if (occ == 0u) {
                        r = i;
                        break;
                    }
                    const VT *q = ev + (uint64_t)(occ - 1u) * U;
                    bool eq = true;
                    for (uint32_t w = lane; w < U; w += 32u) eq &= veq(__ldg(p + w), __ldg(q + w));
                    if (__all_sync(0xffffffffu, eq)) {
                        r = occ - 1u;
                        break;
                    }
                    slot = (slot + 1u) & task.slot_mask;
                }
                records = lane == 0u;
            }
            if (records) {
                const uint64_t b = task.elem + i, rb = task.elem + r;
                const int32_t d = (int32_t)i - (int32_t)r;
                s.rep[b] = d;
                atomicMin(s.first + rb, d);
                atomicXor(s.parity + (rb >> 5), 1u << (rb & 31u));
            }
        }
    }
}

// One block per lane; the survivors of a task are counted with one ballot per warp step and stored once.
__global__ void __launch_bounds__(kSegThreads)
seg_cancel_count_kernel(const SegCancelTask *__restrict__ tasks, const uint32_t n_tasks, const SegCancelScratch s,
                        uint32_t *__restrict__ live) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    pdl_enter();
    for (uint32_t t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < n_tasks; t += warps) {
        const SegCancelTask task = tasks[t];
        uint32_t running = 0;
        for (uint32_t i0 = task.first; i0 < task.end; i0 += 32u) {
            const uint32_t i = i0 + lane;
            const bool keep = i < task.end && cancel_survives(task.elem + i, s);
            running += __popc(__ballot_sync(0xffffffffu, keep));
        }
        if (lane == 0u) live[t] = running;
    }
}

// Groups of G lanes as in the insert pass; a surviving block's rank is the number of surviving group leaders below
// its own in the step's ballot, after the task's running count.
template <typename VT>
__global__ void __launch_bounds__(kSegThreads)
seg_cancel_write_kernel(const VT *__restrict__ v, VT *__restrict__ out, const uint32_t U, const uint32_t log2g,
                        const SegCancelTask *__restrict__ tasks, const uint32_t n_tasks, const SegCancelScratch s,
                        const uint64_t *__restrict__ base) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t G = 1u << log2g, sub = lane & (G - 1u), grp = lane >> log2g, B = 32u >> log2g;
    const uint32_t below = (1u << (grp * G)) - 1u;             // lanes of the groups before this one
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    pdl_enter();
    for (uint32_t t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t < n_tasks; t += warps) {
        const SegCancelTask task = tasks[t];
        const uint64_t pos = __ldg(base + t);
        uint32_t running = 0;
        for (uint32_t i0 = task.first; i0 < task.end; i0 += B) {
            const uint32_t i = i0 + grp;
            const bool keep = i < task.end && cancel_survives(task.elem + i, s);
            const uint32_t vote = __ballot_sync(0xffffffffu, keep && sub == 0u);
            if (keep) {
                const VT *p = v + (task.elem + i) * U;
                VT *o = out + (pos + running + __popc(vote & below)) * U;
                for (uint32_t w = sub; w < U; w += G) __stcs(o + w, __ldg(p + w));
            }
            running += __popc(vote);
        }
    }
}

// log2 of the group width G of the decrypt and cancellation kernels: the power of two >= U, up to 32
uint32_t group_log2(uint32_t U) {
    uint32_t log2g = 0;
    while (log2g < 5 && (1u << log2g) < U) ++log2g;
    return log2g;
}

uint32_t seg_grid(uint32_t n_tasks) {
    const uint32_t warps_per_cta = kSegThreads / 32;
    const uint64_t want = ((uint64_t)n_tasks + warps_per_cta - 1) / warps_per_cta;
    return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(want, (uint64_t)device_props().sm_count * kSegCtasPerSm));
}

}  // namespace

cudaError_t launch_seg_mul(uint64_t *out, uint32_t L, bool units16, const SegMulItem *items, const uint32_t *tasks,
                           uint32_t n_tasks, cudaStream_t stream) {
    if (n_tasks == 0) return cudaSuccess;
    count_launch();
    if (units16)
        return launch_kernel(seg_mul_kernel<uint4, kSegPlain>, seg_grid(n_tasks), kSegThreads, 0, stream,
                             reinterpret_cast<uint4 *>(out), L / 2, items, tasks, n_tasks, 0u, (uint32_t *)nullptr,
                             (const uint64_t *)nullptr);
    return launch_kernel(seg_mul_kernel<uint2, kSegPlain>, seg_grid(n_tasks), kSegThreads, 0, stream,
                         reinterpret_cast<uint2 *>(out), L, items, tasks, n_tasks, 0u, (uint32_t *)nullptr,
                         (const uint64_t *)nullptr);
}

cudaError_t launch_seg_mul_live(uint64_t *out, uint32_t L, bool units16, const SegMulItem *items,
                                const uint32_t *tasks, uint32_t n_tasks, uint32_t min_bits, uint32_t *live,
                                const uint64_t *base, cudaStream_t stream) {
    if (n_tasks == 0) return cudaSuccess;
    count_launch();
    const uint32_t grid = seg_grid(n_tasks);
    if (units16)
        return live ? launch_kernel(seg_mul_kernel<uint4, kSegCount>, grid, kSegThreads, 0, stream,
                                    reinterpret_cast<uint4 *>(out), L / 2, items, tasks, n_tasks, min_bits, live, base)
                    : launch_kernel(seg_mul_kernel<uint4, kSegWriteLive>, grid, kSegThreads, 0, stream,
                                    reinterpret_cast<uint4 *>(out), L / 2, items, tasks, n_tasks, min_bits, live, base);
    return live ? launch_kernel(seg_mul_kernel<uint2, kSegCount>, grid, kSegThreads, 0, stream,
                                reinterpret_cast<uint2 *>(out), L, items, tasks, n_tasks, min_bits, live, base)
                : launch_kernel(seg_mul_kernel<uint2, kSegWriteLive>, grid, kSegThreads, 0, stream,
                                reinterpret_cast<uint2 *>(out), L, items, tasks, n_tasks, min_bits, live, base);
}

cudaError_t launch_seg_decrypt(const uint64_t *v, uint32_t L, const uint64_t *mask, const uint64_t *off,
                               const SegDecTask *tasks, uint32_t n_tasks, uint64_t *counts, cudaStream_t stream) {
    if (n_tasks == 0) return cudaSuccess;
    const bool units16 = !(L & 1u) && ((reinterpret_cast<uintptr_t>(v) | reinterpret_cast<uintptr_t>(mask)) & 15u) == 0;
    const uint32_t U = units16 ? L / 2 : L;
    const uint32_t log2g = group_log2(U);
    count_launch();
    if (units16)
        return launch_kernel(seg_decrypt_kernel<uint4, false>, seg_grid(n_tasks), kSegThreads, 0, stream,
                             reinterpret_cast<const uint4 *>(v), U, log2g, reinterpret_cast<const uint4 *>(mask), off,
                             tasks, n_tasks, counts, (const SegPlane *)nullptr, (const uint32_t *)nullptr);
    return launch_kernel(seg_decrypt_kernel<uint2, false>, seg_grid(n_tasks), kSegThreads, 0, stream,
                         reinterpret_cast<const uint2 *>(v), U, log2g, reinterpret_cast<const uint2 *>(mask), off, tasks,
                         n_tasks, counts, (const SegPlane *)nullptr, (const uint32_t *)nullptr);
}

cudaError_t launch_seg_decrypt_uint(const SegPlane *planes, bool units16, uint32_t L, const uint64_t *mask,
                                    const SegDecTask *tasks, const uint32_t *task_plane, uint32_t n_tasks,
                                    uint64_t *values, cudaStream_t stream) {
    if (n_tasks == 0) return cudaSuccess;
    units16 = units16 && !(L & 1u) && (reinterpret_cast<uintptr_t>(mask) & 15u) == 0;
    const uint32_t U = units16 ? L / 2 : L;
    const uint32_t log2g = group_log2(U);
    count_launch();
    if (units16)
        return launch_kernel(seg_decrypt_kernel<uint4, true>, seg_grid(n_tasks), kSegThreads, 0, stream,
                             (const uint4 *)nullptr, U, log2g, reinterpret_cast<const uint4 *>(mask),
                             (const uint64_t *)nullptr, tasks, n_tasks, values, planes, task_plane);
    return launch_kernel(seg_decrypt_kernel<uint2, true>, seg_grid(n_tasks), kSegThreads, 0, stream,
                         (const uint2 *)nullptr, U, log2g, reinterpret_cast<const uint2 *>(mask),
                         (const uint64_t *)nullptr, tasks, n_tasks, values, planes, task_plane);
}

cudaError_t launch_seg_uint_pack(const uint64_t *counts, const uint64_t *entries, uint32_t n, uint64_t *values,
                                 cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    count_launch();
    const uint32_t grid = std::min<uint32_t>((n + kSegThreads - 1) / kSegThreads, device_props().sm_count * 4);
    return launch_kernel(seg_uint_pack_kernel, grid, kSegThreads, 0, stream, counts, entries, n, values);
}

cudaError_t launch_seg_cancel_insert(const uint64_t *v, uint32_t L, bool units16, const SegCancelTask *tasks,
                                     uint32_t n_tasks, const SegCancelScratch &s, cudaStream_t stream) {
    if (n_tasks == 0) return cudaSuccess;
    const uint32_t U = units16 ? L / 2 : L, log2g = group_log2(U);
    const uint32_t grid = seg_grid(n_tasks);
    count_launch();
    if (units16) {
        const uint4 *v4 = reinterpret_cast<const uint4 *>(v);
        return log2g == 5 ? launch_kernel(seg_cancel_insert_kernel<uint4, true>, grid, kSegThreads, 0, stream, v4, U,
                                          log2g, tasks, n_tasks, s)
                          : launch_kernel(seg_cancel_insert_kernel<uint4, false>, grid, kSegThreads, 0, stream, v4, U,
                                          log2g, tasks, n_tasks, s);
    }
    const uint2 *v2 = reinterpret_cast<const uint2 *>(v);
    return log2g == 5 ? launch_kernel(seg_cancel_insert_kernel<uint2, true>, grid, kSegThreads, 0, stream, v2, U, log2g,
                                      tasks, n_tasks, s)
                      : launch_kernel(seg_cancel_insert_kernel<uint2, false>, grid, kSegThreads, 0, stream, v2, U,
                                      log2g, tasks, n_tasks, s);
}

cudaError_t launch_seg_cancel_count(const SegCancelTask *tasks, uint32_t n_tasks, const SegCancelScratch &s,
                                    uint32_t *live, cudaStream_t stream) {
    if (n_tasks == 0) return cudaSuccess;
    count_launch();
    return launch_kernel(seg_cancel_count_kernel, seg_grid(n_tasks), kSegThreads, 0, stream, tasks, n_tasks, s, live);
}

cudaError_t launch_seg_cancel_write(const uint64_t *v, uint32_t L, bool units16, const SegCancelTask *tasks,
                                    uint32_t n_tasks, const SegCancelScratch &s, const uint64_t *base, uint64_t *out,
                                    cudaStream_t stream) {
    if (n_tasks == 0) return cudaSuccess;
    const uint32_t U = units16 ? L / 2 : L;
    count_launch();
    if (units16)
        return launch_kernel(seg_cancel_write_kernel<uint4>, seg_grid(n_tasks), kSegThreads, 0, stream,
                             reinterpret_cast<const uint4 *>(v), reinterpret_cast<uint4 *>(out), U, group_log2(U),
                             tasks, n_tasks, s, base);
    return launch_kernel(seg_cancel_write_kernel<uint2>, seg_grid(n_tasks), kSegThreads, 0, stream,
                         reinterpret_cast<const uint2 *>(v), reinterpret_cast<uint2 *>(out), U, group_log2(U), tasks,
                         n_tasks, s, base);
}

}  // namespace csgn
