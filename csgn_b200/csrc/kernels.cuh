// kernels.cuh -- internal launch interface between the C ABI (capi.cu) and the
// sm_100a kernels.  Device pointers + sizes + stream; every launcher returns the
// cudaError_t of the launch and bumps the library's launch counter.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "peer.cuh"

namespace csgn {

struct DeviceProps {
    int device = -1;
    int sm_count = 148;
    int cc = 100;
    size_t smem_optin = 227 * 1024;
};
const DeviceProps &device_props();
void set_device_props(const DeviceProps &p);
void count_launch(unsigned n = 1);
uint64_t launches();
// true when the library was built with -DCSGN_BUILD_VARIANTS (the losing kernel variants kept for A/B sweeps)
bool build_has_variants();

// Integer environment knob (tuning sweeps only); `dflt` when unset or malformed.
long env_long(const char *name, long dflt);

// Fused multiply -> fold: what launch_mul needs to also count the satisfied blocks of the product.
struct MulFold {
    const uint64_t *mask;        // key mask, L words, device
    const uint64_t *host_mask;   // the same on the host (optional): small masks ride in the kernel parameters
    uint64_t *scratch;           // the launch's fold scratch word (zero between launches)
    uint64_t *count_out;         // device word for the total; may be null when `peer` is given
    const PeerPush *peer;        // optional: sharded decrypt (push / publish / collect in the same kernel)
    bool overlapped = false;     // the caller runs this launch next to other kernels (batch lanes, automatic lanes)
};
// K1  out[(i*T2+j)*L+k] = a[i*L+k] & b[j*L+k]        (reference src/Ciphertext.cpp:153-163)
// With `fold` the same launch also decrypt-folds the product (src/SecretKey.cpp:131-140) while its units are in
// registers; `out` may then be null (count only, nothing is stored).  cudaErrorNotSupported when a shape has no
// fused kernel (mul_fold_supported(L) is false): the caller multiplies and folds in two launches.
cudaError_t launch_mul(const uint64_t *a, uint64_t T1, const uint64_t *b, uint64_t T2, uint32_t L,
                       uint64_t *out, cudaStream_t stream, const MulFold *fold = nullptr);
bool mul_fold_supported(uint32_t L);

// K2  out = a || b                                     (reference src/Ciphertext.cpp:107-122)
// Either source may be null/empty; out may alias a (append in place) when a == out.
cudaError_t launch_concat(const uint64_t *a, uint64_t n_words_a, const uint64_t *b, uint64_t n_words_b,
                          uint64_t *out, cudaStream_t stream);

// Piece-table copy (ciphertext arrays: element-wise concat, gather, pack): destination units [dst[p], dst[p+1]) come
// from src[p], p < n_pieces; src and dst are device arrays, dst[n_pieces] == total_units.  Units of 16 bytes
// (units16: every source, the destination and every piece 16-byte granular) or 8 bytes.  One launch.
cudaError_t launch_piece_copy(const void *const *src, const uint64_t *dst, uint32_t n_pieces, uint64_t total_units,
                              bool units16, void *out, cudaStream_t stream);

// Ciphertext arrays (segments.cu).  Grouped multiply: work item k multiplies the `rows` blocks at device address a
// (its left operand's first row) by the t2 blocks at device address b (its right operand), into the rows*t2 blocks at
// block `out` of the output (blocks of L words); the operands may lie in any buffers.  A plain (copy) term is an item
// whose left operand is one all-ones block: AND with ~0 is the identity on every word.  A warp task is a run of
// consecutive items [task[t], task[t+1]).  units16: L is even and every operand, the output and the items are 16-byte
// aligned.  One launch.
struct SegMulItem {
    const uint64_t *a, *b;
    uint64_t out;
    uint32_t t2, rows;
};
static_assert(sizeof(SegMulItem) == 32, "SegMulItem is read as one 32-byte record");
cudaError_t launch_seg_mul(uint64_t *out, uint32_t L, bool units16, const SegMulItem *items, const uint32_t *tasks,
                           uint32_t n_tasks, cudaStream_t stream);
// The two passes of a compacting grouped multiply over the same items (a block survives when its L words hold at least
// min_bits set bits).  With `live`: live[k] = surviving blocks of item k, nothing else written.  Without: the surviving
// blocks of item k, in order, to blocks base[k], base[k] + 1, ... of `out`.  One launch each.
cudaError_t launch_seg_mul_live(uint64_t *out, uint32_t L, bool units16, const SegMulItem *items,
                                const uint32_t *tasks, uint32_t n_tasks, uint32_t min_bits, uint32_t *live,
                                const uint64_t *base, cudaStream_t stream);
// Segmented decrypt: a warp task walks blocks [first, end), which belong to elements [elem, elem_last] (element e =
// blocks [off[e], off[e+1]), off on the device), and adds each element's satisfied-block count to counts[e] (zeroed
// by the caller in stream order).  One launch.
struct SegDecTask {
    uint64_t first, end;
    uint64_t elem, elem_last;
};
cudaError_t launch_seg_decrypt(const uint64_t *v, uint32_t L, const uint64_t *mask, const uint64_t *off,
                               const SegDecTask *tasks, uint32_t n_tasks, uint64_t *counts, cudaStream_t stream);
// Cancellation (csgn_seg_cancel): a warp task is the blocks [first, end) of one element, whose first block is block
// `elem` of the array and whose open-addressing region is slots [slot, slot + slot_mask + 1) (a power of two).  Three
// passes over the same tasks, one launch each:
//   insert  every block finds its value's representative r (a slot holds an element-relative block index + 1, taken by
//           atomicCAS; equality is decided on all L words) and stores rep[b] = b - r; first[r] = min of b - r over the
//           value's blocks (atomicMin; the caller sets first to 0x7f7f7f7f), parity bit r ^= 1 (atomicXor; zeroed by the
//           caller, as are the slots);
//   count   live[t] = blocks b of task t with first[r] == b - r and parity bit r set (one plain store per task);
//   write   those blocks of task t, in order, to blocks base[t], base[t] + 1, ... of `out`.
// Blocks are numbered in the whole array; an element holds at most kCancelMaxBlocks blocks, so b - r fits an int32.
struct SegCancelTask {
    uint64_t elem, slot;
    uint32_t first, end, slot_mask, pad;
};
static_assert(sizeof(SegCancelTask) == 32, "SegCancelTask is read as one 32-byte record");
struct SegCancelScratch {
    uint32_t *slots;
    int32_t *first, *rep;
    uint32_t *parity;
};
constexpr uint64_t kCancelMaxBlocks = 1ull << 30;
cudaError_t launch_seg_cancel_insert(const uint64_t *v, uint32_t L, bool units16, const SegCancelTask *tasks,
                                     uint32_t n_tasks, const SegCancelScratch &s, cudaStream_t stream);
cudaError_t launch_seg_cancel_count(const SegCancelTask *tasks, uint32_t n_tasks, const SegCancelScratch &s,
                                    uint32_t *live, cudaStream_t stream);
cudaError_t launch_seg_cancel_write(const uint64_t *v, uint32_t L, bool units16, const SegCancelTask *tasks,
                                    uint32_t n_tasks, const SegCancelScratch &s, const uint64_t *base, uint64_t *out,
                                    cudaStream_t stream);

// out[0] = sum of in[0..n): the partial counts of a ciphertext held as several segments (a lazy sum)
cudaError_t launch_sum_words(const uint64_t *in, uint32_t n, uint64_t *out, cudaStream_t stream);

// K3  count of blocks with all_w((v[w] & M[w]) == M[w]) (reference src/SecretKey.cpp:126-140)
// `scratch` is one zero-initialised uint64 (count | CTA ticket << 40, fold.cuh) that the kernel
// leaves zeroed again; the total is written to *count_out (device memory).  `overlapped`: the caller runs
// this fold next to other kernels (batch lanes), so several shorter waves of CTAs back-fill better than one.
// `host_mask` (optional) is a host copy of the same L words: small masks ride in the
// kernel parameters instead of being fetched from global memory.
cudaError_t launch_decrypt_count(const uint64_t *v, uint64_t T, uint32_t L, const uint64_t *mask,
                                 const uint64_t *host_mask, uint64_t *scratch, uint64_t *count_out,
                                 cudaStream_t stream, const PeerPush *peer = nullptr, bool overlapped = false);
// `peer` (optional, sharded decrypt): the kernel's last CTA also pushes the count into every
// rank's mailbox and, when peer->collect_n > 0, collects the batch's totals (peer.cuh);
// count_out may then be null.  launch_peer_exchange does the push/collect without a fold.
cudaError_t launch_peer_exchange(const PeerPush &pp, bool do_push, uint64_t value, uint64_t *count_out,
                                 cudaStream_t stream);

// K4  out_bit[i] = in_bit[perm[i]] for every block     (reference src/Ciphertext.cpp:24-69)
// src_map[i] = (perm[i]>>6)<<6 | (63 - (perm[i]&63)): source word and right-shift.
// slice_map (optional, 64*L entries; see permute.cu) enables the bit-sliced tile kernel.
// plane_map (optional, 64*L entries): the same gather for the plane kernel (long blocks; slices kept in the tile's own
// 32 x 2L array): byte offset (j_src*2L + c_src)*4, or 4*32*2L (zero words) for pad bits.
cudaError_t launch_permute(const uint64_t *in, uint64_t T, uint32_t L, uint32_t N, const uint32_t *src_map,
                           const uint32_t *slice_map, const uint32_t *plane_map, uint64_t *out, cudaStream_t stream);
bool permute_sliced_supported(uint32_t L);
bool permute_plane_supported(uint32_t L);
// Words between consecutive slice rows of a tile in shared memory (32 slices + padding; 16-byte
// aligned rows, conflict-free 128-bit stores).  The slice map's byte offsets are built with it.
constexpr uint32_t kPermSliceStride = 36;

// n fresh encryptions (one block per plaintext bit) with Philox-4x32-10 keyed by `seed`; see encrypt.cu.
cudaError_t launch_encrypt_batch(const uint8_t *bits, uint64_t n, uint64_t first_block, uint32_t L, uint64_t pad_mask,
                                 const uint64_t *mask, const uint64_t *positions, uint32_t D, uint64_t seed,
                                 uint64_t *out, cudaStream_t stream);

// xor / wrapping sum / sum(w[i]*(2i+1)) of n_words words, accumulated into acc[0..2]
// (device, must be zeroed by the caller).
cudaError_t launch_checksum(const uint64_t *v, uint64_t n_words, uint64_t *acc, cudaStream_t stream);

}  // namespace csgn
