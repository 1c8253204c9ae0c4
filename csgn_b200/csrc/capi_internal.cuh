// capi_internal.cuh -- shared by the translation units that implement include/csgn.h (capi.cu: library, buffers,
// the hot path, batches; capi_comm.cu: the peer communicator; capi_io.cu: save / load; capi_seg.cu: ciphertext arrays): the handle types, the
// process-wide state and the small helpers every entry point uses.  Internal: not part of the C ABI.
#pragma once

#include "../../include/csgn.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "kernels.cuh"

// ---------------------------------------------------------------------------
// handles
// ---------------------------------------------------------------------------
// A use of a buffer on a stream: `tick` is the library's operation counter when the use was enqueued.  The use is
// known to have completed once the host has synchronised that stream at a later tick (State::synced).
struct StreamMark {
    cudaStream_t s = nullptr;
    uint64_t tick = 0;
};

// Device storage shared by the buffers of one batched upload (csgn_buf_upload_batch): one allocation, one release.
struct csgn_slab {
    uint64_t *d = nullptr;
    uint64_t cap_words = 0;
    uint32_t refs = 0;
    std::vector<StreamMark> uses;   // every use of the freed views that may still be in flight, by stream
};

struct csgn_buf {
    uint64_t *d = nullptr;     // device words, n_blocks * L valid
    uint64_t n_blocks = 0;
    uint32_t L = 0;
    uint64_t cap_words = 0;    // allocated words (>= n_blocks*L); 0 for views
    bool owns = true;
    bool recycle = false;      // storage of an upload: goes back to the upload cache, not to the pool
    csgn_slab *slab = nullptr; // a view into a batched upload's shared storage (owns == false)
    // Lazy sum (csgn_concat_lazy): the value is the concatenation of these buffers, each kept alive by a reference,
    // and d == nullptr until some operation needs one dense array (flatten).  decrypt, permute and a product with the
    // sum as LEFT operand walk the segments instead.
    mutable std::vector<csgn_buf *> segs;
    uint32_t refs = 1;         // the caller's handle + one per lazy sum that refers to this buffer
    // An upload on the copy stream that may still be in flight.  EVERY stream that consumes the buffer waits for it
    // (ready_waited remembers which already did); the event goes back to the pool once it is known to have completed.
    mutable cudaEvent_t ready = nullptr;
    mutable std::vector<cudaStream_t> ready_waited;
    // Cross-stream ordering (batch lanes, automatic lanes, callers that multiplex streams): the stream of the last
    // write (allocation counts as one) and the streams that have read since.  A reader on another stream waits for the
    // writer, a writer for the writer and all readers, a free for everybody -- through an event recorded on the
    // other stream at that moment (no event is recorded on the fast path where everything stays on one stream).
    mutable StreamMark writer;
    mutable std::vector<StreamMark> readers;
};

// A decrypt whose count is read later (csgn_decrypt_deferred): device word, pinned host word, completion event.
struct csgn_result {
    uint64_t *h = nullptr;     // pinned host word the count is copied to
    uint64_t *d = nullptr;     // device word the fold writes
    cudaEvent_t done = nullptr;
    bool waited = false;
    uint32_t slot = 0;
};

struct csgn_key {
    uint64_t *d_positions = nullptr;  // D secret positions (for batched encryption)
    uint64_t *d_mask = nullptr;  // L words
    std::vector<uint64_t> h_mask;  // the same, host side (small masks ride in kernel parameters)
    uint64_t N = 0;
    uint32_t L = 0, D = 0;
};

struct csgn_perm {
    uint32_t *d_map = nullptr;   // N entries: (src_word << 6) | right_shift
    uint32_t *d_slice_map = nullptr;  // 64*L entries for the bit-sliced kernel (permute.cu), or null
    uint32_t *d_plane_map = nullptr;  // 64*L entries for the plane kernel (long blocks), or null
    uint64_t N = 0;
    uint32_t L = 0;
};

struct csgn_comm {
    int rank = 0, world = 1;
    uint64_t *box_local = nullptr;                 // this rank's mailbox (cudaMalloc: exportable)
    uint64_t *box[csgn::kPeerMaxWorld] = {};       // every rank's mailbox as mapped here
    bool ipc_opened[csgn::kPeerMaxWorld] = {};
    bool connected = false;
    uint64_t seq = 0;                              // sequence number of the next push
    uint64_t published = 0;                        // pushes [0, published) have been stored to the peers
    uint64_t *d_local_ring = nullptr;              // kPeerRing words: this rank's counts by slot
    uint64_t *d_status = nullptr;                  // [0] timeout flag, [1] blocking-call total
    uint64_t timeout_ns = 30ull * 1000 * 1000 * 1000;
    std::string rendezvous_file;                   // written by csgn_comm_connect_dir, removed on free
};

namespace csgn {
namespace detail {

struct State {
    bool inited = false;
    int device = -1;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;   // H2D uploads run here, overlapping kernels of the work stream
    // Batch entry points (csgn_*_batch) spread their independent items over these streams, forked from and joined
    // back into the current work stream, so that the tail of one kernel overlaps the ramp of the next item's.
    static constexpr int kMaxLanes = 4;
    cudaStream_t lane[kMaxLanes] = {};
    cudaEvent_t lane_done[kMaxLanes] = {};
    cudaEvent_t fork_point = nullptr;
    int n_lanes = 2;
    std::vector<cudaEvent_t> event_pool;
    // Storage of freed uploads, each with the event that marks its last use: an upload takes a slot whose event has
    // COMPLETED, so its copy can start at once on the copy stream and no allocation (which across streams may go to the
    // driver, milliseconds) sits on the steady-state path of "upload operands, multiply, decrypt, free".
    struct UploadSlot {
        uint64_t *d;
        uint64_t cap_words;
        cudaEvent_t freed;
    };
    std::vector<UploadSlot> upload_cache;
    uint64_t upload_cache_words = 0;
    uint64_t *d_scratch = nullptr;   // [2] blocking-call result, [4..6] checksum, [8 + 2k] fold scratch word of stream slot k
    uint64_t *h_result = nullptr;    // pinned, 8 words
    // Fold scratch: one word per STREAM (kernels of one stream never overlap their folds, PDL included, because a
    // kernel touches global memory only after griddepcontrol.wait); streams are given slots on first use.
    std::vector<cudaStream_t> scratch_streams;
    // Operation counter and, per stream, its value at the last host synchronisation of that stream.
    uint64_t tick = 1;
    std::vector<StreamMark> synced;
    // (consumer, producer, tick): `consumer` already waits for everything `producer` had enqueued at `tick`
    struct Waited {
        cudaStream_t consumer, producer;
        uint64_t tick;
    };
    std::vector<Waited> waited;
    // Automatic lanes (csgn_set_auto_lanes): independent operations of the drop-in API go to alternating internal
    // streams, ordered by the buffers they touch; in_batch: a LaneScope is active (it places the items itself).
    bool auto_lanes = false;
    bool in_batch = false;
    bool in_auto = false;
    uint32_t rr = 0;
    // deferred results: pinned host words + device words, handed out by slot
    uint64_t *h_results = nullptr, *d_results = nullptr;
    std::vector<uint32_t> free_results;
};
extern State g;
constexpr uint32_t kResultSlots = 4096;
constexpr uint32_t kScratchSlots = 256;

// Record the message of a failure for csgn_last_error() and return `code`.
int fail(int code, const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what);

#define CU(call)                                            \
    do {                                                    \
        cudaError_t e_ = (call);                            \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call); \
    } while (0)

#define NEED_INIT()                                                                              \
    do {                                                                                         \
        if (!g.inited) return fail(CSGN_ERR_NOT_INITIALIZED, "csgn_init has not been called");   \
        int cur_ = -1;                                                                           \
        if (cudaGetDevice(&cur_) != cudaSuccess || cur_ != g.device) CU(cudaSetDevice(g.device)); \
    } while (0)

int dev_alloc(uint64_t words, uint64_t **out, cudaStream_t stream = nullptr);   // stream-ordered, on the work stream by default
void dev_free(void *p);
cudaEvent_t take_event();
// Called for every operand of every operation, before the launch on the current stream g.stream: order that stream
// after a pending upload of `b` and after the uses of `b` on OTHER streams that conflict (read: the last writer;
// write: the last writer and every reader since), and record this use.
void acquire_read(const csgn_buf *b);
void acquire_write(const csgn_buf *b);
// The host has synchronised `s`: every use recorded on it so far is complete.
void note_synced(cudaStream_t s);
int new_buf(uint64_t n_blocks, uint32_t L, uint64_t cap_words, csgn_buf **out, cudaStream_t stream = nullptr);
// A lazy sum becomes one dense array on the current stream (no-op for a dense buffer).  Every entry point that needs
// `b->d` calls this first; the segment-aware ones (decrypt, permute, product with a lazy LEFT operand, concat) do not.
int need_dense(const csgn_buf *b);
inline bool is_rope(const csgn_buf *b) { return b && !b->segs.empty(); }
// The fold scratch word of the current stream.
uint64_t *fold_scratch();
// True inside a batch call or with automatic lanes: folds run next to other kernels (several shorter waves).
bool folds_overlap();

// Copy a host table of `bytes` bytes to fresh device memory (dev_alloc) on the current stream through the library's
// pinned staging, without a host synchronisation; the caller frees it with dev_free after the launches that read it.
int stage_to_device(const void *host, size_t bytes, void **out);
// The same copy into device memory `d` the caller already holds (a table that contains its own device address).
int stage_into(void *d, const void *host, size_t bytes);
// `bytes` of device memory `d` to `host` on the current stream, through the pinned staging, and wait for the copy.
int read_back(void *host, const void *d, size_t bytes);

// Scope of one batch call: item i runs with the work stream set to way i % n, where way 0 is the caller's own stream
// and ways 1.. are the library's side lanes, forked from the caller's stream on construction; join() makes the
// caller's stream wait for every side lane and restores it.
struct LaneScope {
    cudaStream_t home;
    int used = 1;
    bool active;
    bool was_in_batch;
    explicit LaneScope(uint32_t n_items) : home(g.stream), active(g.n_lanes > 1 && n_items > 1), was_in_batch(g.in_batch) {
        g.in_batch = true;
        if (!active) return;
        used = (int)std::min<uint32_t>(n_items, (uint32_t)g.n_lanes);
        cudaEventRecord(g.fork_point, home);
        for (int i = 1; i < used; ++i) cudaStreamWaitEvent(g.lane[i], g.fork_point, 0);
    }
    void enter(uint32_t item) {
        if (!active) return;
        const uint32_t way = item % (uint32_t)used;
        g.stream = way == 0 ? home : g.lane[way];
    }
    void join() {
        g.in_batch = was_in_batch;
        if (!active) return;
        g.stream = home;
        for (int i = 1; i < used; ++i) {
            cudaEventRecord(g.lane_done[i], g.lane[i]);
            cudaStreamWaitEvent(home, g.lane_done[i], 0);
        }
        active = false;
    }
    ~LaneScope() { join(); }
};

// Argument checks and the enqueue shared by the multiply entry points (capi.cu) and the sharded ones (capi_comm.cu).
int check_mul_operands(const csgn_buf *a, const csgn_buf *b);
int check_mul_out(const csgn_buf *a, const csgn_buf *b, const csgn_buf *out);
int check_key(const csgn_buf *a, const csgn_key *key);
// `out` convention of the fused entry points: null = count only; *out null = allocate; else write into *out.
int fused_out(const csgn_buf *a, const csgn_buf *b, csgn_buf **out, csgn_buf **dst, bool *allocated);
// Multiply (out != null) and/or fold the product under `key` (key != null) on the current stream; with a key the
// count goes to device_count and/or into the peer exchange `pp`.  One launch wherever a fused kernel exists.
int enqueue_mul(const csgn_buf *a, const csgn_buf *b, csgn_buf *out, const csgn_key *key, uint64_t *device_count,
                const csgn::PeerPush *pp);

// Scope of one operation of the drop-in API under automatic lanes (csgn_set_auto_lanes): the operation runs on the
// way where its largest operand was last written while that write may still be in flight (a chain stays on one
// stream and keeps its programmatic-dependent-launch overlap), or -- operands at rest -- on the next way round-robin,
// so that consecutive independent operations overlap.  Ordering comes from acquire_read / acquire_write.
struct AutoLane {
    cudaStream_t home;
    bool active = false;
    AutoLane(const csgn_buf *x, const csgn_buf *y = nullptr);
    ~AutoLane() {
        if (active) {
            g.stream = home;
            g.in_auto = false;
        }
    }
};

}  // namespace detail
}  // namespace csgn
