// capi.cu -- the C ABI of include/csgn.h: device state, buffer handles, and the
// thin argument checking in front of the kernel launchers.  No CPU compute path
// exists here: every operation either launches an sm_100a kernel or fails.
#include "capi_internal.cuh"

#include <atomic>
#include <cstdarg>
#if defined(__x86_64__) && !defined(__CUDA_ARCH__)
#include <emmintrin.h>
#define CSGN_HAVE_SSE2_STREAM 1
#endif

#ifdef CSGN_BUILD_VARIANTS
#define CSGN_VERSION_STRING "csgn-b200 0.2 (sm_100a) +variants"
#else
#define CSGN_VERSION_STRING "csgn-b200 0.2 (sm_100a)"
#endif

namespace csgn {
namespace detail {

State g;
DeviceProps g_props;
std::atomic<uint64_t> g_launches{0};
thread_local std::string t_error;

int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    t_error = buf;
    return code;
}

int cuda_fail(cudaError_t e, const char *what) {
    // leave the sticky-error state readable but do not hide it
    cudaGetLastError();
    return fail(e == cudaErrorMemoryAllocation ? CSGN_ERR_OUT_OF_MEMORY : CSGN_ERR_CUDA, "%s: %s (%s)", what,
                cudaGetErrorString(e), cudaGetErrorName(e));
}

// One fold scratch word per stream: folds of one stream never overlap (a kernel touches global memory only after
// griddepcontrol.wait, i.e. after its predecessor has completed), folds of different streams never share a word.
uint64_t *fold_scratch() {
    size_t i = 0;
    for (; i < g.scratch_streams.size(); ++i)
        if (g.scratch_streams[i] == g.stream) break;
    if (i == g.scratch_streams.size()) {
        if (i < kScratchSlots) {
            g.scratch_streams.push_back(g.stream);
        } else {
            // more distinct streams than slots (a caller cycling through hundreds of its own): share the last word,
            // ordering this stream after everything that may still use it
            i = kScratchSlots - 1;
            cudaDeviceSynchronize();
        }
    }
    return g.d_scratch + 8 + 2 * i;
}

bool folds_overlap() { return g.in_batch || g.auto_lanes; }

int dev_alloc(uint64_t words, uint64_t **out, cudaStream_t stream) {
    *out = nullptr;
    if (words == 0) return CSGN_OK;
    void *p = nullptr;
    cudaError_t e = cudaMallocAsync(&p, words * sizeof(uint64_t), stream ? stream : g.stream);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMallocAsync");
    *out = static_cast<uint64_t *>(p);
    return CSGN_OK;
}

void dev_free(void *p) {
    if (p) cudaFreeAsync(p, g.stream);
}

cudaEvent_t take_event() {
    if (!g.event_pool.empty()) {
        cudaEvent_t e = g.event_pool.back();
        g.event_pool.pop_back();
        return e;
    }
    cudaEvent_t e = nullptr;
    if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    return e;
}

constexpr uint64_t kUploadCacheMaxWords = (64ull << 20) / 8;      // per buffer: larger uploads are not latency-bound
constexpr uint64_t kUploadCacheTotalWords = (1ull << 30) / 8;     // all slots together
constexpr size_t kUploadCacheSlots = 512;

// Storage for an upload of `words` words: a cached slot whose last use has completed, or null.
uint64_t *take_upload_slot(uint64_t words, uint64_t *cap_words) {
    size_t best = SIZE_MAX;
    for (size_t i = 0; i < g.upload_cache.size(); ++i) {
        const State::UploadSlot &sl = g.upload_cache[i];
        if (sl.cap_words < words || sl.cap_words > 2 * words + 64) continue;
        if (best != SIZE_MAX && g.upload_cache[best].cap_words <= sl.cap_words) continue;
        if (cudaEventQuery(sl.freed) != cudaSuccess) {
            cudaGetLastError();      // cudaErrorNotReady is not an error
            continue;
        }
        best = i;
    }
    if (best == SIZE_MAX) return nullptr;
    State::UploadSlot sl = g.upload_cache[best];
    g.upload_cache[best] = g.upload_cache.back();
    g.upload_cache.pop_back();
    g.upload_cache_words -= sl.cap_words;
    g.event_pool.push_back(sl.freed);
    *cap_words = sl.cap_words;
    return sl.d;
}

// Hand the storage of a freed upload to the cache (true), or decline (the caller frees it).
bool give_upload_slot(uint64_t *d, uint64_t cap_words) {
    if (!d || cap_words == 0 || cap_words > kUploadCacheMaxWords || g.upload_cache.size() >= kUploadCacheSlots ||
        g.upload_cache_words + cap_words > kUploadCacheTotalWords)
        return false;
    cudaEvent_t e = nullptr;
    if (!g.event_pool.empty()) {
        e = g.event_pool.back();
        g.event_pool.pop_back();
    } else if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    if (cudaEventRecord(e, g.stream) != cudaSuccess) {      // everything enqueued so far may still read the buffer
        cudaGetLastError();
        g.event_pool.push_back(e);
        return false;
    }
    g.upload_cache.push_back({d, cap_words, e});
    g.upload_cache_words += cap_words;
    return true;
}

uint64_t synced_tick(cudaStream_t st) {
    for (const StreamMark &m : g.synced)
        if (m.s == st) return m.tick;
    return 0;
}

void note_synced(cudaStream_t st) {
    for (StreamMark &m : g.synced)
        if (m.s == st) {
            m.tick = g.tick - 1;         // every use recorded so far has a smaller tick
            return;
        }
    g.synced.push_back({st, g.tick - 1});
}

// Make `consumer` wait for everything `mark.s` had enqueued up to now (a superset of the marked use), unless that
// use is on the same stream, is known to have completed, or `consumer` already waits for it.
void wait_for_mark(cudaStream_t consumer, const StreamMark &mark) {
    if (!mark.s || mark.s == consumer || synced_tick(mark.s) >= mark.tick) return;
    for (State::Waited &w : g.waited)
        if (w.consumer == consumer && w.producer == mark.s) {
            if (w.tick >= mark.tick) return;
            cudaEvent_t e = take_event();
            if (!e) return;
            if (cudaEventRecord(e, mark.s) == cudaSuccess) cudaStreamWaitEvent(consumer, e, 0);
            else cudaGetLastError();     // the caller destroyed that stream: its work was enqueued before, nothing to order
            g.event_pool.push_back(e);
            w.tick = g.tick - 1;         // every use recorded so far has a smaller tick
            return;
        }
    cudaEvent_t e = take_event();
    if (!e) return;
    if (cudaEventRecord(e, mark.s) == cudaSuccess) cudaStreamWaitEvent(consumer, e, 0);
    else cudaGetLastError();
    g.event_pool.push_back(e);
    if (g.waited.size() < 256) g.waited.push_back({consumer, mark.s, g.tick - 1});
}

// A pending upload of `b`: the current stream waits for it unless it already does; once the copy is known to have
// completed the event is recycled.
void await_ready(const csgn_buf *b) {
    if (!b->ready) return;
    if (cudaEventQuery(b->ready) == cudaSuccess) {
        g.event_pool.push_back(b->ready);
        b->ready = nullptr;
        b->ready_waited.clear();
        return;
    }
    cudaGetLastError();      // cudaErrorNotReady is not an error
    for (cudaStream_t st : b->ready_waited)
        if (st == g.stream) return;
    cudaStreamWaitEvent(g.stream, b->ready, 0);
    b->ready_waited.push_back(g.stream);
}

void acquire_read(const csgn_buf *b) {
    if (!b) return;
    await_ready(b);
    wait_for_mark(g.stream, b->writer);
    const uint64_t now = g.tick++;
    if (b->writer.s == g.stream) {       // same stream as the writer: stream order already covers later writers' needs
        b->writer.tick = now;
        return;
    }
    for (StreamMark &m : b->readers)
        if (m.s == g.stream) {
            m.tick = now;
            return;
        }
    b->readers.push_back({g.stream, now});
}

void acquire_write(const csgn_buf *b) {
    if (!b) return;
    await_ready(b);
    wait_for_mark(g.stream, b->writer);
    for (const StreamMark &m : b->readers) wait_for_mark(g.stream, m);
    b->readers.clear();
    b->writer = {g.stream, g.tick++};
}

// Before storage is handed back (pool or upload cache) on the CURRENT stream: that stream first waits for every
// other stream that used the words (the caller multiplexes streams, or the library's lanes did).
void order_after_all_uses(const csgn_buf *b) {
    wait_for_mark(g.stream, b->writer);
    for (const StreamMark &m : b->readers) wait_for_mark(g.stream, m);
}

AutoLane::AutoLane(const csgn_buf *x, const csgn_buf *y) : home(g.stream) {
    if (!g.auto_lanes || g.in_batch || g.in_auto || g.n_lanes < 2) return;
    g.in_auto = true;
    // ways: 0 = the caller's stream, 1.. = the library's side lanes
    const csgn_buf *big = (y && (!x || y->n_blocks > x->n_blocks)) ? y : x;
    cudaStream_t pick = nullptr;
    if (big && big->writer.s && synced_tick(big->writer.s) < big->writer.tick) {
        if (big->writer.s == home) pick = home;
        for (int i = 1; i < g.n_lanes && !pick; ++i)
            if (big->writer.s == g.lane[i]) pick = g.lane[i];
    }
    if (!pick) {
        const uint32_t way = g.rr++ % (uint32_t)g.n_lanes;
        pick = way == 0 ? home : g.lane[way];
    }
    g.stream = pick;
    active = true;
}

int new_buf(uint64_t n_blocks, uint32_t L, uint64_t cap_words, csgn_buf **out, cudaStream_t stream) {
    if (L == 0) return fail(CSGN_ERR_INVALID_ARGUMENT, "words per block must be > 0");
    if (n_blocks > (UINT64_MAX / 8) / L) return fail(CSGN_ERR_INVALID_ARGUMENT, "block count overflows");
    csgn_buf *b = new csgn_buf;
    b->n_blocks = n_blocks;
    b->L = L;
    b->cap_words = std::max<uint64_t>(cap_words, n_blocks * L);
    int rc = dev_alloc(b->cap_words, &b->d, stream);
    if (rc != CSGN_OK) {
        delete b;
        return rc;
    }
    b->writer = {stream ? stream : g.stream, g.tick++};      // the allocation is ordered on that stream
    *out = b;
    return CSGN_OK;
}

// Copy the words of `src` (dense or a lazy sum) to dst on the current stream.
int copy_words_into(const csgn_buf *src, uint64_t *dst) {
    if (!is_rope(src)) {
        acquire_read(src);
        cudaError_t e = launch_concat(src->d, src->n_blocks * src->L, nullptr, 0, dst, g.stream);
        return e == cudaSuccess ? CSGN_OK : cuda_fail(e, "copy kernel");
    }
    uint64_t off = 0;
    for (size_t i = 0; i < src->segs.size(); i += 2) {          // two segments per launch (the copy kernel has two sources)
        const csgn_buf *x = src->segs[i], *y = i + 1 < src->segs.size() ? src->segs[i + 1] : nullptr;
        acquire_read(x);
        if (y) acquire_read(y);
        const uint64_t nx = x->n_blocks * x->L, ny = y ? y->n_blocks * y->L : 0;
        cudaError_t e = launch_concat(x->d, nx, y ? y->d : nullptr, ny, dst + off, g.stream);
        if (e != cudaSuccess) return cuda_fail(e, "copy kernel");
        off += nx + ny;
    }
    return CSGN_OK;
}

void drop_segments(const csgn_buf *b) {
    std::vector<csgn_buf *> segs;
    segs.swap(b->segs);
    for (csgn_buf *x : segs) csgn_buf_free(x);
}

int need_dense(const csgn_buf *b) {
    if (!is_rope(b)) return CSGN_OK;
    csgn_buf *m = const_cast<csgn_buf *>(b);
    uint64_t *d = nullptr;
    const uint64_t words = b->n_blocks * b->L;
    int rc = dev_alloc(words, &d);
    if (rc != CSGN_OK) return rc;
    rc = copy_words_into(b, d);
    if (rc != CSGN_OK) {
        dev_free(d);
        return rc;
    }
    m->d = d;
    m->cap_words = words;
    m->owns = true;
    m->writer = {g.stream, g.tick++};
    m->readers.clear();
    drop_segments(b);          // the segments' storage is released in stream order, after the copies that read it
    return CSGN_OK;
}

}  // namespace detail

using namespace detail;

const DeviceProps &device_props() { return g_props; }
void set_device_props(const DeviceProps &p) { g_props = p; }
void count_launch(unsigned n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
uint64_t launches() { return g_launches.load(std::memory_order_relaxed); }

// Tuning knobs (CSGN_MUL_*, CSGN_DEC_*, CSGN_PERM_*, CSGN_PDL ...) are looked up only when
// CSGN_TUNING is set in the environment at csgn_init: a production launch does not pay a
// dozen getenv() scans (~4 us per launch), tests and tools/ opt in.
static bool g_tuning = true;   // until csgn_init has looked

long env_long(const char *name, long dflt) {
    if (!g_tuning) return dflt;
    const char *s = std::getenv(name);
    if (!s || !*s) return dflt;
    char *end = nullptr;
    long v = std::strtol(s, &end, 10);
    return (end && *end == 0) ? v : dflt;
}

}  // namespace csgn

// Pinned staging for csgn_buf_upload_copy: the caller's words are copied here by the host and go to the device
// from here, so the call needs no synchronisation and the caller may reuse its array at once.
namespace {
struct StagingSlot {
    void *p;
    size_t cap;
    cudaEvent_t done;     // the H2D copy that last read this slot
};
std::vector<StagingSlot> g_staging;
size_t g_staging_bytes = 0;
constexpr size_t kStagingMaxTotal = 512ull << 20, kStagingMaxOne = 64ull << 20;

StagingSlot *take_staging(size_t bytes) {
    StagingSlot *best = nullptr;
    for (StagingSlot &sl : g_staging) {
        if (sl.cap < bytes || (best && best->cap <= sl.cap)) continue;
        if (cudaEventQuery(sl.done) != cudaSuccess) {
            cudaGetLastError();
            continue;
        }
        best = &sl;
    }
    if (best) return best;
    size_t cap = 64 << 10;
    while (cap < bytes) cap <<= 1;
    if (g_staging_bytes + cap > kStagingMaxTotal) return nullptr;
    StagingSlot sl = {nullptr, cap, nullptr};
    if (cudaHostAlloc(&sl.p, cap, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    if (cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming) != cudaSuccess) {
        cudaGetLastError();
        cudaFreeHost(sl.p);
        return nullptr;
    }
    g_staging.push_back(sl);
    g_staging_bytes += cap;
    return &g_staging.back();
}
}  // namespace

using namespace csgn;
using namespace csgn::detail;

// ---------------------------------------------------------------------------
// library
// ---------------------------------------------------------------------------
extern "C" {

int csgn_init(int device) {
    csgn::g_tuning = true;
    if (device < 0) device = (int)env_long("CSGN_DEVICE", env_long("LOCAL_RANK", 0));
    csgn::g_tuning = std::getenv("CSGN_TUNING") != nullptr;
    if (g.inited) {
        if (g.device == device) return CSGN_OK;
        return fail(CSGN_ERR_INVALID_ARGUMENT, "already bound to device %d (one process per GPU)", g.device);
    }
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(CSGN_ERR_NO_DEVICE, "no CUDA device visible (%s); this engine has no CPU path",
                    e == cudaSuccess ? "count = 0" : cudaGetErrorString(e));
    }
    if (device >= n) return fail(CSGN_ERR_NO_DEVICE, "device %d requested, %d visible", device, n);
    CU(cudaSetDevice(device));
    cudaDeviceProp p;
    CU(cudaGetDeviceProperties(&p, device));
    if (p.major != 10)
        return fail(CSGN_ERR_NO_DEVICE, "device %d is sm_%d%d; the kernels are built for sm_100a (B200) only",
                    device, p.major, p.minor);
    DeviceProps dp;
    dp.device = device;
    dp.sm_count = p.multiProcessorCount;
    dp.cc = p.major * 10 + p.minor;
    dp.smem_optin = p.sharedMemPerBlockOptin;
    set_device_props(dp);

    CU(cudaStreamCreateWithFlags(&g.own_stream, cudaStreamNonBlocking));
    g.stream = g.own_stream;
    CU(cudaStreamCreateWithFlags(&g.copy_stream, cudaStreamNonBlocking));
    {
        const char *e = std::getenv("CSGN_LANES");
        g.n_lanes = e && *e ? std::max(1, std::min((int)State::kMaxLanes, std::atoi(e))) : 2;
    }
    for (int i = 0; i < g.n_lanes; ++i) {
        CU(cudaStreamCreateWithFlags(&g.lane[i], cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&g.lane_done[i], cudaEventDisableTiming));
    }
    CU(cudaEventCreateWithFlags(&g.fork_point, cudaEventDisableTiming));
    // keep freed blocks in the pool: a*b chains reuse them without going to the driver
    cudaMemPool_t pool;
    CU(cudaDeviceGetDefaultMemPool(&pool, device));
    uint64_t keep = UINT64_MAX;
    CU(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    // Callers may enqueue independent ciphertexts on several streams (csgn_set_stream) so that kernels overlap.  An
    // allocation must then never make its stream wait for another stream's pending frees -- that would serialise the
    // streams again -- so the pool only reuses memory whose free has completed or is ordered by the caller's own events.
    int off = 0;
    CU(cudaMemPoolSetAttribute(pool, cudaMemPoolReuseAllowInternalDependencies, &off));
    CU(cudaMalloc(reinterpret_cast<void **>(&g.d_scratch), (8 + 2 * kScratchSlots) * sizeof(uint64_t)));
    CU(cudaMemset(g.d_scratch, 0, (8 + 2 * kScratchSlots) * sizeof(uint64_t)));
    CU(cudaHostAlloc(reinterpret_cast<void **>(&g.h_result), 8 * sizeof(uint64_t), cudaHostAllocDefault));
    CU(cudaMalloc(reinterpret_cast<void **>(&g.d_results), kResultSlots * sizeof(uint64_t)));
    CU(cudaHostAlloc(reinterpret_cast<void **>(&g.h_results), kResultSlots * sizeof(uint64_t), cudaHostAllocDefault));
    g.free_results.clear();
    for (uint32_t i = kResultSlots; i > 0; --i) g.free_results.push_back(i - 1);
    {
        const char *e = std::getenv("CSGN_AUTO_LANES");
        g.auto_lanes = e && *e && std::atoi(e) != 0;
    }
    g.device = device;
    g.inited = true;
    return CSGN_OK;
}

int csgn_shutdown(void) {
    if (!g.inited) return CSGN_OK;
    cudaSetDevice(g.device);
    cudaDeviceSynchronize();
    for (const State::UploadSlot &sl : g.upload_cache) {
        cudaFreeAsync(sl.d, g.stream);
        cudaEventDestroy(sl.freed);
    }
    cudaStreamSynchronize(g.stream);
    for (StagingSlot &sl : g_staging) {
        cudaFreeHost(sl.p);
        cudaEventDestroy(sl.done);
    }
    g_staging.clear();
    g_staging_bytes = 0;
    cudaFree(g.d_scratch);
    cudaFreeHost(g.h_result);
    if (g.d_results) cudaFree(g.d_results);
    if (g.h_results) cudaFreeHost(g.h_results);
    for (cudaEvent_t e : g.event_pool) cudaEventDestroy(e);
    for (int i = 0; i < State::kMaxLanes; ++i) {
        if (g.lane[i]) {
            cudaStreamSynchronize(g.lane[i]);
            cudaStreamDestroy(g.lane[i]);
        }
        if (g.lane_done[i]) cudaEventDestroy(g.lane_done[i]);
    }
    if (g.fork_point) cudaEventDestroy(g.fork_point);
    cudaStreamDestroy(g.copy_stream);
    cudaStreamDestroy(g.own_stream);
    g = State();
    return CSGN_OK;
}

int csgn_is_initialized(void) { return g.inited ? 1 : 0; }
const char *csgn_last_error(void) { return t_error.c_str(); }
const char *csgn_version(void) { return CSGN_VERSION_STRING; }

int csgn_device_info(int *sm_count, uint64_t *hbm_total, uint64_t *hbm_free, int *cc) {
    NEED_INIT();
    size_t fr = 0, tot = 0;
    CU(cudaMemGetInfo(&fr, &tot));
    if (sm_count) *sm_count = device_props().sm_count;
    if (hbm_total) *hbm_total = tot;
    if (hbm_free) *hbm_free = fr;
    if (cc) *cc = device_props().cc;
    return CSGN_OK;
}

int csgn_set_stream(void *cuda_stream) {
    NEED_INIT();
    g.stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : g.own_stream;
    return CSGN_OK;
}

int csgn_set_auto_lanes(int on) {
    NEED_INIT();
    g.auto_lanes = on != 0;
    return CSGN_OK;
}

int csgn_get_auto_lanes(void) { return g.inited && g.auto_lanes ? 1 : 0; }

void *csgn_get_stream(void) { return g.inited ? static_cast<void *>(g.stream) : nullptr; }

int csgn_sync(void) {
    NEED_INIT();
    CU(cudaStreamSynchronize(g.copy_stream));   // uploads whose buffers nobody has consumed yet
    CU(cudaStreamSynchronize(g.stream));
    note_synced(g.copy_stream);
    note_synced(g.stream);
    for (int i = 1; i < g.n_lanes; ++i) {       // work the library itself placed on its side lanes (automatic lanes)
        CU(cudaStreamSynchronize(g.lane[i]));
        note_synced(g.lane[i]);
    }
    return CSGN_OK;
}

uint64_t csgn_launch_count(void) { return launches(); }

uint32_t csgn_words_per_block(uint64_t N) { return (uint32_t)(N / 64 + (N % 64 ? 1 : 0)); }

int csgn_host_alloc(size_t bytes, void **out) {
    NEED_INIT();
    if (!out) return fail(CSGN_ERR_INVALID_ARGUMENT, "null output pointer");
    CU(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
    return CSGN_OK;
}

int csgn_host_free(void *p) {
    NEED_INIT();
    if (p) CU(cudaFreeHost(p));
    return CSGN_OK;
}

// ---------------------------------------------------------------------------
// buffers
// ---------------------------------------------------------------------------
int csgn_buf_alloc(uint64_t n_blocks, uint32_t L, csgn_buf **out) {
    NEED_INIT();
    if (!out) return fail(CSGN_ERR_INVALID_ARGUMENT, "null output handle");
    return new_buf(n_blocks, L, 0, out);
}

int csgn_buf_upload(const uint64_t *host_words, uint64_t n_blocks, uint32_t L, csgn_buf **out) {
    NEED_INIT();
    if (!out) return fail(CSGN_ERR_INVALID_ARGUMENT, "null output handle");
    if (n_blocks && !host_words) return fail(CSGN_ERR_INVALID_ARGUMENT, "null host words");
    if (L == 0) return fail(CSGN_ERR_INVALID_ARGUMENT, "words per block must be > 0");
    // Allocation and copy are ordered on the copy stream, so an upload overlaps whatever the work
    // stream is running; the first consumer on the work stream waits for the `ready` event.
    csgn_buf *b = nullptr;
    uint64_t cap = 0;
    uint64_t *cached = (n_blocks && n_blocks <= kUploadCacheMaxWords / L) ? take_upload_slot(n_blocks * L, &cap) : nullptr;
    if (cached) {
        b = new csgn_buf;
        b->d = cached;
        b->n_blocks = n_blocks;
        b->L = L;
        b->cap_words = cap;
        b->writer = {g.copy_stream, g.tick++};
    } else {
        int rc = new_buf(n_blocks, L, 0, &b, g.copy_stream);
        if (rc != CSGN_OK) return rc;
    }
    b->recycle = true;
    if (n_blocks) {
        cudaError_t e = cudaMemcpyAsync(b->d, host_words, n_blocks * L * sizeof(uint64_t), cudaMemcpyHostToDevice,
                                        g.copy_stream);
        if (e == cudaSuccess) {
            b->ready = take_event();
            e = b->ready ? cudaEventRecord(b->ready, g.copy_stream) : cudaStreamSynchronize(g.copy_stream);
            // the `ready` event is the precise ordering for the copy; the writer mark on the copy stream is dropped so
            // that consumers do not also wait for LATER uploads queued behind this one
            if (e == cudaSuccess) b->writer = StreamMark();
        }
        if (e != cudaSuccess) {
            csgn_buf_free(b);
            return cuda_fail(e, "cudaMemcpyAsync(H2D)");
        }
    }
    *out = b;
    return CSGN_OK;
}

namespace {
// The caller's words -> pinned staging.  The destination is written once and next read by the copy engine, never by this
// core: streaming stores skip the read-for-ownership of every destination line (an ordinary memcpy of 160 KB into a slot that
// has left the cache reads the slot first), 20 -> 16 us per 160 KB on the build host.
void copy_to_staging(void *dst, const void *src, size_t bytes) {
#ifdef CSGN_HAVE_SSE2_STREAM
    if (bytes >= (32u << 10)) {
        char *d = static_cast<char *>(dst);
        const char *s = static_cast<const char *>(src);
        size_t head = (16u - (reinterpret_cast<uintptr_t>(d) & 15u)) & 15u;
        memcpy(d, s, head);
        d += head, s += head, bytes -= head;
        const size_t n = bytes / 64;
        for (size_t i = 0; i < n; ++i, s += 64, d += 64) {
            const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i *>(s));
            const __m128i b = _mm_loadu_si128(reinterpret_cast<const __m128i *>(s + 16));
            const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i *>(s + 32));
            const __m128i e = _mm_loadu_si128(reinterpret_cast<const __m128i *>(s + 48));
            _mm_stream_si128(reinterpret_cast<__m128i *>(d), a);
            _mm_stream_si128(reinterpret_cast<__m128i *>(d + 16), b);
            _mm_stream_si128(reinterpret_cast<__m128i *>(d + 32), c);
            _mm_stream_si128(reinterpret_cast<__m128i *>(d + 48), e);
        }
        memcpy(d, s, bytes - n * 64);
        _mm_sfence();            // the stores are globally visible before the copy engine is told about them
        return;
    }
#endif
    memcpy(dst, src, bytes);
}
}  // namespace

}  // extern "C"

namespace csgn {
namespace detail {

// A small host table (work items, offsets) to fresh device memory on the current stream, through the pinned staging:
// no host synchronisation, and the caller may reuse its array at once.  Tables beyond the staging limit are copied
// straight from the caller's memory, and the call waits for that copy.
int stage_into(void *d, const void *host, size_t bytes) {
    if (bytes == 0) return CSGN_OK;
    StagingSlot *sl = bytes <= kStagingMaxOne ? take_staging(bytes) : nullptr;
    cudaError_t e;
    if (sl) {
        copy_to_staging(sl->p, host, bytes);
        e = cudaMemcpyAsync(d, sl->p, bytes, cudaMemcpyHostToDevice, g.stream);
        cudaEventRecord(sl->done, g.stream);
    } else {
        e = cudaMemcpyAsync(d, host, bytes, cudaMemcpyHostToDevice, g.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g.stream);
        if (e == cudaSuccess) note_synced(g.stream);
    }
    return e == cudaSuccess ? CSGN_OK : cuda_fail(e, "table upload");
}

int stage_to_device(const void *host, size_t bytes, void **out) {
    *out = nullptr;
    if (bytes == 0) return CSGN_OK;
    uint64_t *d = nullptr;
    int rc = dev_alloc((bytes + 7) / 8, &d);
    if (rc != CSGN_OK) return rc;
    rc = stage_into(d, host, bytes);
    if (rc != CSGN_OK) {
        dev_free(d);
        return rc;
    }
    *out = d;
    return CSGN_OK;
}

int read_back(void *host, const void *d, size_t bytes) {
    if (bytes == 0) return CSGN_OK;
    StagingSlot *sl = bytes <= kStagingMaxOne ? take_staging(bytes) : nullptr;
    cudaError_t e = cudaMemcpyAsync(sl ? sl->p : host, d, bytes, cudaMemcpyDeviceToHost, g.stream);
    if (e == cudaSuccess && sl) e = cudaEventRecord(sl->done, g.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g.stream);
    if (e != cudaSuccess) return cuda_fail(e, "table read-back");
    note_synced(g.stream);
    if (sl) memcpy(host, sl->p, bytes);
    return CSGN_OK;
}

}  // namespace detail
}  // namespace csgn

extern "C" {

int csgn_buf_upload_copy(const uint64_t *host_words, uint64_t n_blocks, uint32_t L, csgn_buf **out) {
    NEED_INIT();
    if (L == 0) return fail(CSGN_ERR_INVALID_ARGUMENT, "words per block must be > 0");
    if (n_blocks > (UINT64_MAX / 8) / L) return fail(CSGN_ERR_INVALID_ARGUMENT, "block count overflows");
    const size_t bytes = (size_t)n_blocks * L * sizeof(uint64_t);
    StagingSlot *sl = (bytes && bytes <= kStagingMaxOne && host_words) ? take_staging(bytes) : nullptr;
    if (!sl) {
        // too large for staging (or none free): copy straight from the caller's memory and wait for it
        int rc = csgn_buf_upload(host_words, n_blocks, L, out);
        if (rc != CSGN_OK) return rc;
        CU(cudaStreamSynchronize(g.copy_stream));
        note_synced(g.copy_stream);
        return CSGN_OK;
    }
    copy_to_staging(sl->p, host_words, bytes);
    int rc = csgn_buf_upload(static_cast<const uint64_t *>(sl->p), n_blocks, L, out);
    // whatever happened, later users of the slot wait for everything the copy stream holds so far
    cudaEventRecord(sl->done, g.copy_stream);
    return rc;
}

int csgn_buf_upload_batch(const uint64_t *const *host_words, const uint64_t *n_blocks, uint32_t n, uint32_t L,
                          csgn_buf **out) {
    NEED_INIT();
    if (n == 0) return CSGN_OK;
    if (!host_words || !n_blocks || !out) return fail(CSGN_ERR_INVALID_ARGUMENT, "null argument");
    if (L == 0) return fail(CSGN_ERR_INVALID_ARGUMENT, "words per block must be > 0");
    // one slab for the n operands (each 256-byte aligned), copies back to back on the copy stream
    constexpr uint64_t kAlignWords = 32;
    std::vector<uint64_t> off(n);
    uint64_t total = 0;
    for (uint32_t i = 0; i < n; ++i) {
        if (n_blocks[i] && !host_words[i]) return fail(CSGN_ERR_INVALID_ARGUMENT, "null host words (operand %u)", i);
        if (n_blocks[i] > (UINT64_MAX / 16) / L) return fail(CSGN_ERR_INVALID_ARGUMENT, "block count overflows");
        off[i] = total;
        total += (n_blocks[i] * L + kAlignWords - 1) / kAlignWords * kAlignWords;
    }
    if (total == 0) total = kAlignWords;
    csgn_slab *sl = new csgn_slab;
    uint64_t cap = 0;
    sl->d = total <= kUploadCacheMaxWords ? take_upload_slot(total, &cap) : nullptr;
    if (sl->d) sl->cap_words = cap;
    else {
        int rc = dev_alloc(total, &sl->d, g.copy_stream);
        if (rc != CSGN_OK) {
            delete sl;
            return rc;
        }
        sl->cap_words = total;
    }
    std::vector<void *> dsts, srcs;
    std::vector<size_t> sizes;
    for (uint32_t i = 0; i < n; ++i)
        if (n_blocks[i]) {
            dsts.push_back(sl->d + off[i]);
            srcs.push_back(const_cast<uint64_t *>(host_words[i]));
            sizes.push_back((size_t)n_blocks[i] * L * sizeof(uint64_t));
        }
    // operands that follow one another in host memory AND in the slab (rows of one pinned array whose size is a
    // multiple of 256 bytes) travel as one copy: fewer, larger copies
    cudaError_t e = cudaSuccess;
    for (size_t i = 0; i < dsts.size() && e == cudaSuccess;) {
        size_t j = i + 1, bytes = sizes[i];
        while (j < dsts.size() && static_cast<char *>(srcs[i]) + bytes == static_cast<char *>(srcs[j]) &&
               static_cast<char *>(dsts[i]) + bytes == static_cast<char *>(dsts[j])) {
            bytes += sizes[j];
            ++j;
        }
        e = cudaMemcpyAsync(dsts[i], srcs[i], bytes, cudaMemcpyHostToDevice, g.copy_stream);
        i = j;
    }
    if (e != cudaSuccess) {
        cudaStreamSynchronize(g.copy_stream);
        dev_free(sl->d);
        delete sl;
        return cuda_fail(e, "cudaMemcpyAsync(H2D batch)");
    }
    // the views are ordered after the copies through their writer mark on the copy stream: the first consumer on a
    // stream records ONE event there for the whole batch (wait_for_mark remembers what a stream already waits for)
    const uint64_t tick = g.tick++;
    for (uint32_t i = 0; i < n; ++i) {
        csgn_buf *b = new csgn_buf;
        b->d = sl->d + off[i];
        b->n_blocks = n_blocks[i];
        b->L = L;
        b->cap_words = 0;
        b->owns = false;
        b->slab = sl;
        b->writer = {g.copy_stream, tick};
        out[i] = b;
    }
    sl->refs = n;
    return CSGN_OK;
}

int csgn_buf_wrap(void *device_words, uint64_t n_blocks, uint32_t L, csgn_buf **out) {
    NEED_INIT();
    if (!out || L == 0) return fail(CSGN_ERR_INVALID_ARGUMENT, "bad view arguments");
    if (n_blocks && !device_words) return fail(CSGN_ERR_INVALID_ARGUMENT, "null device pointer");
    if (reinterpret_cast<uintptr_t>(device_words) & 7u)
        return fail(CSGN_ERR_INVALID_ARGUMENT, "device pointer must be 8-byte aligned");
    csgn_buf *b = new csgn_buf;
    b->d = static_cast<uint64_t *>(device_words);
    b->n_blocks = n_blocks;
    b->L = L;
    b->cap_words = 0;
    b->owns = false;
    b->writer = {g.stream, g.tick++};   // whatever produced the words was enqueued on the caller's current stream
    *out = b;
    return CSGN_OK;
}

int csgn_buf_clone(const csgn_buf *src, csgn_buf **out) {
    NEED_INIT();
    if (!src || !out) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    csgn_buf *b = nullptr;
    AutoLane lane(src);
    int rc = new_buf(src->n_blocks, src->L, 0, &b);
    if (rc != CSGN_OK) return rc;
    rc = copy_words_into(src, b->d);       // a lazy sum is copied segment by segment
    if (rc != CSGN_OK) {
        csgn_buf_free(b);
        return rc;
    }
    *out = b;
    return CSGN_OK;
}

int csgn_buf_slice(const csgn_buf *src, uint64_t first_block, uint64_t n_blocks, csgn_buf **out) {
    NEED_INIT();
    if (!src || !out) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    if (first_block > src->n_blocks || n_blocks > src->n_blocks - first_block)
        return fail(CSGN_ERR_INVALID_ARGUMENT, "block range [%llu,+%llu) outside %llu blocks",
                    (unsigned long long)first_block, (unsigned long long)n_blocks, (unsigned long long)src->n_blocks);
    csgn_buf *b = nullptr;
    AutoLane lane(src);
    int rc = need_dense(src);
    if (rc != CSGN_OK) return rc;
    rc = new_buf(n_blocks, src->L, 0, &b);
    if (rc != CSGN_OK) return rc;
    acquire_read(src);
    cudaError_t e = launch_concat(src->d + first_block * src->L, n_blocks * src->L, nullptr, 0, b->d, g.stream);
    if (e != cudaSuccess) {
        csgn_buf_free(b);
        return cuda_fail(e, "slice kernel");
    }
    *out = b;
    return CSGN_OK;
}

int csgn_buf_download_range(const csgn_buf *buf, uint64_t first_block, uint64_t n_blocks, uint64_t *host_words) {
    NEED_INIT();
    if (!buf) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    if (first_block > buf->n_blocks || n_blocks > buf->n_blocks - first_block)
        return fail(CSGN_ERR_INVALID_ARGUMENT, "block range [%llu,+%llu) outside %llu blocks",
                    (unsigned long long)first_block, (unsigned long long)n_blocks, (unsigned long long)buf->n_blocks);
    if (n_blocks == 0) return CSGN_OK;
    if (!host_words) return fail(CSGN_ERR_INVALID_ARGUMENT, "null host destination");
    {
        int rc = need_dense(buf);
        if (rc != CSGN_OK) return rc;
    }
    acquire_read(buf);
    CU(cudaMemcpyAsync(host_words, buf->d + first_block * buf->L, n_blocks * buf->L * sizeof(uint64_t),
                       cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    note_synced(g.stream);
    return CSGN_OK;
}

int csgn_buf_download(const csgn_buf *buf, uint64_t *host_words) {
    if (!buf) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    return csgn_buf_download_range(buf, 0, buf->n_blocks, host_words);
}

namespace {
// A view of a batched upload goes away: its uses are remembered by the slab (no CUDA call), and the last view's
// release orders the current stream after all of them and hands the storage back -- one event for the whole batch.
void release_slab_view(csgn_buf *buf) {
    csgn_slab *sl = buf->slab;
    auto note = [&](const StreamMark &m) {
        if (!m.s) return;
        for (StreamMark &u : sl->uses)
            if (u.s == m.s) {
                u.tick = std::max(u.tick, m.tick);
                return;
            }
        sl->uses.push_back(m);
    };
    note(buf->writer);
    for (const StreamMark &m : buf->readers) note(m);
    if (--sl->refs != 0) return;
    if (g.inited) {
        for (const StreamMark &m : sl->uses) wait_for_mark(g.stream, m);
        if (!give_upload_slot(sl->d, sl->cap_words)) dev_free(sl->d);
    }
    delete sl;
}
}  // namespace

int csgn_buf_free(csgn_buf *buf) {
    if (!buf) return CSGN_OK;
    if (buf->refs > 1) {            // a lazy sum still refers to it: the last reference releases the storage
        --buf->refs;
        return CSGN_OK;
    }
    if (is_rope(buf)) {
        drop_segments(buf);
        delete buf;
        return CSGN_OK;
    }
    if (buf->slab) {
        release_slab_view(buf);
        delete buf;
        return CSGN_OK;
    }
    // Pool memory whose every use that may still be in flight sits on ONE stream is freed on THAT stream: the next
    // allocation there (the same lane's next product) reuses it in stream order.  Freed on the caller's stream instead, the
    // pool could hand it out again only after the free had completed -- a loop over the lanes then keeps missing the
    // pool and goes to the driver (C++ drop-in with automatic lanes: 13 -> 27 us of host time per decrypt).
    if (g.inited && buf->owns && !buf->recycle && !buf->ready) {
        cudaStream_t one = nullptr;
        bool single = true;
        auto see = [&](const StreamMark &m) {
            if (!m.s || synced_tick(m.s) >= m.tick) return;          // nothing in flight from this use
            if (!one) one = m.s;
            else if (one != m.s) single = false;
        };
        see(buf->writer);
        for (const StreamMark &m : buf->readers) see(m);
        if (single && one && one != g.stream) {
            bool ours = one == g.own_stream || one == g.copy_stream;
            for (int i = 0; i < g.n_lanes && !ours; ++i) ours = one == g.lane[i];
            if (ours) {                                              // never enqueue on a stream the caller may have destroyed
                cudaFreeAsync(buf->d, one);
                delete buf;
                return CSGN_OK;
            }
        }
    }
    if (g.inited) {
        await_ready(buf);                      // a never-consumed upload must land before its memory is recycled
        order_after_all_uses(buf);
        if (buf->ready) g.event_pool.push_back(buf->ready);     // the current stream waits for it: safe to re-record
    }
    if (g.inited && buf->owns && !(buf->recycle && give_upload_slot(buf->d, buf->cap_words))) dev_free(buf->d);
    delete buf;
    return CSGN_OK;
}

int csgn_buf_free_batch(csgn_buf *const *bufs, uint32_t n) {
    if (!bufs) return CSGN_OK;
    for (uint32_t i = 0; i < n; ++i) csgn_buf_free(bufs[i]);
    return CSGN_OK;
}

uint64_t csgn_buf_blocks(const csgn_buf *buf) { return buf ? buf->n_blocks : 0; }
uint32_t csgn_buf_words_per_block(const csgn_buf *buf) { return buf ? buf->L : 0; }
void *csgn_buf_device_ptr(const csgn_buf *buf) {
    // Whoever uses the pointer does so on the caller's current stream, in ways the library cannot see: order that
    // stream after everything the library has in flight on the words, and treat it as their writer from now on.
    if (buf && g.inited) {
        if (need_dense(buf) != CSGN_OK) return nullptr;
        acquire_write(buf);
    }
    return buf ? buf->d : nullptr;
}

// ---------------------------------------------------------------------------
// K1 multiply
// ---------------------------------------------------------------------------
}  // extern "C"

namespace csgn {
namespace detail {

int check_mul_operands(const csgn_buf *a, const csgn_buf *b) {
    if (!a || !b) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    if (a->L != b->L) return fail(CSGN_ERR_SHAPE_MISMATCH, "words per block differ (%u vs %u)", a->L, b->L);
    if (b->n_blocks && a->n_blocks > UINT64_MAX / b->n_blocks)
        return fail(CSGN_ERR_INVALID_ARGUMENT, "product block count overflows");
    return CSGN_OK;
}

int check_mul_out(const csgn_buf *a, const csgn_buf *b, const csgn_buf *out) {
    if (out->L != a->L) return fail(CSGN_ERR_SHAPE_MISMATCH, "words per block differ (%u, %u, %u)", a->L, b->L, out->L);
    if (out->n_blocks != a->n_blocks * b->n_blocks)
        return fail(CSGN_ERR_SHAPE_MISMATCH, "output holds %llu blocks, product has %llu",
                    (unsigned long long)out->n_blocks, (unsigned long long)(a->n_blocks * b->n_blocks));
    if (out->d && (out->d == a->d || out->d == b->d)) return fail(CSGN_ERR_INVALID_ARGUMENT, "output aliases an operand");
    if (out->refs > 1) return fail(CSGN_ERR_INVALID_ARGUMENT, "output is part of a lazy sum (csgn_concat_lazy): clone it first");
    return CSGN_OK;
}

// Multiply (out != null) and/or fold the product under `key` (key != null) on the current stream.  With a key the
// count goes to device_count and/or into the peer exchange `pp`.  One launch where a fused kernel exists.
int enqueue_mul(const csgn_buf *a, const csgn_buf *b, csgn_buf *out, const csgn_key *key, uint64_t *device_count,
                const PeerPush *pp) {
    int rc0 = need_dense(b);                       // a lazy RIGHT operand interleaves with every row: one dense array
    if (rc0 == CSGN_OK && out) rc0 = need_dense(out);
    if (rc0 == CSGN_OK && (key || !out)) rc0 = need_dense(a);
    if (rc0 != CSGN_OK) return rc0;
    if (is_rope(a)) {
        // (A1 || A2 || ...) * B = (A1*B) || (A2*B) || ...  (output is i-major, src/Ciphertext.cpp:159): one launch per
        // segment of the left operand, each into its own row range of the dense product -- the sum is never copied
        acquire_read(b);
        acquire_write(out);
        uint64_t row = 0;
        for (const csgn_buf *x : a->segs) {
            acquire_read(x);
            cudaError_t e = launch_mul(x->d, x->n_blocks, b->d, b->n_blocks, a->L, out->d + row * b->n_blocks * a->L, g.stream);
            if (e != cudaSuccess) return cuda_fail(e, "multiply kernel");
            row += x->n_blocks;
        }
        return CSGN_OK;
    }
    acquire_read(a);
    acquire_read(b);
    if (out) acquire_write(out);
    if (!key) {
        cudaError_t e = launch_mul(a->d, a->n_blocks, b->d, b->n_blocks, a->L, out->d, g.stream);
        return e == cudaSuccess ? CSGN_OK : cuda_fail(e, "multiply kernel");
    }
    const uint64_t *hm = key->h_mask.empty() ? nullptr : key->h_mask.data();
    const uint64_t T = a->n_blocks * b->n_blocks;
    if (T == 0 || !mul_fold_supported(a->L)) {
        // no fused kernel for this shape (blocks of more than 512 units): multiply, then fold -- two launches;
        // a count-only request multiplies into a temporary
        csgn_buf *tmp = nullptr;
        if (!out && T) {
            int rc = new_buf(T, a->L, 0, &tmp);
            if (rc != CSGN_OK) return rc;
        }
        csgn_buf *dst = out ? out : tmp;
        cudaError_t e = T ? launch_mul(a->d, a->n_blocks, b->d, b->n_blocks, a->L, dst->d, g.stream) : cudaSuccess;
        if (e == cudaSuccess)
            e = launch_decrypt_count(dst ? dst->d : nullptr, T, a->L, key->d_mask, hm, fold_scratch(), device_count, g.stream,
                                     pp, folds_overlap());
        if (tmp) csgn_buf_free(tmp);
        return e == cudaSuccess ? CSGN_OK : cuda_fail(e, "multiply + decrypt kernels");
    }
    MulFold mf;
    mf.mask = key->d_mask;
    mf.host_mask = hm;
    mf.scratch = fold_scratch();
    mf.count_out = device_count;
    mf.overlapped = folds_overlap();
    mf.peer = pp;
    cudaError_t e = launch_mul(a->d, a->n_blocks, b->d, b->n_blocks, a->L, out ? out->d : nullptr, g.stream, &mf);
    return e == cudaSuccess ? CSGN_OK : cuda_fail(e, "fused multiply-decrypt kernel");
}

// Resolve the `out` convention of the fused entry points: null = count only; *out null = allocate; else write into.
int fused_out(const csgn_buf *a, const csgn_buf *b, csgn_buf **out, csgn_buf **dst, bool *allocated) {
    *dst = nullptr;
    *allocated = false;
    if (!out) return CSGN_OK;
    if (*out) {
        *dst = *out;
        return check_mul_out(a, b, *out);
    }
    int rc = new_buf(a->n_blocks * b->n_blocks, a->L, 0, dst);
    if (rc == CSGN_OK) *allocated = true;
    return rc;
}

int check_key(const csgn_buf *a, const csgn_key *key) {
    if (!key) return fail(CSGN_ERR_INVALID_ARGUMENT, "null key");
    if (a->L != key->L)
        return fail(CSGN_ERR_SHAPE_MISMATCH, "ciphertext has %u words per block, key expects %u", a->L, key->L);
    return CSGN_OK;
}

}  // namespace detail
}  // namespace csgn

extern "C" {

int csgn_mul_into(const csgn_buf *a, const csgn_buf *b, csgn_buf *out) {
    NEED_INIT();
    int rc = check_mul_operands(a, b);
    if (rc != CSGN_OK) return rc;
    if (!out) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    rc = check_mul_out(a, b, out);
    if (rc != CSGN_OK) return rc;
    AutoLane lane(out->owns ? a : nullptr, out->owns ? b : nullptr);     // a view's consumer is on the caller's stream
    return enqueue_mul(a, b, out, nullptr, nullptr, nullptr);
}

int csgn_mul(const csgn_buf *a, const csgn_buf *b, csgn_buf **out) {
    NEED_INIT();
    int rc = check_mul_operands(a, b);
    if (rc != CSGN_OK) return rc;
    if (!out) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    AutoLane lane(a, b);
    csgn_buf *c = nullptr;
    rc = new_buf(a->n_blocks * b->n_blocks, a->L, 0, &c);
    if (rc != CSGN_OK) return rc;
    rc = enqueue_mul(a, b, c, nullptr, nullptr, nullptr);
    if (rc != CSGN_OK) {
        csgn_buf_free(c);
        return rc;
    }
    *out = c;
    return CSGN_OK;
}

// ---------------------------------------------------------------------------
// fused multiply -> decrypt
// ---------------------------------------------------------------------------
int csgn_mul_count_async(const csgn_buf *a, const csgn_buf *b, const csgn_key *key, csgn_buf **out, uint64_t *device_count) {
    NEED_INIT();
    int rc = check_mul_operands(a, b);
    if (rc == CSGN_OK) rc = check_key(a, key);
    if (rc != CSGN_OK) return rc;
    if (!device_count) return fail(CSGN_ERR_INVALID_ARGUMENT, "null count destination");
    csgn_buf *dst = nullptr;
    bool allocated = false;
    rc = fused_out(a, b, out, &dst, &allocated);
    if (rc != CSGN_OK) return rc;
    rc = enqueue_mul(a, b, dst, key, device_count, nullptr);
    if (rc != CSGN_OK) {
        if (allocated) csgn_buf_free(dst);
        return rc;
    }
    if (allocated) *out = dst;
    return CSGN_OK;
}

int csgn_mul_decrypt(const csgn_buf *a, const csgn_buf *b, const csgn_key *key, csgn_buf **out, uint8_t *bit,
                     uint64_t *count) {
    NEED_INIT();
    if (!bit && !count) return fail(CSGN_ERR_INVALID_ARGUMENT, "no output");
    int rc = csgn_mul_count_async(a, b, key, out, g.d_scratch + 2);
    if (rc != CSGN_OK) return rc;
    CU(cudaMemcpyAsync(g.h_result, g.d_scratch + 2, sizeof(uint64_t), cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    note_synced(g.stream);
    if (bit) *bit = (uint8_t)(g.h_result[0] & 1u);
    if (count) *count = g.h_result[0];
    return CSGN_OK;
}

int csgn_mul_count_batch_async(const csgn_buf *const *a, const csgn_buf *const *b, uint32_t n, const csgn_key *key,
                               csgn_buf **out, uint64_t *device_counts) {
    NEED_INIT();
    if (n && (!a || !b || !device_counts)) return fail(CSGN_ERR_INVALID_ARGUMENT, "null argument");
    std::vector<bool> ours(n, false);
    if (out)
        for (uint32_t i = 0; i < n; ++i) ours[i] = out[i] == nullptr;
    LaneScope lanes(n);
    for (uint32_t i = 0; i < n; ++i) {
        lanes.enter(i);
        int rc = csgn_mul_count_async(a[i], b[i], key, out ? &out[i] : nullptr, device_counts + i);
        if (rc != CSGN_OK) {
            lanes.join();
            for (uint32_t k = 0; k < i; ++k)
                if (ours[k]) {
                    csgn_buf_free(out[k]);
                    out[k] = nullptr;
                }
            return rc;
        }
    }
    return CSGN_OK;
}

// ---------------------------------------------------------------------------
// K2 add
// ---------------------------------------------------------------------------
int csgn_concat(const csgn_buf *a, const csgn_buf *b, csgn_buf **out) {
    NEED_INIT();
    if (!a || !b || !out) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    if (a->L != b->L) return fail(CSGN_ERR_SHAPE_MISMATCH, "words per block differ (%u vs %u)", a->L, b->L);
    AutoLane lane(a, b);
    csgn_buf *c = nullptr;
    int rc = new_buf(a->n_blocks + b->n_blocks, a->L, 0, &c);
    if (rc != CSGN_OK) return rc;
    if (is_rope(a) || is_rope(b)) {
        rc = copy_words_into(a, c->d);
        if (rc == CSGN_OK) rc = copy_words_into(b, c->d + a->n_blocks * a->L);
        if (rc != CSGN_OK) {
            csgn_buf_free(c);
            return rc;
        }
        *out = c;
        return CSGN_OK;
    }
    acquire_read(a);
    acquire_read(b);
    cudaError_t e = launch_concat(a->d, a->n_blocks * a->L, b->d, b->n_blocks * b->L, c->d, g.stream);
    if (e != cudaSuccess) {
        csgn_buf_free(c);
        return cuda_fail(e, "concat kernel");
    }
    *out = c;
    return CSGN_OK;
}

// a || b without moving a word: the result refers to the operands' storage.
namespace {
constexpr size_t kRopeMaxSegments = 32;
constexpr uint64_t kRopeMinWords = (1ull << 20) / 8;      // below 1 MiB a copy is cheaper than one more segment to walk
void add_segments(csgn_buf *r, const csgn_buf *x) {
    if (is_rope(x)) {
        for (csgn_buf *sgm : x->segs) {
            ++sgm->refs;
            r->segs.push_back(sgm);
        }
    } else if (x->n_blocks) {
        csgn_buf *m = const_cast<csgn_buf *>(x);
        ++m->refs;
        r->segs.push_back(m);
    }
}
}  // namespace

int csgn_concat_lazy(const csgn_buf *a, const csgn_buf *b, csgn_buf **out) {
    NEED_INIT();
    if (!a || !b || !out) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    if (a->L != b->L) return fail(CSGN_ERR_SHAPE_MISMATCH, "words per block differ (%u vs %u)", a->L, b->L);
    const size_t na = is_rope(a) ? a->segs.size() : 1, nb = is_rope(b) ? b->segs.size() : 1;
    const uint64_t wa = a->n_blocks * a->L, wb = b->n_blocks * b->L;
    // small operands, and sums that would grow a long tail of segments, are copied (csgn_concat)
    if (wa < kRopeMinWords || wb < kRopeMinWords || na + nb > kRopeMaxSegments) return csgn_concat(a, b, out);
    csgn_buf *r = new csgn_buf;
    r->L = a->L;
    r->n_blocks = a->n_blocks + b->n_blocks;
    r->cap_words = 0;
    add_segments(r, a);
    add_segments(r, b);
    *out = r;
    return CSGN_OK;
}

int csgn_buf_segments(const csgn_buf *buf) { return !buf ? 0 : is_rope(buf) ? (int)buf->segs.size() : 1; }
int csgn_buf_retained(const csgn_buf *buf) { return buf && buf->refs > 1 ? 1 : 0; }

int csgn_buf_flatten(csgn_buf *buf) {
    NEED_INIT();
    if (!buf) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    AutoLane lane(buf);
    return need_dense(buf);
}

int csgn_append(csgn_buf *a, const csgn_buf *b) {
    NEED_INIT();
    if (!a || !b) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    if (!a->owns) return fail(CSGN_ERR_INVALID_ARGUMENT, "cannot grow a non-owning view");
    if (a->refs > 1) return fail(CSGN_ERR_INVALID_ARGUMENT, "cannot grow a buffer that is part of a lazy sum: clone it first");
    if (a->L != b->L) return fail(CSGN_ERR_SHAPE_MISMATCH, "words per block differ (%u vs %u)", a->L, b->L);
    const uint64_t na = a->n_blocks * a->L, nb = b->n_blocks * b->L;
    if (nb == 0) return CSGN_OK;
    AutoLane lane(a, nullptr);           // the grown ciphertext stays on the stream that built it
    {
        int rc = need_dense(a);
        if (rc == CSGN_OK) rc = need_dense(b);
        if (rc != CSGN_OK) return rc;
    }
    acquire_write(a);
    if (b != a) acquire_read(b);
    if (na + nb <= a->cap_words) {
        // b == a is fine: source [0,na) and destination [na,2na) do not overlap
        cudaError_t e = launch_concat(a->d, na, b->d, nb, a->d, g.stream);
        if (e != cudaSuccess) return cuda_fail(e, "append kernel");
    } else {
        const uint64_t cap = std::max<uint64_t>(na + nb, 2 * a->cap_words);
        uint64_t *nd = nullptr;
        int rc = dev_alloc(cap, &nd);
        if (rc != CSGN_OK && cap > na + nb) rc = dev_alloc(na + nb, &nd);  // no room to double
        if (rc != CSGN_OK) return rc;
        cudaError_t e = launch_concat(a->d, na, b->d, nb, nd, g.stream);
        if (e != cudaSuccess) {
            dev_free(nd);
            return cuda_fail(e, "append kernel");
        }
        dev_free(a->d);  // stream-ordered: the copy above still reads it safely
        a->d = nd;
        a->cap_words = cap;
        a->recycle = false;
    }
    a->n_blocks += b->n_blocks;
    return CSGN_OK;
}

// ---------------------------------------------------------------------------
// K3 decrypt
// ---------------------------------------------------------------------------
int csgn_key_create(uint64_t N, const uint64_t *positions, uint32_t D, csgn_key **out) {
    NEED_INIT();
    if (!out || N == 0) return fail(CSGN_ERR_INVALID_ARGUMENT, "bad key arguments");
    if (D && !positions) return fail(CSGN_ERR_INVALID_ARGUMENT, "null positions");
    const uint32_t L = csgn_words_per_block(N);
    std::vector<uint64_t> mask(L, 0);
    for (uint32_t i = 0; i < D; ++i) {
        if (positions[i] >= N)
            return fail(CSGN_ERR_INVALID_ARGUMENT, "secret position %llu outside [0,%llu)",
                        (unsigned long long)positions[i], (unsigned long long)N);
        mask[positions[i] >> 6] |= 1ull << (63u - (positions[i] & 63u));
    }
    csgn_key *k = new csgn_key;
    k->N = N;
    k->L = L;
    k->D = D;
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&k->d_mask), (size_t)L * sizeof(uint64_t));
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(k->d_mask, mask.data(), (size_t)L * sizeof(uint64_t), cudaMemcpyHostToDevice, g.stream);
    if (e == cudaSuccess && D) e = cudaMalloc(reinterpret_cast<void **>(&k->d_positions), (size_t)D * sizeof(uint64_t));
    if (e == cudaSuccess && D)
        e = cudaMemcpyAsync(k->d_positions, positions, (size_t)D * sizeof(uint64_t), cudaMemcpyHostToDevice, g.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g.stream);  // `mask` dies with this frame
    if (e == cudaSuccess) k->h_mask = mask;
    std::fill(mask.begin(), mask.end(), 0);
    if (e != cudaSuccess) {
        if (k->d_mask) cudaFree(k->d_mask);
        if (k->d_positions) cudaFree(k->d_positions);
        delete k;
        return cuda_fail(e, "key upload");
    }
    *out = k;
    return CSGN_OK;
}

int csgn_key_free(csgn_key *key) {
    if (!key) return CSGN_OK;
    if (g.inited && key->d_mask) {
        cudaMemsetAsync(key->d_mask, 0, (size_t)key->L * sizeof(uint64_t), g.stream);  // zeroise, as the reference's dtor does
        if (key->d_positions) cudaMemsetAsync(key->d_positions, 0, (size_t)key->D * sizeof(uint64_t), g.stream);
        cudaStreamSynchronize(g.stream);
        cudaFree(key->d_mask);
        if (key->d_positions) cudaFree(key->d_positions);
    }
    std::fill(key->h_mask.begin(), key->h_mask.end(), 0);
    delete key;
    return CSGN_OK;
}

int csgn_decrypt_count_async(const csgn_buf *c, const csgn_key *key, uint64_t *device_count) {
    NEED_INIT();
    if (!c || !key || !device_count) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    if (c->L != key->L)
        return fail(CSGN_ERR_SHAPE_MISMATCH, "ciphertext has %u words per block, key expects %u", c->L, key->L);
    const uint64_t *hm = key->h_mask.empty() ? nullptr : key->h_mask.data();
    if (is_rope(c)) {
        // the count of a concatenation is the sum of its parts' counts (src/SecretKey.cpp:139 XORs block by block):
        // one fold per segment into a scratch word each, then a one-warp sum -- the sum is never copied together
        const uint32_t n = (uint32_t)c->segs.size();
        uint64_t *part = nullptr;
        int rc = dev_alloc(n, &part);
        if (rc != CSGN_OK) return rc;
        cudaError_t e = cudaSuccess;
        for (uint32_t i = 0; i < n && e == cudaSuccess; ++i) {
            const csgn_buf *x = c->segs[i];
            acquire_read(x);
            e = launch_decrypt_count(x->d, x->n_blocks, x->L, key->d_mask, hm, fold_scratch(), part + i, g.stream, nullptr,
                                     folds_overlap());
        }
        if (e == cudaSuccess) e = launch_sum_words(part, n, device_count, g.stream);
        dev_free(part);
        return e == cudaSuccess ? CSGN_OK : cuda_fail(e, "decrypt kernel");
    }
    acquire_read(c);
    cudaError_t e = launch_decrypt_count(c->d, c->n_blocks, c->L, key->d_mask, hm, fold_scratch(), device_count,
                                         g.stream, nullptr, folds_overlap());
    if (e != cudaSuccess) return cuda_fail(e, "decrypt kernel");
    return CSGN_OK;
}

int csgn_decrypt_count(const csgn_buf *c, const csgn_key *key, uint64_t *count) {
    NEED_INIT();
    if (!count) return fail(CSGN_ERR_INVALID_ARGUMENT, "null output");
    int rc = csgn_decrypt_count_async(c, key, g.d_scratch + 2);
    if (rc != CSGN_OK) return rc;
    CU(cudaMemcpyAsync(g.h_result, g.d_scratch + 2, sizeof(uint64_t), cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    note_synced(g.stream);
    *count = g.h_result[0];
    return CSGN_OK;
}

int csgn_decrypt(const csgn_buf *c, const csgn_key *key, uint8_t *bit) {
    if (!bit) return fail(CSGN_ERR_INVALID_ARGUMENT, "null output");
    uint64_t count = 0;
    int rc = csgn_decrypt_count(c, key, &count);
    if (rc != CSGN_OK) return rc;
    *bit = (uint8_t)(count & 1u);
    return CSGN_OK;
}

// ---- deferred results: the fold and the copy of its count are enqueued, the host reads later -------------
namespace {

int take_result(csgn_result **out) {
    if (g.free_results.empty()) return fail(CSGN_ERR_OUT_OF_MEMORY, "more than %u decrypt results pending", kResultSlots);
    csgn_result *r = new csgn_result;
    r->slot = g.free_results.back();
    g.free_results.pop_back();
    r->h = g.h_results + r->slot;
    r->d = g.d_results + r->slot;
    r->done = take_event();
    if (!r->done) {
        g.free_results.push_back(r->slot);
        delete r;
        return fail(CSGN_ERR_CUDA, "cannot create an event");
    }
    *out = r;
    return CSGN_OK;
}

int finish_result(csgn_result *r, int rc) {
    cudaError_t e = cudaSuccess;
    if (rc == CSGN_OK) {
        e = cudaMemcpyAsync(r->h, r->d, sizeof(uint64_t), cudaMemcpyDeviceToHost, g.stream);
        if (e == cudaSuccess) e = cudaEventRecord(r->done, g.stream);
    }
    if (rc != CSGN_OK || e != cudaSuccess) {
        r->waited = true;
        csgn_result_free(r);
        return rc != CSGN_OK ? rc : cuda_fail(e, "result copy");
    }
    return CSGN_OK;
}

}  // namespace

int csgn_decrypt_deferred(const csgn_buf *c, const csgn_key *key, csgn_result **out) {
    NEED_INIT();
    if (!c || !key || !out) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    csgn_result *r = nullptr;
    int rc = take_result(&r);
    if (rc != CSGN_OK) return rc;
    AutoLane lane(c);
    rc = finish_result(r, csgn_decrypt_count_async(c, key, r->d));
    if (rc == CSGN_OK) *out = r;
    return rc;
}

int csgn_mul_decrypt_deferred(const csgn_buf *a, const csgn_buf *b, const csgn_key *key, csgn_buf **prod,
                              csgn_result **out) {
    NEED_INIT();
    if (!out) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    int rc = check_mul_operands(a, b);
    if (rc != CSGN_OK) return rc;
    csgn_result *r = nullptr;
    rc = take_result(&r);
    if (rc != CSGN_OK) return rc;
    AutoLane lane((!prod || !*prod || (*prod)->owns) ? a : nullptr, (!prod || !*prod || (*prod)->owns) ? b : nullptr);
    rc = finish_result(r, csgn_mul_count_async(a, b, key, prod, r->d));
    if (rc == CSGN_OK) *out = r;
    return rc;
}

int csgn_result_ready(const csgn_result *r) {
    if (!r) return 0;
    if (r->waited) return 1;
    const cudaError_t e = cudaEventQuery(r->done);
    if (e != cudaSuccess) cudaGetLastError();
    return e == cudaSuccess ? 1 : 0;
}

int csgn_result_wait(csgn_result *r, uint64_t *count) {
    NEED_INIT();
    if (!r) return fail(CSGN_ERR_INVALID_ARGUMENT, "null result");
    if (!r->waited) {
        CU(cudaEventSynchronize(r->done));
        r->waited = true;
    }
    if (count) *count = *r->h;
    return CSGN_OK;
}

int csgn_result_free(csgn_result *r) {
    if (!r) return CSGN_OK;
    if (g.inited) {
        if (!r->waited && r->done) cudaEventSynchronize(r->done);   // the slot is reused: its copy must have landed
        if (r->done) g.event_pool.push_back(r->done);
        g.free_results.push_back(r->slot);
    }
    delete r;
    return CSGN_OK;
}

int csgn_decrypt_product(const csgn_buf *const *factors, uint32_t n_factors, const csgn_key *key, uint8_t *bit,
                         uint64_t *count) {
    NEED_INIT();
    if (!factors || !key || !bit || n_factors == 0) return fail(CSGN_ERR_INVALID_ARGUMENT, "bad product arguments");
    for (uint32_t i = 0; i < n_factors; ++i) {
        if (!factors[i]) return fail(CSGN_ERR_INVALID_ARGUMENT, "null factor %u", i);
        if (factors[i]->L != key->L)
            return fail(CSGN_ERR_SHAPE_MISMATCH, "factor %u has %u words per block, key expects %u", i, factors[i]->L,
                        key->L);
    }
    uint64_t *d_counts = nullptr;
    int rc = dev_alloc(n_factors, &d_counts);
    if (rc != CSGN_OK) return rc;
    for (uint32_t i = 0; i < n_factors; ++i) {
        rc = csgn_decrypt_count_async(factors[i], key, d_counts + i);
        if (rc != CSGN_OK) {
            dev_free(d_counts);
            return rc;
        }
    }
    std::vector<uint64_t> h(n_factors);
    cudaError_t e = cudaMemcpyAsync(h.data(), d_counts, n_factors * sizeof(uint64_t), cudaMemcpyDeviceToHost, g.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(g.stream);
    if (e == cudaSuccess) note_synced(g.stream);
    dev_free(d_counts);
    if (e != cudaSuccess) return cuda_fail(e, "product decrypt readback");
    uint64_t prod = 1;
    uint8_t parity = 1;
    for (uint32_t i = 0; i < n_factors; ++i) {
        parity &= (uint8_t)(h[i] & 1u);
        prod = (h[i] != 0 && prod > UINT64_MAX / h[i]) ? UINT64_MAX : prod * h[i];
    }
    *bit = parity;
    if (count) *count = prod;
    return CSGN_OK;
}

int csgn_decrypt_positions(const csgn_buf *c, uint64_t N, const uint64_t *positions, uint32_t D, uint8_t *bit) {
    csgn_key *k = nullptr;
    int rc = csgn_key_create(N, positions, D, &k);
    if (rc != CSGN_OK) return rc;
    rc = csgn_decrypt(c, k, bit);
    csgn_key_free(k);
    return rc;
}


// ---------------------------------------------------------------------------
// batches of independent items
// ---------------------------------------------------------------------------
int csgn_mul_into_batch(const csgn_buf *const *a, const csgn_buf *const *b, uint32_t n, csgn_buf *const *out) {
    NEED_INIT();
    if (n && (!a || !b || !out)) return fail(CSGN_ERR_INVALID_ARGUMENT, "null argument");
    LaneScope lanes(n);
    for (uint32_t i = 0; i < n; ++i) {
        lanes.enter(i);
        int rc = csgn_mul_into(a[i], b[i], out[i]);
        if (rc != CSGN_OK) return rc;        // ~LaneScope joins what was enqueued
    }
    return CSGN_OK;
}

int csgn_mul_batch(const csgn_buf *const *a, const csgn_buf *const *b, uint32_t n, csgn_buf **out) {
    NEED_INIT();
    if (n && (!a || !b || !out)) return fail(CSGN_ERR_INVALID_ARGUMENT, "null argument");
    for (uint32_t i = 0; i < n; ++i) out[i] = nullptr;
    LaneScope lanes(n);
    for (uint32_t i = 0; i < n; ++i) {
        lanes.enter(i);
        int rc = csgn_mul(a[i], b[i], &out[i]);
        if (rc != CSGN_OK) {
            lanes.join();
            for (uint32_t k = 0; k < i; ++k) {
                csgn_buf_free(out[k]);
                out[k] = nullptr;
            }
            return rc;
        }
    }
    return CSGN_OK;
}

int csgn_decrypt_count_batch_async(const csgn_buf *const *c, uint32_t n, const csgn_key *key, uint64_t *device_counts) {
    NEED_INIT();
    if (n && (!c || !device_counts)) return fail(CSGN_ERR_INVALID_ARGUMENT, "null argument");
    LaneScope lanes(n);
    for (uint32_t i = 0; i < n; ++i) {
        lanes.enter(i);
        int rc = csgn_decrypt_count_async(c[i], key, device_counts + i);
        if (rc != CSGN_OK) return rc;
    }
    return CSGN_OK;
}

int csgn_decrypt_batch(const csgn_buf *const *c, uint32_t n, const csgn_key *key, uint8_t *bits, uint64_t *counts) {
    NEED_INIT();
    if (n == 0) return CSGN_OK;
    if (!bits && !counts) return fail(CSGN_ERR_INVALID_ARGUMENT, "no output");
    uint64_t *d = nullptr;
    int rc = dev_alloc(n, &d);
    if (rc != CSGN_OK) return rc;
    rc = csgn_decrypt_count_batch_async(c, n, key, d);
    std::vector<uint64_t> h(n);
    cudaError_t e = cudaSuccess;
    if (rc == CSGN_OK) {
        e = cudaMemcpyAsync(h.data(), d, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, g.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g.stream);
        if (e == cudaSuccess) note_synced(g.stream);
    }
    dev_free(d);
    if (rc != CSGN_OK) return rc;
    if (e != cudaSuccess) return cuda_fail(e, "batch decrypt readback");
    for (uint32_t i = 0; i < n; ++i) {
        if (bits) bits[i] = (uint8_t)(h[i] & 1u);
        if (counts) counts[i] = h[i];
    }
    return CSGN_OK;
}


// ---------------------------------------------------------------------------
// batched encryption
// ---------------------------------------------------------------------------
int csgn_encrypt_batch(const csgn_key *key, const uint8_t *bits, uint64_t n, uint64_t first_block, uint64_t seed,
                       csgn_buf **out) {
    NEED_INIT();
    if (!key || !out || (n && !bits)) return fail(CSGN_ERR_INVALID_ARGUMENT, "null argument");
    if (key->D == 0) return fail(CSGN_ERR_INVALID_ARGUMENT, "the key has no secret positions");
    csgn_buf *b = nullptr;
    int rc = new_buf(n, key->L, 0, &b);
    if (rc != CSGN_OK) return rc;
    if (n) {
        uint8_t *d_bits = nullptr;
        cudaError_t e = cudaMallocAsync(reinterpret_cast<void **>(&d_bits), n, g.stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_bits, bits, n, cudaMemcpyHostToDevice, g.stream);
        const uint64_t rem = key->N % 64;
        const uint64_t pad = rem ? ~0ull << (64 - rem) : ~0ull;
        if (e == cudaSuccess)
            e = launch_encrypt_batch(d_bits, n, first_block, key->L, pad, key->d_mask, key->d_positions, key->D, seed,
                                     b->d, g.stream);
        if (d_bits) cudaFreeAsync(d_bits, g.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g.stream);   // `bits` may be a temporary of the caller
        if (e != cudaSuccess) {
            csgn_buf_free(b);
            return cuda_fail(e, "batched encryption");
        }
    }
    *out = b;
    return CSGN_OK;
}

int csgn_encrypt_uint(const csgn_key *key, const uint64_t *values, uint64_t n, uint32_t width, uint64_t first_block,
                      uint64_t seed, csgn_buf **out) {
    NEED_INIT();
    if (!key || !out || (n && !values)) return fail(CSGN_ERR_INVALID_ARGUMENT, "null argument");
    if (width < 1 || width > 64) return fail(CSGN_ERR_INVALID_ARGUMENT, "width %u outside 1..64", width);
    if (key->D == 0) return fail(CSGN_ERR_INVALID_ARGUMENT, "the key has no secret positions");
    if (width < 64)
        for (uint64_t k = 0; k < n; ++k)
            if (values[k] >> width)
                return fail(CSGN_ERR_INVALID_ARGUMENT, "values[%llu] = %llu does not fit in %u bits",
                            (unsigned long long)k, (unsigned long long)values[k], width);
    const uint32_t L = key->L;
    if (n > UINT64_MAX / 64) return fail(CSGN_ERR_INVALID_ARGUMENT, "block count overflows");
    int rc = check_blocks(width * n, L);
    if (rc != CSGN_OK) return rc;
    // one allocation for the width planes, laid one after another as the kernel writes them
    csgn_slab *sl = new csgn_slab;
    sl->cap_words = std::max<uint64_t>(1, width * n * L);
    rc = dev_alloc(sl->cap_words, &sl->d);
    if (rc != CSGN_OK) {
        delete sl;
        return rc;
    }
    if (n) {
        DevTable v;
        rc = stage_to_device(values, n * sizeof(uint64_t), &v.d);
        const uint64_t rem = key->N % 64;
        const uint64_t pad = rem ? ~0ull << (64 - rem) : ~0ull;
        cudaError_t e = cudaSuccess;
        if (rc == CSGN_OK)
            e = launch_encrypt_uint(static_cast<const uint64_t *>(v.d), n, width, first_block, L, pad, key->d_mask,
                                    key->d_positions, key->D, seed, sl->d, g.stream);
        if (rc == CSGN_OK && e != cudaSuccess) rc = cuda_fail(e, "integer encryption");
        if (rc != CSGN_OK) {
            dev_free(sl->d);
            delete sl;
            return rc;
        }
    }
    const uint64_t tick = g.tick++;
    for (uint32_t j = 0; j < width; ++j) {
        csgn_buf *b = new csgn_buf;
        b->d = sl->d + j * n * L;
        b->n_blocks = n;
        b->L = L;
        b->cap_words = 0;
        b->owns = false;
        b->slab = sl;
        b->writer = {g.stream, tick};
        out[j] = b;
    }
    sl->refs = width;
    return CSGN_OK;
}

// ---------------------------------------------------------------------------
// K4 permute
// ---------------------------------------------------------------------------
int csgn_perm_create(uint64_t N, const uint64_t *perm, csgn_perm **out) {
    NEED_INIT();
    if (!out || !perm || N == 0) return fail(CSGN_ERR_INVALID_ARGUMENT, "bad permutation arguments");
    if (N >= (1ull << 32)) return fail(CSGN_ERR_INVALID_ARGUMENT, "N too large for the source map");
    std::vector<uint32_t> map(N);
    std::vector<uint8_t> seen(N, 0);
    for (uint64_t i = 0; i < N; ++i) {
        const uint64_t p = perm[i];
        if (p >= N || seen[p])
            return fail(CSGN_ERR_INVALID_ARGUMENT, "not a permutation of [0,%llu): entry %llu = %llu",
                        (unsigned long long)N, (unsigned long long)i, (unsigned long long)p);
        seen[p] = 1;
        map[i] = (uint32_t)(((p >> 6) << 6) | (63u - (p & 63u)));
    }
    csgn_perm *h = new csgn_perm;
    h->N = N;
    h->L = csgn_words_per_block(N);
    // Bit-sliced form: a block is W = 2L 32-bit words; bit j of word c holds position
    // 64*(c>>1) + (c odd ? 31-j : 63-j).  Entry j*W + c' names the source slice of output
    // (c', j) as a shared-memory BYTE offset 4*(stride*c + j_src), or the zero slot 4*stride*W for pad bits.
    std::vector<uint32_t> slices;
    if (permute_sliced_supported(h->L)) {
        const uint32_t W = 2 * h->L, stride = kPermSliceStride;
        slices.assign((size_t)32 * W, 4u * stride * W);   // byte offsets; default = the zero slot
        for (uint32_t c = 0; c < W; ++c)
            for (uint32_t j = 0; j < 32; ++j) {
                const uint64_t i = 64ull * (c >> 1) + ((c & 1u) ? 31u - j : 63u - j);
                if (i >= N) continue;
                const uint64_t p = perm[i];
                const uint32_t sc = 2u * (uint32_t)(p >> 6) + (((p & 63u) < 32u) ? 1u : 0u);
                slices[(size_t)j * W + c] = 4u * (stride * sc + (31u - (uint32_t)(p & 31u)));
            }
    }
    // The plane kernel keeps slice (c, j) at word j*W + c of the tile itself: the same gather, other offsets.
    std::vector<uint32_t> planes;
    if (permute_plane_supported(h->L)) {
        const uint32_t W = 2 * h->L;
        planes.assign((size_t)32 * W, 4u * 32u * W);      // default = the zero words behind the tile
        for (uint32_t c = 0; c < W; ++c)
            for (uint32_t j = 0; j < 32; ++j) {
                const uint64_t i = 64ull * (c >> 1) + ((c & 1u) ? 31u - j : 63u - j);
                if (i >= N) continue;
                const uint64_t p = perm[i];
                const uint32_t sc = 2u * (uint32_t)(p >> 6) + (((p & 63u) < 32u) ? 1u : 0u);
                planes[(size_t)j * W + c] = 4u * ((31u - (uint32_t)(p & 31u)) * W + sc);
            }
    }
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&h->d_map), (size_t)N * sizeof(uint32_t));
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(h->d_map, map.data(), (size_t)N * sizeof(uint32_t), cudaMemcpyHostToDevice, g.stream);
    if (e == cudaSuccess && !slices.empty()) {
        e = cudaMalloc(reinterpret_cast<void **>(&h->d_slice_map), slices.size() * sizeof(uint32_t));
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(h->d_slice_map, slices.data(), slices.size() * sizeof(uint32_t), cudaMemcpyHostToDevice,
                                g.stream);
    }
    if (e == cudaSuccess && !planes.empty()) {
        e = cudaMalloc(reinterpret_cast<void **>(&h->d_plane_map), planes.size() * sizeof(uint32_t));
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(h->d_plane_map, planes.data(), planes.size() * sizeof(uint32_t), cudaMemcpyHostToDevice,
                                g.stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(g.stream);
    if (e != cudaSuccess) {
        if (h->d_map) cudaFree(h->d_map);
        if (h->d_slice_map) cudaFree(h->d_slice_map);
        if (h->d_plane_map) cudaFree(h->d_plane_map);
        delete h;
        return cuda_fail(e, "permutation upload");
    }
    *out = h;
    return CSGN_OK;
}

int csgn_perm_free(csgn_perm *perm) {
    if (!perm) return CSGN_OK;
    if (g.inited && perm->d_map) {
        cudaStreamSynchronize(g.stream);
        cudaFree(perm->d_map);
        if (perm->d_slice_map) cudaFree(perm->d_slice_map);
        if (perm->d_plane_map) cudaFree(perm->d_plane_map);
    }
    delete perm;
    return CSGN_OK;
}

int csgn_permute_into(const csgn_buf *c, const csgn_perm *perm, csgn_buf *out) {
    NEED_INIT();
    if (!c || !perm || !out) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    if (c->L != perm->L || out->L != perm->L)
        return fail(CSGN_ERR_SHAPE_MISMATCH, "words per block: ciphertext %u, output %u, permutation %u", c->L,
                    out->L, perm->L);
    if (out->n_blocks > c->n_blocks)
        return fail(CSGN_ERR_SHAPE_MISMATCH, "output holds more blocks than the input");
    if (out->d && out->d == c->d) return fail(CSGN_ERR_INVALID_ARGUMENT, "permute cannot run in place");
    if (out->refs > 1) return fail(CSGN_ERR_INVALID_ARGUMENT, "output is part of a lazy sum (csgn_concat_lazy): clone it first");
    AutoLane lane(out->owns ? c : nullptr);
    {
        int rc = need_dense(out);
        if (rc != CSGN_OK) return rc;
    }
    if (is_rope(c)) {
        // a permutation acts on every block by itself: each segment goes straight to its place in the dense result
        acquire_write(out);
        uint64_t done = 0;
        for (const csgn_buf *x : c->segs) {
            if (done >= out->n_blocks) break;
            const uint64_t n = std::min<uint64_t>(x->n_blocks, out->n_blocks - done);
            acquire_read(x);
            cudaError_t e = launch_permute(x->d, n, c->L, (uint32_t)perm->N, perm->d_map, perm->d_slice_map, perm->d_plane_map,
                                           out->d + done * c->L, g.stream);
            if (e != cudaSuccess) return cuda_fail(e, "permute kernel");
            done += n;
        }
        return CSGN_OK;
    }
    acquire_read(c);
    acquire_write(out);
    cudaError_t e = launch_permute(c->d, out->n_blocks, c->L, (uint32_t)perm->N, perm->d_map, perm->d_slice_map,
                                   perm->d_plane_map, out->d, g.stream);
    if (e != cudaSuccess) return cuda_fail(e, "permute kernel");
    return CSGN_OK;
}

int csgn_permute(const csgn_buf *c, const csgn_perm *perm, int strict_ref_truncate, csgn_buf **out) {
    NEED_INIT();
    if (!c || !perm || !out) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    if (c->n_blocks == 0) return fail(CSGN_ERR_INVALID_ARGUMENT, "cannot permute an empty ciphertext");
    AutoLane lane(c);
    csgn_buf *r = nullptr;
    int rc = new_buf(strict_ref_truncate ? 1 : c->n_blocks, c->L, 0, &r);
    if (rc != CSGN_OK) return rc;
    rc = csgn_permute_into(c, perm, r);
    if (rc != CSGN_OK) {
        csgn_buf_free(r);
        return rc;
    }
    *out = r;
    return CSGN_OK;
}

// ---------------------------------------------------------------------------
// checksum, sharding
// ---------------------------------------------------------------------------
int csgn_buf_checksum(const csgn_buf *buf, uint64_t *xor_out, uint64_t *sum_out, uint64_t *wsum_out) {
    NEED_INIT();
    if (!buf) return fail(CSGN_ERR_INVALID_ARGUMENT, "null handle");
    uint64_t *acc = g.d_scratch + 4;
    {
        int rc = need_dense(buf);
        if (rc != CSGN_OK) return rc;
    }
    acquire_read(buf);
    CU(cudaMemsetAsync(acc, 0, 3 * sizeof(uint64_t), g.stream));
    cudaError_t e = launch_checksum(buf->d, buf->n_blocks * buf->L, acc, g.stream);
    if (e != cudaSuccess) return cuda_fail(e, "checksum kernel");
    CU(cudaMemcpyAsync(g.h_result + 4, acc, 3 * sizeof(uint64_t), cudaMemcpyDeviceToHost, g.stream));
    CU(cudaStreamSynchronize(g.stream));
    note_synced(g.stream);
    if (xor_out) *xor_out = g.h_result[4];
    if (sum_out) *sum_out = g.h_result[5];
    if (wsum_out) *wsum_out = g.h_result[6];
    return CSGN_OK;
}

int csgn_shard_range(uint64_t n_blocks, int rank, int world, uint64_t *first, uint64_t *count) {
    if (world < 1 || rank < 0 || rank >= world || !first || !count)
        return fail(CSGN_ERR_INVALID_ARGUMENT, "bad shard arguments (rank %d of %d)", rank, world);
    const uint64_t base = n_blocks / (uint64_t)world, extra = n_blocks % (uint64_t)world;
    const uint64_t r = (uint64_t)rank;
    *first = r * base + std::min<uint64_t>(r, extra);
    *count = base + (r < extra ? 1 : 0);
    return CSGN_OK;
}

}  // extern "C"
