// capi_seg.cu -- the "ciphertext arrays" section of include/csgn.h: n independent ciphertexts held as ONE dense buffer
// plus host block offsets (element k = blocks [off[k], off[k+1])).  Every entry point validates the offsets on the
// host, builds the kernels' work tables from them, copies the tables through the pinned staging (no host
// synchronisation) and makes one launch for all small elements (segments.cu, misc.cu's piece copy).  Elements above
// kSegLargeBytes go to the tuned single-ciphertext kernels, one launch each, straight into the output array.
#include "capi_internal.cuh"

using namespace csgn;
using namespace csgn::detail;

namespace {

// Products (multiply) and elements (decrypt) of at least this many bytes run on launch_mul / launch_decrypt_count,
// where one launch per element costs little against the element's own traffic.  Not yet set from a measurement:
// tools/seg_bench.py's sweep compares both sides of it, with CSGN_SEG_LARGE_BYTES overriding it.
constexpr long kSegLargeBytes = 8l << 20;
// Warps resident at once (segments.cu: 8 CTAs of 8 warps per SM); the work of the small elements is cut into about
// two tasks per resident warp, within these bounds (in words).
constexpr uint64_t kSegTaskMinWords = 1024, kSegTaskMaxWords = 32768;

uint64_t large_bytes() { return (uint64_t)std::max(0l, env_long("CSGN_SEG_LARGE_BYTES", kSegLargeBytes)); }

uint64_t task_words(uint64_t total_words) {
    const uint64_t warps = (uint64_t)device_props().sm_count * 8 * 8;
    return std::min(kSegTaskMaxWords, std::max(kSegTaskMinWords, total_words / (2 * warps)));
}

int check_offsets(const csgn_buf *buf, const uint64_t *off, uint64_t n, const char *what) {
    if (!off) return fail(CSGN_ERR_INVALID_ARGUMENT, "%s: null offsets", what);
    if (off[0] != 0)
        return fail(CSGN_ERR_INVALID_ARGUMENT, "%s: offsets[0] = %llu, must be 0", what, (unsigned long long)off[0]);
    for (uint64_t k = 0; k < n; ++k)
        if (off[k + 1] < off[k])
            return fail(CSGN_ERR_INVALID_ARGUMENT, "%s: offsets decrease at element %llu (%llu -> %llu)", what,
                        (unsigned long long)k, (unsigned long long)off[k], (unsigned long long)off[k + 1]);
    if (off[n] != buf->n_blocks)
        return fail(CSGN_ERR_SHAPE_MISMATCH, "%s: offsets[%llu] = %llu, the storage holds %llu blocks", what,
                    (unsigned long long)n, (unsigned long long)off[n], (unsigned long long)buf->n_blocks);
    return CSGN_OK;
}

int check_blocks(uint64_t total, uint32_t L) {
    if (total > (UINT64_MAX / 8) / L) return fail(CSGN_ERR_INVALID_ARGUMENT, "output block count overflows");
    return CSGN_OK;
}

// A device table, released in stream order after the launches that read it.
struct DevTable {
    void *d = nullptr;
    ~DevTable() { dev_free(d); }
};

// out = src[0] || src[1] || ... (words[p] words from src[p]) in one launch of the piece copy.
int copy_pieces(const std::vector<const uint64_t *> &src, const std::vector<uint64_t> &words, csgn_buf *out) {
    const size_t n = src.size();
    if (n == 0) return CSGN_OK;
    if (n >= UINT32_MAX) return fail(CSGN_ERR_INVALID_ARGUMENT, "more than 2^32 - 2 pieces to copy");
    bool u16 = (reinterpret_cast<uintptr_t>(out->d) & 15u) == 0;
    for (size_t p = 0; p < n && u16; ++p) u16 = (reinterpret_cast<uintptr_t>(src[p]) & 15u) == 0 && words[p] % 2 == 0;
    // table: n + 1 destination offsets (units), then n source pointers
    std::vector<uint64_t> tab(2 * n + 1);
    for (size_t p = 0; p < n; ++p) {
        tab[p + 1] = tab[p] + (u16 ? words[p] / 2 : words[p]);
        tab[n + 1 + p] = (uint64_t)reinterpret_cast<uintptr_t>(src[p]);
    }
    DevTable t;
    int rc = stage_to_device(tab.data(), tab.size() * sizeof(uint64_t), &t.d);
    if (rc != CSGN_OK) return rc;
    const uint64_t *d = static_cast<const uint64_t *>(t.d);
    cudaError_t e = launch_piece_copy(reinterpret_cast<const void *const *>(d + n + 1), d, (uint32_t)n, tab[n], u16,
                                      out->d, g.stream);
    return e == cudaSuccess ? CSGN_OK : cuda_fail(e, "piece copy kernel");
}

// Allocate an output of `blocks` blocks and fill it from `src`/`words`; *out only on success.
int gather_into_new(uint64_t blocks, uint32_t L, const std::vector<const uint64_t *> &src,
                    const std::vector<uint64_t> &words, csgn_buf **out) {
    csgn_buf *c = nullptr;
    int rc = new_buf(blocks, L, 0, &c);
    if (rc != CSGN_OK) return rc;
    acquire_write(c);
    rc = copy_pieces(src, words, c);
    if (rc != CSGN_OK) {
        csgn_buf_free(c);
        return rc;
    }
    *out = c;
    return CSGN_OK;
}

}  // namespace

extern "C" {

int csgn_seg_mul(const csgn_buf *a, const uint64_t *a_off, const csgn_buf *b, const uint64_t *b_off, uint64_t n,
                 uint64_t *out_off, csgn_buf **out) {
    NEED_INIT();
    if (!a || !b || !out || !out_off) return fail(CSGN_ERR_INVALID_ARGUMENT, "null argument");
    if (a->L != b->L) return fail(CSGN_ERR_SHAPE_MISMATCH, "words per block differ (%u vs %u)", a->L, b->L);
    int rc = check_offsets(a, a_off, n, "left operand");
    if (rc == CSGN_OK) rc = check_offsets(b, b_off, n, "right operand");
    if (rc != CSGN_OK) return rc;
    const uint32_t L = a->L;
    std::vector<uint64_t> oo(n + 1, 0);
    for (uint64_t k = 0; k < n; ++k) {
        const uint64_t t1 = a_off[k + 1] - a_off[k], t2 = b_off[k + 1] - b_off[k];
        if (t2 && t1 > UINT64_MAX / t2) return fail(CSGN_ERR_INVALID_ARGUMENT, "product %llu overflows", (unsigned long long)k);
        if (oo[k] + t1 * t2 < oo[k]) return fail(CSGN_ERR_INVALID_ARGUMENT, "output block count overflows");
        oo[k + 1] = oo[k] + t1 * t2;
    }
    rc = check_blocks(oo[n], L);
    if (rc != CSGN_OK) return rc;
    AutoLane lane(a, b);
    rc = need_dense(a);
    if (rc == CSGN_OK) rc = need_dense(b);
    if (rc != CSGN_OK) return rc;
    csgn_buf *c = nullptr;
    rc = new_buf(oo[n], L, 0, &c);
    if (rc != CSGN_OK) return rc;
    acquire_read(a);
    acquire_read(b);
    acquire_write(c);
    // work items: small products whole or cut into row ranges of about one task each, packed into tasks in element
    // order; large products: one launch_mul each
    const uint64_t large = large_bytes() / 8;
    uint64_t small_words = 0;
    for (uint64_t k = 0; k < n; ++k) {
        const uint64_t w = (oo[k + 1] - oo[k]) * L;
        if (w < large) small_words += w;
    }
    const uint64_t target = task_words(small_words);
    std::vector<SegMulItem> items;
    std::vector<uint32_t> tasks(1, 0);
    uint64_t in_task = 0;
    cudaError_t e = cudaSuccess;
    for (uint64_t k = 0; k < n && e == cudaSuccess; ++k) {
        const uint64_t t1 = a_off[k + 1] - a_off[k], t2 = b_off[k + 1] - b_off[k];
        if (t1 == 0 || t2 == 0) continue;
        if (t1 * t2 * L >= large) {
            e = launch_mul(a->d + a_off[k] * L, t1, b->d + b_off[k] * L, t2, L, c->d + oo[k] * L, g.stream);
            continue;
        }
        const uint64_t row = t2 * L, step = std::max<uint64_t>(1, target / row);
        for (uint64_t r = 0; r < t1; r += step) {
            const uint64_t rows = std::min(step, t1 - r);
            items.push_back({a_off[k] + r, b_off[k], oo[k] + r * t2, (uint32_t)t2, (uint32_t)rows});
            in_task += rows * row;
            if (in_task >= target) {
                tasks.push_back((uint32_t)items.size());
                in_task = 0;
            }
        }
    }
    if (tasks.back() != items.size()) tasks.push_back((uint32_t)items.size());
    if (e == cudaSuccess && !items.empty()) {
        if (items.size() >= UINT32_MAX) {
            csgn_buf_free(c);
            return fail(CSGN_ERR_INVALID_ARGUMENT, "too many work items");
        }
        std::vector<uint8_t> tab(items.size() * sizeof(SegMulItem) + tasks.size() * sizeof(uint32_t));
        memcpy(tab.data(), items.data(), items.size() * sizeof(SegMulItem));
        memcpy(tab.data() + items.size() * sizeof(SegMulItem), tasks.data(), tasks.size() * sizeof(uint32_t));
        DevTable t;
        rc = stage_to_device(tab.data(), tab.size(), &t.d);
        if (rc != CSGN_OK) {
            csgn_buf_free(c);
            return rc;
        }
        const SegMulItem *d_items = static_cast<const SegMulItem *>(t.d);
        e = launch_seg_mul(a->d, b->d, c->d, L, d_items, reinterpret_cast<const uint32_t *>(d_items + items.size()),
                           (uint32_t)(tasks.size() - 1), g.stream);
    }
    if (e != cudaSuccess) {
        csgn_buf_free(c);
        return cuda_fail(e, "grouped multiply kernel");
    }
    memcpy(out_off, oo.data(), (n + 1) * sizeof(uint64_t));
    *out = c;
    return CSGN_OK;
}

int csgn_seg_concat(const csgn_buf *a, const uint64_t *a_off, const csgn_buf *b, const uint64_t *b_off, uint64_t n,
                    uint64_t *out_off, csgn_buf **out) {
    NEED_INIT();
    if (!a || !b || !out || !out_off) return fail(CSGN_ERR_INVALID_ARGUMENT, "null argument");
    if (a->L != b->L) return fail(CSGN_ERR_SHAPE_MISMATCH, "words per block differ (%u vs %u)", a->L, b->L);
    int rc = check_offsets(a, a_off, n, "left operand");
    if (rc == CSGN_OK) rc = check_offsets(b, b_off, n, "right operand");
    if (rc == CSGN_OK && a->n_blocks + b->n_blocks < a->n_blocks)
        rc = fail(CSGN_ERR_INVALID_ARGUMENT, "output block count overflows");
    if (rc == CSGN_OK) rc = check_blocks(a->n_blocks + b->n_blocks, a->L);
    if (rc != CSGN_OK) return rc;
    const uint32_t L = a->L;
    AutoLane lane(a, b);
    rc = need_dense(a);
    if (rc == CSGN_OK) rc = need_dense(b);
    if (rc != CSGN_OK) return rc;
    acquire_read(a);
    acquire_read(b);
    std::vector<const uint64_t *> src;
    std::vector<uint64_t> words;
    for (uint64_t k = 0; k < n; ++k) {
        const uint64_t ta = a_off[k + 1] - a_off[k], tb = b_off[k + 1] - b_off[k];
        if (ta) {
            src.push_back(a->d + a_off[k] * L);
            words.push_back(ta * L);
        }
        if (tb) {
            src.push_back(b->d + b_off[k] * L);
            words.push_back(tb * L);
        }
    }
    rc = gather_into_new(a->n_blocks + b->n_blocks, L, src, words, out);
    if (rc != CSGN_OK) return rc;
    for (uint64_t k = 0; k <= n; ++k) out_off[k] = a_off[k] + b_off[k];
    return CSGN_OK;
}

int csgn_seg_gather(const csgn_buf *src, const uint64_t *src_off, uint64_t n_src, const uint64_t *idx, uint64_t m,
                    uint64_t *out_off, csgn_buf **out) {
    NEED_INIT();
    if (!src || !out || !out_off || (m && !idx)) return fail(CSGN_ERR_INVALID_ARGUMENT, "null argument");
    int rc = check_offsets(src, src_off, n_src, "source");
    if (rc != CSGN_OK) return rc;
    const uint32_t L = src->L;
    std::vector<uint64_t> oo(m + 1, 0);
    for (uint64_t j = 0; j < m; ++j) {
        if (idx[j] >= n_src)
            return fail(CSGN_ERR_INVALID_ARGUMENT, "idx[%llu] = %llu outside the %llu source elements",
                        (unsigned long long)j, (unsigned long long)idx[j], (unsigned long long)n_src);
        const uint64_t t = src_off[idx[j] + 1] - src_off[idx[j]];
        if (oo[j] + t < oo[j]) return fail(CSGN_ERR_INVALID_ARGUMENT, "output block count overflows");
        oo[j + 1] = oo[j] + t;
    }
    rc = check_blocks(oo[m], L);
    if (rc != CSGN_OK) return rc;
    AutoLane lane(src);
    rc = need_dense(src);
    if (rc != CSGN_OK) return rc;
    acquire_read(src);
    std::vector<const uint64_t *> p;
    std::vector<uint64_t> words;
    for (uint64_t j = 0; j < m; ++j)
        if (oo[j + 1] > oo[j]) {
            p.push_back(src->d + src_off[idx[j]] * L);
            words.push_back((oo[j + 1] - oo[j]) * L);
        }
    rc = gather_into_new(oo[m], L, p, words, out);
    if (rc != CSGN_OK) return rc;
    memcpy(out_off, oo.data(), (m + 1) * sizeof(uint64_t));
    return CSGN_OK;
}

int csgn_concat_n(const csgn_buf *const *parts, uint64_t n, csgn_buf **out) {
    NEED_INIT();
    if (!parts || !out || n == 0) return fail(CSGN_ERR_INVALID_ARGUMENT, "no parts");
    uint64_t total = 0;
    for (uint64_t i = 0; i < n; ++i) {
        if (!parts[i]) return fail(CSGN_ERR_INVALID_ARGUMENT, "null part %llu", (unsigned long long)i);
        if (parts[i]->L != parts[0]->L)
            return fail(CSGN_ERR_SHAPE_MISMATCH, "part %llu has %u words per block, part 0 has %u", (unsigned long long)i,
                        parts[i]->L, parts[0]->L);
        if (total + parts[i]->n_blocks < total) return fail(CSGN_ERR_INVALID_ARGUMENT, "output block count overflows");
        total += parts[i]->n_blocks;
    }
    const uint32_t L = parts[0]->L;
    int rc = check_blocks(total, L);
    if (rc != CSGN_OK) return rc;
    AutoLane lane(parts[0]);
    std::vector<const uint64_t *> src;
    std::vector<uint64_t> words;
    for (uint64_t i = 0; i < n; ++i) {
        rc = need_dense(parts[i]);
        if (rc != CSGN_OK) return rc;
        acquire_read(parts[i]);
        if (parts[i]->n_blocks) {
            src.push_back(parts[i]->d);
            words.push_back(parts[i]->n_blocks * L);
        }
    }
    return gather_into_new(total, L, src, words, out);
}

int csgn_seg_decrypt_count_async(const csgn_buf *c, const uint64_t *c_off, uint64_t n, const csgn_key *key,
                                 uint64_t *device_counts) {
    NEED_INIT();
    if (!c || !key || (n && !device_counts)) return fail(CSGN_ERR_INVALID_ARGUMENT, "null argument");
    if (c->L != key->L)
        return fail(CSGN_ERR_SHAPE_MISMATCH, "ciphertext has %u words per block, key expects %u", c->L, key->L);
    int rc = check_offsets(c, c_off, n, "ciphertext array");
    if (rc != CSGN_OK || n == 0) return rc;
    const uint32_t L = c->L;
    rc = need_dense(c);
    if (rc != CSGN_OK) return rc;
    acquire_read(c);
    CU(cudaMemsetAsync(device_counts, 0, n * sizeof(uint64_t), g.stream));
    // tasks: runs of consecutive small elements cut into pieces of about `target` blocks; large elements: one fold each
    const uint64_t large = large_bytes() / 8;
    uint64_t small_words = 0;
    for (uint64_t k = 0; k < n; ++k) {
        const uint64_t w = (c_off[k + 1] - c_off[k]) * L;
        if (w < large) small_words += w;
    }
    const uint64_t target = std::max<uint64_t>(1, task_words(small_words) / L);
    const uint64_t *hm = key->h_mask.empty() ? nullptr : key->h_mask.data();
    std::vector<SegDecTask> tasks;
    SegDecTask cur = {0, 0, 0, 0};
    bool open = false;
    auto close = [&]() {
        if (open) tasks.push_back(cur);
        open = false;
    };
    cudaError_t e = cudaSuccess;
    for (uint64_t k = 0; k < n && e == cudaSuccess; ++k) {
        const uint64_t o0 = c_off[k], o1 = c_off[k + 1];
        if (o0 == o1) continue;
        if ((o1 - o0) * L >= large) {
            close();
            e = launch_decrypt_count(c->d + o0 * L, o1 - o0, L, key->d_mask, hm, fold_scratch(), device_counts + k,
                                     g.stream, nullptr, folds_overlap());
            continue;
        }
        for (uint64_t p = o0; p < o1;) {
            if (!open) {
                cur = {p, p, k, k};
                open = true;
            }
            const uint64_t take = std::min(o1 - p, target - (cur.end - cur.first));
            cur.end = p + take;
            cur.elem_last = k;
            p += take;
            if (cur.end - cur.first >= target) close();
        }
    }
    close();
    if (e == cudaSuccess && !tasks.empty()) {
        if (tasks.size() >= UINT32_MAX) return fail(CSGN_ERR_INVALID_ARGUMENT, "too many work items");
        std::vector<uint64_t> tab((n + 1) + tasks.size() * 4);
        memcpy(tab.data(), c_off, (n + 1) * sizeof(uint64_t));
        memcpy(tab.data() + n + 1, tasks.data(), tasks.size() * sizeof(SegDecTask));
        DevTable t;
        rc = stage_to_device(tab.data(), tab.size() * sizeof(uint64_t), &t.d);
        if (rc != CSGN_OK) return rc;
        const uint64_t *d = static_cast<const uint64_t *>(t.d);
        e = launch_seg_decrypt(c->d, L, key->d_mask, d, reinterpret_cast<const SegDecTask *>(d + n + 1),
                               (uint32_t)tasks.size(), device_counts, g.stream);
    }
    return e == cudaSuccess ? CSGN_OK : cuda_fail(e, "segmented decrypt kernel");
}

int csgn_seg_decrypt(const csgn_buf *c, const uint64_t *c_off, uint64_t n, const csgn_key *key, uint8_t *bits,
                     uint64_t *counts) {
    NEED_INIT();
    if (!bits && !counts) return fail(CSGN_ERR_INVALID_ARGUMENT, "no output");
    if (!c || !key) return fail(CSGN_ERR_INVALID_ARGUMENT, "null argument");
    if (c->L != key->L)
        return fail(CSGN_ERR_SHAPE_MISMATCH, "ciphertext has %u words per block, key expects %u", c->L, key->L);
    int rc = check_offsets(c, c_off, n, "ciphertext array");
    if (rc != CSGN_OK || n == 0) return rc;
    uint64_t *d = nullptr;
    rc = dev_alloc(n, &d);
    if (rc != CSGN_OK) return rc;
    rc = csgn_seg_decrypt_count_async(c, c_off, n, key, d);
    std::vector<uint64_t> h(n);
    cudaError_t e = cudaSuccess;
    if (rc == CSGN_OK) {
        e = cudaMemcpyAsync(h.data(), d, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, g.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g.stream);
        if (e == cudaSuccess) note_synced(g.stream);
    }
    dev_free(d);
    if (rc != CSGN_OK) return rc;
    if (e != cudaSuccess) return cuda_fail(e, "array decrypt readback");
    for (uint64_t k = 0; k < n; ++k) {
        if (bits) bits[k] = (uint8_t)(h[k] & 1u);
        if (counts) counts[k] = h[k];
    }
    return CSGN_OK;
}

}  // extern "C"
