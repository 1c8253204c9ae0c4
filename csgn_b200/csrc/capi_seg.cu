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
uint64_t large_words() { return large_bytes() / 8; }

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

// The work of one grouped multiply (seg_mul_kernel), added piece by piece in output order: products, and plain terms
// (items whose left operand is the all-ones block at the head of the staged table).  Small pieces become items packed
// into tasks of about task_words(small_words) words; a long term is cut into items of about one task each.  A piece of
// large_words() or more goes straight into its position: launch_mul for a product, a device-to-device copy for a term.
// The compacting form (out null, then compact()) has no large pieces, since launch_mul and the copy write every block:
// every piece becomes items of about one task, a long row being cut into column ranges.
class SegMulWork {
public:
    SegMulWork(uint32_t L, uint64_t small_words, csgn_buf *out)
        : L_(L), large_(out ? large_words() : UINT64_MAX), target_(task_words(small_words)), out_(out) {}

    void product(const uint64_t *a, uint64_t t1, const uint64_t *b, uint64_t t2) {
        if (t1 && t2 && e_ == cudaSuccess) {
            if (t1 * t2 * L_ >= large_) {
                e_ = launch_mul(a, t1, b, t2, L_, out_->d + pos_ * L_, g.stream);
            } else if (!out_ && t2 * L_ > target_) {
                const uint64_t cols = std::max<uint64_t>(1, target_ / L_);
                for (uint64_t r = 0; r < t1; ++r)
                    for (uint64_t j = 0; j < t2; j += cols) {
                        const uint64_t m = std::min(cols, t2 - j);
                        add({a + r * L_, b + j * L_, pos_ + r * t2 + j, (uint32_t)m, 1}, m * L_);
                    }
            } else {
                const uint64_t row = t2 * L_, step = std::max<uint64_t>(1, target_ / row);
                for (uint64_t r = 0; r < t1; r += step) {
                    const uint64_t rows = std::min(step, t1 - r);
                    add({a + r * L_, b, pos_ + r * t2, (uint32_t)t2, (uint32_t)rows}, rows * row);
                }
            }
        }
        pos_ += t1 * t2;
    }

    void term(const uint64_t *c, uint64_t t) {
        if (t && e_ == cudaSuccess) {
            if (t * L_ >= large_) {
                e_ = cudaMemcpyAsync(out_->d + pos_ * L_, c, t * L_ * sizeof(uint64_t), cudaMemcpyDeviceToDevice, g.stream);
            } else {
                const uint64_t step = std::max<uint64_t>(1, target_ / L_);
                for (uint64_t r = 0; r < t; r += step) {
                    const uint64_t blocks = std::min(step, t - r);
                    add({nullptr, c + r * L_, pos_ + r, (uint32_t)blocks, 1}, blocks * L_);   // a: the ones block
                }
                terms_ = true;
            }
        }
        pos_ += t;
    }

    // Stage the table and make the one grouped launch (none without small pieces).
    int launch() {
        if (e_ != cudaSuccess) return cuda_fail(e_, "grouped multiply kernel");
        if (items_.empty()) return CSGN_OK;
        Table tb;
        int rc = stage(0, &tb);
        if (rc != CSGN_OK) return rc;
        const bool units16 = tb.units16 && (reinterpret_cast<uintptr_t>(out_->d) & 15u) == 0;
        const cudaError_t e = launch_seg_mul(out_->d, L_, units16, tb.items, tb.tasks, n_tasks(), g.stream);
        return e == cudaSuccess ? CSGN_OK : cuda_fail(e, "grouped multiply kernel");
    }

    // The compacting form: count the blocks of at least min_bits set bits of every item (one launch), read the counts
    // back (the call's one host synchronisation), allocate exactly those blocks and write them (a second launch), each
    // item from the total of the items before it, which keeps the blocks of every element in order.  oo: the offsets
    // of the n elements without compaction.  out_off and *out on success only.
    int compact(uint32_t min_bits, const std::vector<uint64_t> &oo, uint64_t *out_off, csgn_buf **out) {
        const uint64_t n = oo.size() - 1;
        const size_t ni = items_.size();
        std::vector<uint64_t> off(n + 1, 0), base(ni);
        csgn_buf *res = nullptr;
        if (ni == 0) {
            const int rc = new_buf(0, L_, 0, &res);
            if (rc != CSGN_OK) return rc;
        } else {
            // after the table: the items' output bases (uint64), then their counts (uint32)
            Table tb;
            int rc = stage(ni * (sizeof(uint64_t) + sizeof(uint32_t)), &tb);
            if (rc != CSGN_OK) return rc;
            uint64_t *d_base = reinterpret_cast<uint64_t *>(tb.extra);
            uint32_t *d_live = reinterpret_cast<uint32_t *>(d_base + ni);
            cudaError_t e = launch_seg_mul_live(nullptr, L_, tb.units16, tb.items, tb.tasks, n_tasks(), min_bits,
                                                d_live, nullptr, g.stream);
            if (e != cudaSuccess) return cuda_fail(e, "grouped multiply kernel (count)");
            std::vector<uint32_t> live(ni);
            rc = read_back(live.data(), d_live, ni * sizeof(uint32_t));
            if (rc != CSGN_OK) return rc;
            uint64_t total = 0;
            for (size_t i = 0, k = 0; i < ni; ++i) {
                while (oo[k + 1] <= items_[i].out) ++k;           // element of item i (items are non-empty)
                base[i] = total;
                total += live[i];
                off[k + 1] += live[i];
            }
            for (uint64_t k = 0; k < n; ++k) off[k + 1] += off[k];
            rc = new_buf(total, L_, 0, &res);
            if (rc != CSGN_OK) return rc;
            acquire_write(res);
            if (total) {
                rc = stage_into(d_base, base.data(), ni * sizeof(uint64_t));
                if (rc == CSGN_OK) {
                    const bool units16 = tb.units16 && (reinterpret_cast<uintptr_t>(res->d) & 15u) == 0;
                    e = launch_seg_mul_live(res->d, L_, units16, tb.items, tb.tasks, n_tasks(), min_bits, nullptr,
                                            d_base, g.stream);
                    if (e != cudaSuccess) rc = cuda_fail(e, "grouped multiply kernel (write)");
                }
                if (rc != CSGN_OK) {
                    csgn_buf_free(res);
                    return rc;
                }
            }
        }
        memcpy(out_off, off.data(), (n + 1) * sizeof(uint64_t));
        *out = res;
        return CSGN_OK;
    }

private:
    // The staged table on the device, released in stream order after the launches that read it.
    struct Table {
        DevTable t;
        const SegMulItem *items = nullptr;
        const uint32_t *tasks = nullptr;
        uint8_t *extra = nullptr;   // `extra` bytes after the table, 8-byte aligned, left to the caller
        bool units16 = false;       // 16-byte units fit the operands and the table (not yet the output)
    };

    uint32_t n_tasks() const { return (uint32_t)(tasks_.size() - 1); }

    // table: [the all-ones block, L words rounded up to 16 bytes, when there are terms] [items] [task bounds]
    int stage(size_t extra, Table *tb) {
        if (tasks_.back() != items_.size()) tasks_.push_back((uint32_t)items_.size());
        if (items_.size() >= UINT32_MAX) return fail(CSGN_ERR_INVALID_ARGUMENT, "too many work items");
        const size_t head = terms_ ? (size_t)((L_ + 1) & ~1u) * sizeof(uint64_t) : 0;
        const size_t item_bytes = items_.size() * sizeof(SegMulItem);
        const size_t bytes = head + item_bytes + tasks_.size() * sizeof(uint32_t);
        const size_t words = (bytes + 7) / 8;
        uint64_t *d = nullptr;
        int rc = dev_alloc(words + (extra + 7) / 8, &d);
        if (rc != CSGN_OK) return rc;
        tb->t.d = d;
        uintptr_t addr = reinterpret_cast<uintptr_t>(d);
        std::vector<uint8_t> tab(bytes);
        std::fill_n(reinterpret_cast<uint64_t *>(tab.data()), head / sizeof(uint64_t), ~0ull);
        SegMulItem *it = reinterpret_cast<SegMulItem *>(tab.data() + head);
        for (size_t i = 0; i < items_.size(); ++i) {
            it[i] = items_[i];
            if (!it[i].a) it[i].a = d;
            addr |= reinterpret_cast<uintptr_t>(it[i].a) | reinterpret_cast<uintptr_t>(it[i].b);
        }
        memcpy(tab.data() + head + item_bytes, tasks_.data(), tasks_.size() * sizeof(uint32_t));
        rc = stage_into(d, tab.data(), bytes);
        if (rc != CSGN_OK) return rc;
        tb->items = reinterpret_cast<const SegMulItem *>(reinterpret_cast<const uint8_t *>(d) + head);
        tb->tasks = reinterpret_cast<const uint32_t *>(tb->items + items_.size());
        tb->extra = reinterpret_cast<uint8_t *>(d + words);
        tb->units16 = !(L_ & 1u) && (addr & 15u) == 0;
        return CSGN_OK;
    }

    void add(const SegMulItem &m, uint64_t words) {
        items_.push_back(m);
        in_task_ += words;
        if (in_task_ >= target_) {
            tasks_.push_back((uint32_t)items_.size());
            in_task_ = 0;
        }
    }

    const uint32_t L_;
    const uint64_t large_, target_;
    csgn_buf *const out_;
    uint64_t pos_ = 0, in_task_ = 0;   // output block of the next piece; words in the open task
    bool terms_ = false;
    cudaError_t e_ = cudaSuccess;
    std::vector<SegMulItem> items_;
    std::vector<uint32_t> tasks_ = std::vector<uint32_t>(1, 0);
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

// csgn_seg_mul_sum, and with compact csgn_seg_mul_sum_compact: the same checks, items and output order, plus
// 1 <= min_bits <= 64 L.
int mul_sum(const csgn_buf *const *a, const uint64_t *const *a_off, const csgn_buf *const *b,
            const uint64_t *const *b_off, uint32_t n_products, const csgn_buf *const *c, const uint64_t *const *c_off,
            uint32_t n_terms, uint64_t n, bool compact, uint32_t min_bits, uint64_t *out_off, csgn_buf **out) {
    if (!out || !out_off) return fail(CSGN_ERR_INVALID_ARGUMENT, "null argument");
    if (n_products == 0 && n_terms == 0) return fail(CSGN_ERR_INVALID_ARGUMENT, "no products and no terms");
    if (n_products && (!a || !a_off || !b || !b_off)) return fail(CSGN_ERR_INVALID_ARGUMENT, "null product arrays");
    if (n_terms && (!c || !c_off)) return fail(CSGN_ERR_INVALID_ARGUMENT, "null term arrays");
    // operand j: the left operands of the products, their right operands, then the terms
    const uint64_t p = n_products, m = p * 2 + n_terms;
    auto op = [&](uint64_t j) { return j < p ? a[j] : j < 2 * p ? b[j - p] : c[j - 2 * p]; };
    auto off = [&](uint64_t j) { return j < p ? a_off[j] : j < 2 * p ? b_off[j - p] : c_off[j - 2 * p]; };
    auto name = [&](uint64_t j) {
        char s[48];
        snprintf(s, sizeof s, "%s %llu", j < p ? "left operand" : j < 2 * p ? "right operand" : "term",
                 (unsigned long long)(j < p ? j : j < 2 * p ? j - p : j - 2 * p));
        return std::string(s);
    };
    for (uint64_t j = 0; j < m; ++j)
        if (!op(j)) return fail(CSGN_ERR_INVALID_ARGUMENT, "null %s", name(j).c_str());
    const uint32_t L = op(0)->L;
    for (uint64_t j = 1; j < m; ++j)
        if (op(j)->L != L)
            return fail(CSGN_ERR_SHAPE_MISMATCH, "words per block differ (%s: %u vs %s: %u)", name(0).c_str(), L,
                        name(j).c_str(), op(j)->L);
    if (compact && (min_bits < 1 || min_bits > 64ull * L))
        return fail(CSGN_ERR_INVALID_ARGUMENT, "min_bits = %u outside [1, %llu] (64 bits of %u words)", min_bits,
                    64ull * L, L);
    for (uint64_t j = 0; j < m; ++j) {
        const int rc = check_offsets(op(j), off(j), n, name(j).c_str());
        if (rc != CSGN_OK) return rc;
    }
    std::vector<uint64_t> oo(n + 1, 0);
    for (uint64_t k = 0; k < n; ++k) {
        uint64_t o = oo[k];
        for (uint64_t i = 0; i < p; ++i) {
            const uint64_t t1 = a_off[i][k + 1] - a_off[i][k], t2 = b_off[i][k + 1] - b_off[i][k];
            if (t2 && t1 > UINT64_MAX / t2)
                return fail(CSGN_ERR_INVALID_ARGUMENT, "product %llu of element %llu overflows", (unsigned long long)i,
                            (unsigned long long)k);
            if (o + t1 * t2 < o) return fail(CSGN_ERR_INVALID_ARGUMENT, "output block count overflows");
            o += t1 * t2;
        }
        for (uint64_t i = 0; i < n_terms; ++i) {
            const uint64_t t = c_off[i][k + 1] - c_off[i][k];
            if (o + t < o) return fail(CSGN_ERR_INVALID_ARGUMENT, "output block count overflows");
            o += t;
        }
        oo[k + 1] = o;
    }
    int rc = check_blocks(oo[n], L);
    if (rc != CSGN_OK) return rc;
    // every distinct buffer once; the automatic lane follows the two largest
    std::vector<const csgn_buf *> bufs;
    for (uint64_t j = 0; j < m; ++j) bufs.push_back(op(j));
    std::sort(bufs.begin(), bufs.end());
    bufs.erase(std::unique(bufs.begin(), bufs.end()), bufs.end());
    std::stable_sort(bufs.begin(), bufs.end(),
                     [](const csgn_buf *x, const csgn_buf *y) { return x->n_blocks > y->n_blocks; });
    AutoLane lane(bufs[0], bufs.size() > 1 ? bufs[1] : nullptr);
    for (const csgn_buf *x : bufs) {
        rc = need_dense(x);
        if (rc != CSGN_OK) return rc;
    }
    csgn_buf *res = nullptr;
    if (!compact) {
        rc = new_buf(oo[n], L, 0, &res);
        if (rc != CSGN_OK) return rc;
    }
    for (const csgn_buf *x : bufs) acquire_read(x);
    if (res) acquire_write(res);
    const uint64_t large = compact ? UINT64_MAX : large_words();
    uint64_t small_words = 0;
    for (uint64_t k = 0; k < n; ++k) {
        for (uint64_t i = 0; i < p; ++i) {
            const uint64_t w = (a_off[i][k + 1] - a_off[i][k]) * (b_off[i][k + 1] - b_off[i][k]) * L;
            if (w < large) small_words += w;
        }
        for (uint64_t i = 0; i < n_terms; ++i) {
            const uint64_t w = (c_off[i][k + 1] - c_off[i][k]) * L;
            if (w < large) small_words += w;
        }
    }
    // output order: element by element, its products first, then its terms
    SegMulWork work(L, small_words, res);
    for (uint64_t k = 0; k < n; ++k) {
        for (uint64_t i = 0; i < p; ++i)
            work.product(a[i]->d + a_off[i][k] * L, a_off[i][k + 1] - a_off[i][k], b[i]->d + b_off[i][k] * L,
                         b_off[i][k + 1] - b_off[i][k]);
        for (uint64_t i = 0; i < n_terms; ++i) work.term(c[i]->d + c_off[i][k] * L, c_off[i][k + 1] - c_off[i][k]);
    }
    if (compact) return work.compact(min_bits, oo, out_off, out);
    rc = work.launch();
    if (rc != CSGN_OK) {
        csgn_buf_free(res);
        return rc;
    }
    memcpy(out_off, oo.data(), (n + 1) * sizeof(uint64_t));
    *out = res;
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
    const uint64_t large = large_words();
    uint64_t small_words = 0;
    for (uint64_t k = 0; k < n; ++k) {
        const uint64_t w = (oo[k + 1] - oo[k]) * L;
        if (w < large) small_words += w;
    }
    SegMulWork work(L, small_words, c);
    for (uint64_t k = 0; k < n; ++k)
        work.product(a->d + a_off[k] * L, a_off[k + 1] - a_off[k], b->d + b_off[k] * L, b_off[k + 1] - b_off[k]);
    rc = work.launch();
    if (rc != CSGN_OK) {
        csgn_buf_free(c);
        return rc;
    }
    memcpy(out_off, oo.data(), (n + 1) * sizeof(uint64_t));
    *out = c;
    return CSGN_OK;
}

int csgn_seg_mul_sum(const csgn_buf *const *a, const uint64_t *const *a_off, const csgn_buf *const *b,
                     const uint64_t *const *b_off, uint32_t n_products, const csgn_buf *const *c,
                     const uint64_t *const *c_off, uint32_t n_terms, uint64_t n, uint64_t *out_off, csgn_buf **out) {
    NEED_INIT();
    return mul_sum(a, a_off, b, b_off, n_products, c, c_off, n_terms, n, false, 0, out_off, out);
}

int csgn_seg_mul_sum_compact(const csgn_buf *const *a, const uint64_t *const *a_off, const csgn_buf *const *b,
                             const uint64_t *const *b_off, uint32_t n_products, const csgn_buf *const *c,
                             const uint64_t *const *c_off, uint32_t n_terms, uint64_t n, uint32_t min_bits,
                             uint64_t *out_off, csgn_buf **out) {
    NEED_INIT();
    return mul_sum(a, a_off, b, b_off, n_products, c, c_off, n_terms, n, true, min_bits, out_off, out);
}

// Every element is cut into tasks of about one task's words (segments.cu, SegCancelTask); element k gets a hash region
// of the power of two >= 2 T_k slots.  One staged allocation holds the task table, the tasks' output bases, then the
// scratch of the three passes: slots and parity bits (zeroed by one memset), first (0x7f bytes), rep, and the tasks'
// survivor counts.
int csgn_seg_cancel(const csgn_buf *c, const uint64_t *c_off, uint64_t n, uint64_t *out_off, csgn_buf **out) {
    NEED_INIT();
    if (!c || !out || !out_off) return fail(CSGN_ERR_INVALID_ARGUMENT, "null argument");
    int rc = check_offsets(c, c_off, n, "ciphertext array");
    if (rc != CSGN_OK) return rc;
    const uint32_t L = c->L;
    const uint64_t T = c->n_blocks;
    const uint64_t target = std::max<uint64_t>(1, task_words(T * L) / L);
    std::vector<SegCancelTask> tasks;
    std::vector<uint64_t> owner;   // element of every task
    uint64_t slots = 0;
    for (uint64_t k = 0; k < n; ++k) {
        const uint64_t t = c_off[k + 1] - c_off[k];
        if (t > kCancelMaxBlocks)
            return fail(CSGN_ERR_INVALID_ARGUMENT, "element %llu holds %llu blocks, more than the 2^30 of one element",
                        (unsigned long long)k, (unsigned long long)t);
        if (t == 0) continue;
        uint64_t cap = 2;
        while (cap < 2 * t) cap <<= 1;
        for (uint64_t i = 0; i < t; i += target) {
            tasks.push_back({c_off[k], slots, (uint32_t)i, (uint32_t)std::min(t, i + target), (uint32_t)(cap - 1), 0});
            owner.push_back(k);
        }
        slots += cap;
    }
    const uint64_t nt = tasks.size();
    if (nt >= UINT32_MAX) return fail(CSGN_ERR_INVALID_ARGUMENT, "too many work items");
    AutoLane lane(c);
    rc = need_dense(c);
    if (rc != CSGN_OK) return rc;
    acquire_read(c);
    std::vector<uint64_t> off(n + 1, 0);
    csgn_buf *res = nullptr;
    if (nt == 0) {   // no blocks
        rc = new_buf(0, L, 0, &res);
        if (rc != CSGN_OK) return rc;
        memcpy(out_off, off.data(), (n + 1) * sizeof(uint64_t));
        *out = res;
        return CSGN_OK;
    }
    // words: tasks, bases, then slots + parity (uint32 each, zeroed together), first, rep, live
    const uint64_t w_tab = nt * sizeof(SegCancelTask) / 8, w_zero = slots / 2 + (T + 63) / 64, w_t = (T + 1) / 2;
    uint64_t *d = nullptr;
    rc = dev_alloc(w_tab + nt + w_zero + 2 * w_t + (nt + 1) / 2, &d);
    if (rc != CSGN_OK) return rc;
    DevTable scratch;
    scratch.d = d;
    const SegCancelTask *d_tasks = reinterpret_cast<const SegCancelTask *>(d);
    uint64_t *d_base = d + w_tab, *zero = d_base + nt;
    SegCancelScratch s;
    s.slots = reinterpret_cast<uint32_t *>(zero);
    s.parity = s.slots + slots;
    s.first = reinterpret_cast<int32_t *>(zero + w_zero);
    s.rep = reinterpret_cast<int32_t *>(zero + w_zero + w_t);
    uint32_t *d_live = reinterpret_cast<uint32_t *>(zero + w_zero + 2 * w_t);
    rc = stage_into(d, tasks.data(), nt * sizeof(SegCancelTask));
    if (rc != CSGN_OK) return rc;
    CU(cudaMemsetAsync(zero, 0, w_zero * sizeof(uint64_t), g.stream));
    CU(cudaMemsetAsync(s.first, 0x7f, T * sizeof(int32_t), g.stream));
    const bool units16 = !(L & 1u) && (reinterpret_cast<uintptr_t>(c->d) & 15u) == 0;
    cudaError_t e = launch_seg_cancel_insert(c->d, L, units16, d_tasks, (uint32_t)nt, s, g.stream);
    if (e == cudaSuccess) e = launch_seg_cancel_count(d_tasks, (uint32_t)nt, s, d_live, g.stream);
    if (e != cudaSuccess) return cuda_fail(e, "cancellation kernel");
    std::vector<uint32_t> live(nt);
    rc = read_back(live.data(), d_live, nt * sizeof(uint32_t));
    if (rc != CSGN_OK) return rc;
    // every task's base is the total of the tasks before it, which keeps the survivors of every element in order
    std::vector<uint64_t> base(nt);
    uint64_t total = 0;
    for (uint64_t t = 0; t < nt; ++t) {
        base[t] = total;
        total += live[t];
        off[owner[t] + 1] += live[t];
    }
    for (uint64_t k = 0; k < n; ++k) off[k + 1] += off[k];
    rc = new_buf(total, L, 0, &res);
    if (rc != CSGN_OK) return rc;
    acquire_write(res);
    if (total) {
        rc = stage_into(d_base, base.data(), nt * sizeof(uint64_t));
        if (rc == CSGN_OK) {
            const bool out16 = units16 && (reinterpret_cast<uintptr_t>(res->d) & 15u) == 0;
            e = launch_seg_cancel_write(c->d, L, out16, d_tasks, (uint32_t)nt, s, d_base, res->d, g.stream);
            if (e != cudaSuccess) rc = cuda_fail(e, "cancellation kernel (write)");
        }
        if (rc != CSGN_OK) {
            csgn_buf_free(res);
            return rc;
        }
    }
    memcpy(out_off, off.data(), (n + 1) * sizeof(uint64_t));
    *out = res;
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
    const uint64_t large = large_words();
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
