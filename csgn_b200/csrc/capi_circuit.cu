// capi_circuit.cu -- csgn_seg_circuit (include/csgn.h, "ciphertext arrays", circuits): a whole netlist of gates over
// every lane of a set of ciphertext arrays.  The host validates the netlist, computes every wire's last use, stages the
// tables through the pinned staging and makes ONE launch of the circuit kernel (circuit.cu), whose per-lane output
// sizes and fallback flags it reads back (the call's one host synchronisation on the fast path).  Lanes that did not
// fit in their arena slice are evaluated gate by gate with the existing array calls, over gathered copies of their
// inputs; then every output is assembled by one piece copy from the arena and from those results.
#include "capi_internal.cuh"

using namespace csgn;
using namespace csgn::detail;

namespace {

// Without a caller's lane_capacity the arena takes half the free device memory, at most this much.
constexpr uint64_t kArenaMaxBytes = 16ull << 30;
// A lane holds less than 2^31 blocks, so the kernel's 32-bit wire lengths and their products fit.
constexpr uint64_t kLaneMaxBlocks = 1ull << 31;

// An array produced by the gate-by-gate path of the fallback lanes.
struct FallbackWire {
    csgn_buf *b = nullptr;
    std::vector<uint64_t> off;
};

// Gate g starts at gates[at[g]]; checks the encoding, p + q >= 1 and that every operand is a wire below the gate's own.
int parse_gates(const uint32_t *gates, uint64_t gates_len, uint32_t n_gates, uint32_t n_inputs,
                std::vector<uint32_t> *at) {
    if (gates_len > UINT32_MAX)
        return fail(CSGN_ERR_INVALID_ARGUMENT, "gates_len = %llu, at most 2^32 - 1", (unsigned long long)gates_len);
    at->assign(n_gates + 1ull, 0);
    uint64_t pos = 0;
    for (uint32_t gi = 0; gi < n_gates; ++gi) {
        if (gates_len - pos < 2)
            return fail(CSGN_ERR_INVALID_ARGUMENT, "gates_len = %llu ends inside gate %u of %u",
                        (unsigned long long)gates_len, gi, n_gates);
        const uint64_t p = gates[pos], q = gates[pos + 1], len = 2 + 2 * p + q;
        if (p + q == 0) return fail(CSGN_ERR_INVALID_ARGUMENT, "gate %u has no products and no terms", gi);
        if (gates_len - pos < len)
            return fail(CSGN_ERR_INVALID_ARGUMENT, "gates_len = %llu ends inside gate %u of %u",
                        (unsigned long long)gates_len, gi, n_gates);
        const uint64_t wire = (uint64_t)n_inputs + gi;
        for (uint64_t i = pos + 2; i < pos + len; ++i)
            if (gates[i] >= wire)
                return fail(CSGN_ERR_INVALID_ARGUMENT, "gate %u (wire %llu) reads wire %u: operands must be wires below it",
                            gi, (unsigned long long)wire, gates[i]);
        (*at)[gi] = (uint32_t)pos;
        pos += len;
    }
    if (pos != gates_len)
        return fail(CSGN_ERR_INVALID_ARGUMENT, "gates_len = %llu, the %u gates encode %llu words",
                    (unsigned long long)gates_len, n_gates, (unsigned long long)pos);
    (*at)[n_gates] = (uint32_t)pos;
    return CSGN_OK;
}

// The gate-by-gate path over the fallback lanes: the inputs gathered at `lanes`, then each gate with csgn_seg_mul_sum
// (or _compact, and csgn_seg_cancel), every gate wire freed at its last use.  `w` gets the wires still alive.
int run_gate_by_gate(const csgn_buf *const *in, const uint64_t *const *in_off, uint32_t n_inputs, uint64_t n,
                     const std::vector<uint64_t> &lanes, const uint32_t *gates, const std::vector<uint32_t> &at,
                     const std::vector<uint32_t> &frees, const std::vector<uint32_t> &free_at, uint32_t min_bits,
                     bool cancel, std::vector<FallbackWire> *w) {
    const uint64_t m = lanes.size();
    for (uint32_t i = 0; i < n_inputs; ++i) {
        FallbackWire &x = (*w)[i];
        x.off.resize(m + 1);
        const int rc = csgn_seg_gather(in[i], in_off[i], n, lanes.data(), m, x.off.data(), &x.b);
        if (rc != CSGN_OK) return rc;
    }
    const uint32_t n_gates = (uint32_t)at.size() - 1;
    std::vector<const csgn_buf *> a, b, c;
    std::vector<const uint64_t *> ao, bo, co;
    for (uint32_t gi = 0; gi < n_gates; ++gi) {
        const uint32_t *gp = gates + at[gi], p = gp[0], q = gp[1];
        a.clear(), b.clear(), c.clear(), ao.clear(), bo.clear(), co.clear();
        for (uint32_t i = 0; i < p; ++i) {
            const FallbackWire &x = (*w)[gp[2 + 2 * i]], &y = (*w)[gp[3 + 2 * i]];
            a.push_back(x.b), ao.push_back(x.off.data()), b.push_back(y.b), bo.push_back(y.off.data());
        }
        for (uint32_t i = 0; i < q; ++i) {
            const FallbackWire &z = (*w)[gp[2 + 2 * p + i]];
            c.push_back(z.b), co.push_back(z.off.data());
        }
        FallbackWire &o = (*w)[n_inputs + gi];
        o.off.resize(m + 1);
        int rc = min_bits ? csgn_seg_mul_sum_compact(a.data(), ao.data(), b.data(), bo.data(), p, c.data(), co.data(), q,
                                                     m, min_bits, o.off.data(), &o.b)
                          : csgn_seg_mul_sum(a.data(), ao.data(), b.data(), bo.data(), p, c.data(), co.data(), q, m,
                                             o.off.data(), &o.b);
        if (rc == CSGN_OK && cancel) {
            csgn_buf *pre = o.b;
            std::vector<uint64_t> pre_off = o.off;
            o.b = nullptr;
            rc = csgn_seg_cancel(pre, pre_off.data(), m, o.off.data(), &o.b);
            csgn_buf_free(pre);
        }
        if (rc != CSGN_OK) return rc;
        for (uint32_t f = free_at[gi]; f < free_at[gi + 1]; ++f) {
            csgn_buf_free((*w)[frees[f]].b);
            (*w)[frees[f]].b = nullptr;
        }
    }
    return CSGN_OK;
}

}  // namespace

extern "C" {

int csgn_seg_circuit(const csgn_buf *const *in, const uint64_t *const *in_off, uint32_t n_inputs, uint64_t n,
                     const uint32_t *gates, uint64_t gates_len, uint32_t n_gates, const uint32_t *outputs,
                     uint32_t n_outputs, uint32_t min_bits, int cancel, uint64_t lane_capacity,
                     uint64_t *const *out_off, csgn_buf **out, uint64_t *n_fallback) {
    NEED_INIT();
    if (!in || !in_off || !outputs || !out_off || !out || (gates_len && !gates))
        return fail(CSGN_ERR_INVALID_ARGUMENT, "null argument");
    if (n_inputs == 0) return fail(CSGN_ERR_INVALID_ARGUMENT, "a circuit needs at least one input");
    if (n_outputs == 0) return fail(CSGN_ERR_INVALID_ARGUMENT, "a circuit needs at least one output");
    for (uint32_t i = 0; i < n_inputs; ++i)
        if (!in[i]) return fail(CSGN_ERR_INVALID_ARGUMENT, "null input %u", i);
    const uint32_t L = in[0]->L;
    for (uint32_t i = 1; i < n_inputs; ++i)
        if (in[i]->L != L)
            return fail(CSGN_ERR_SHAPE_MISMATCH, "words per block differ (input 0: %u vs input %u: %u)", L, i, in[i]->L);
    if (min_bits > 64ull * L)
        return fail(CSGN_ERR_INVALID_ARGUMENT, "min_bits = %u outside [0, %llu] (64 bits of %u words)", min_bits,
                    64ull * L, L);
    for (uint32_t i = 0; i < n_inputs; ++i) {
        char what[32];
        snprintf(what, sizeof what, "input %u", i);
        const int rc = check_offsets(in[i], in_off[i], n, what);
        if (rc != CSGN_OK) return rc;
    }
    const uint64_t n_wires = (uint64_t)n_inputs + n_gates;
    if (n_wires > UINT32_MAX) return fail(CSGN_ERR_INVALID_ARGUMENT, "more than 2^32 - 1 wires");
    std::vector<uint32_t> at;
    int rc = parse_gates(gates, gates_len, n_gates, n_inputs, &at);
    if (rc != CSGN_OK) return rc;
    bool gate_outputs = false;
    for (uint32_t j = 0; j < n_outputs; ++j) {
        if (outputs[j] >= n_wires)
            return fail(CSGN_ERR_INVALID_ARGUMENT, "output %u names wire %u, the circuit has %llu", j, outputs[j],
                        (unsigned long long)n_wires);
        if (!out_off[j]) return fail(CSGN_ERR_INVALID_ARGUMENT, "null offsets of output %u", j);
        gate_outputs |= outputs[j] >= n_inputs;
    }

    // last uses: a gate wire dies after the last gate that reads it (its own gate when none does), unless it is an output
    std::vector<uint64_t> last(n_gates);
    for (uint32_t gi = 0; gi < n_gates; ++gi) {
        last[gi] = gi;
        for (uint32_t i = at[gi] + 2; i < at[gi + 1]; ++i)
            if (gates[i] >= n_inputs) last[gates[i] - n_inputs] = gi;
    }
    for (uint32_t j = 0; j < n_outputs; ++j)
        if (outputs[j] >= n_inputs) last[outputs[j] - n_inputs] = UINT64_MAX;
    std::vector<uint32_t> free_at(n_gates + 1ull, 0), frees;
    for (uint32_t gi = 0; gi < n_gates; ++gi)
        if (last[gi] != UINT64_MAX) ++free_at[last[gi] + 1];
    for (uint32_t gi = 0; gi < n_gates; ++gi) free_at[gi + 1] += free_at[gi];
    frees.resize(free_at[n_gates]);
    {
        std::vector<uint32_t> fill(free_at.begin(), free_at.end() - 1);
        for (uint32_t gi = 0; gi < n_gates; ++gi)
            if (last[gi] != UINT64_MAX) frees[fill[last[gi]]++] = n_inputs + gi;
    }

    std::vector<const csgn_buf *> bufs(in, in + n_inputs);
    std::stable_sort(bufs.begin(), bufs.end(),
                     [](const csgn_buf *x, const csgn_buf *y) { return x->n_blocks > y->n_blocks; });
    AutoLane lane(bufs[0], bufs.size() > 1 ? bufs[1] : nullptr);
    for (uint32_t i = 0; i < n_inputs; ++i) {
        rc = need_dense(in[i]);
        if (rc != CSGN_OK) return rc;
    }
    for (uint32_t i = 0; i < n_inputs; ++i) acquire_read(in[i]);

    // the lanes' arena slices
    uint64_t cap = lane_capacity;
    if (cap == 0 && n) {
        size_t free_b = 0, total_b = 0;
        CU(cudaMemGetInfo(&free_b, &total_b));
        cap = std::min<uint64_t>(free_b / 2, kArenaMaxBytes) / n / L / sizeof(uint64_t);
    }
    cap = std::min(cap, kLaneMaxBlocks);
    if (n && cap > (UINT64_MAX / 8) / L / n) cap = (UINT64_MAX / 8) / L / n;

    std::vector<uint32_t> flag(n, gate_outputs ? 1u : 0u);   // 1: the lane takes the gate-by-gate path
    std::vector<uint64_t> res;
    DevTable scratch, arena;
    if (gate_outputs && cap && n) {
        // u64 table: input bases, input offsets; u32 table: gates, gate_at, frees, free_at, outputs
        const uint64_t w_off = n_inputs + (uint64_t)n_inputs * (n + 1);
        const uint64_t n32 = gates_len + at.size() + frees.size() + free_at.size() + n_outputs;
        const uint64_t w_tab = w_off + (n32 + 1) / 2;
        std::vector<uint64_t> tab(w_tab, 0);
        for (uint32_t i = 0; i < n_inputs; ++i) {
            tab[i] = (uint64_t)reinterpret_cast<uintptr_t>(in[i]->d);
            memcpy(tab.data() + n_inputs + (uint64_t)i * (n + 1), in_off[i], (n + 1) * sizeof(uint64_t));
        }
        uint32_t *t32 = reinterpret_cast<uint32_t *>(tab.data() + w_off);
        if (gates_len) memcpy(t32, gates, gates_len * sizeof(uint32_t));
        uint32_t *d_at = t32 + gates_len;
        memcpy(d_at, at.data(), at.size() * sizeof(uint32_t));
        uint32_t *d_frees = d_at + at.size();
        if (!frees.empty()) memcpy(d_frees, frees.data(), frees.size() * sizeof(uint32_t));
        uint32_t *d_free_at = d_frees + frees.size();
        memcpy(d_free_at, free_at.data(), free_at.size() * sizeof(uint32_t));
        memcpy(d_free_at + free_at.size(), outputs, n_outputs * sizeof(uint32_t));
        // after the table: the lane counter, the per-lane results (read back with the flags), the wire tables
        const bool units16 = [&] {
            bool u = !(L & 1u);
            for (uint32_t i = 0; i < n_inputs && u; ++i) u = (reinterpret_cast<uintptr_t>(in[i]->d) & 15u) == 0;
            return u;
        }();
        const uint64_t w_res = 2 * n * n_outputs, w_flag = (n + 1) / 2;
        const uint64_t w_wires = (uint64_t)circuit_warps(n, units16, cancel != 0) * n_wires * kCircuitWireBytes / 8;
        uint64_t *d = nullptr, *d_arena = nullptr;
        rc = dev_alloc(w_tab + 2 + w_res + w_flag + w_wires, &d);
        if (rc != CSGN_OK) return rc;
        scratch.d = d;
        rc = dev_alloc(n * cap * L, &d_arena);
        if (rc != CSGN_OK) return rc;
        arena.d = d_arena;
        rc = stage_into(d, tab.data(), w_tab * sizeof(uint64_t));
        if (rc != CSGN_OK) return rc;
        CU(cudaMemsetAsync(d + w_tab, 0, sizeof(uint64_t), g.stream));
        const uint32_t *d32 = reinterpret_cast<const uint32_t *>(d + w_off);
        CircuitArgs args;
        args.gates = d32;
        args.gate_at = d32 + gates_len;
        args.frees = args.gate_at + at.size();
        args.free_at = args.frees + frees.size();
        args.outputs = args.free_at + free_at.size();
        args.in_base = d;
        args.in_off = d + n_inputs;
        args.next = reinterpret_cast<unsigned long long *>(d + w_tab);
        args.res = d + w_tab + 2;
        args.fallback = reinterpret_cast<uint32_t *>(args.res + w_res);
        args.wires = args.res + w_res + w_flag;
        args.arena = d_arena;
        args.n = n;
        args.cap = cap;
        args.n_inputs = n_inputs;
        args.n_gates = n_gates;
        args.n_outputs = n_outputs;
        args.min_bits = min_bits;
        args.cancel = cancel ? 1u : 0u;
        const cudaError_t e = launch_circuit(args, L, units16, g.stream);
        if (e != cudaSuccess) return cuda_fail(e, "circuit kernel");
        res.resize(w_res + w_flag);
        rc = read_back(res.data(), args.res, (w_res + w_flag) * sizeof(uint64_t));
        if (rc != CSGN_OK) return rc;
        memcpy(flag.data(), res.data() + w_res, n * sizeof(uint32_t));
    }

    std::vector<uint64_t> fb_lanes, fb_index(n, 0);
    for (uint64_t k = 0; k < n; ++k)
        if (flag[k]) {
            fb_index[k] = fb_lanes.size();
            fb_lanes.push_back(k);
        }
    std::vector<FallbackWire> fw(n_wires);
    auto release = [&]() {
        for (FallbackWire &x : fw) csgn_buf_free(x.b);
    };
    if (!fb_lanes.empty()) {
        rc = run_gate_by_gate(in, in_off, n_inputs, n, fb_lanes, gates, at, frees, free_at, min_bits, cancel != 0, &fw);
        if (rc != CSGN_OK) {
            release();
            return rc;
        }
    }

    // every output: one piece copy, lane by lane, from the input, the arena or the fallback result
    const uint64_t *d_arena = static_cast<const uint64_t *>(arena.d);
    std::vector<const uint64_t *> src;
    std::vector<uint64_t> words;
    for (uint32_t j = 0; j < n_outputs; ++j) {
        const uint32_t w = outputs[j];
        uint64_t *oo = out_off[j];
        oo[0] = 0;
        src.clear();
        words.clear();
        for (uint64_t k = 0; k < n; ++k) {
            const uint64_t *p;
            uint64_t t;
            if (w < n_inputs) {
                p = in[w]->d + in_off[w][k] * L;
                t = in_off[w][k + 1] - in_off[w][k];
            } else if (!flag[k]) {
                const uint64_t *r = res.data() + 2 * (k * n_outputs + j);
                p = d_arena + (k * cap + r[0]) * L;
                t = r[1];
            } else {
                const FallbackWire &x = fw[w];
                const uint64_t f = fb_index[k];
                p = x.b->d + x.off[f] * L;
                t = x.off[f + 1] - x.off[f];
            }
            if (t) {
                src.push_back(p);
                words.push_back(t * L);
            }
            oo[k + 1] = oo[k] + t;
        }
        rc = check_blocks(oo[n], L);
        if (rc == CSGN_OK) rc = gather_into_new(oo[n], L, src, words, &out[j]);
        if (rc != CSGN_OK) {
            for (uint32_t i = 0; i < j; ++i) {
                csgn_buf_free(out[i]);
                out[i] = nullptr;
            }
            release();
            return rc;
        }
    }
    release();
    if (n_fallback) *n_fallback = fb_lanes.size();
    return CSGN_OK;
}

}  // extern "C"
