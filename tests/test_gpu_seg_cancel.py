"""Cancellation on ciphertext arrays (csgn_seg_cancel; CiphertextArray.cancel(), Ciphertext.cancel();
CiphertextArray::cancel in C++): element k keeps, in order, the first occurrence of every block value that occurs an odd
number of times in element k.  Checked word for word against a numpy restatement, and under random keys against the
decryptions before the call (same bits, counts lower by an even number)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle.pyoracle import random_blocks, random_key, words_per_block

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NS = [64, 191, 1247, 4097, 16383, 33000]          # L = 1, 3, 20, 65, 256, 516
DISTS = ["one", "rand", "mixed"]
PATTERNS = ["none", "pairs", "multi", "single"]   # duplicates: none, pairs, multiplicities 1-5, one repeated value
BIT = np.uint64(1) << np.uint64(63)               # the first bit of a word (valid in every word, the last one too)

pytestmark = pytest.mark.gpu


def _cancelled(elements, L):
    """the numpy restatement: per element, the first occurrence of every row that occurs an odd number of times, in
    order"""
    out = []
    for w in elements:
        rows = np.ascontiguousarray(w).reshape(-1, L)
        keep = np.zeros(rows.shape[0], dtype=bool)
        if rows.shape[0]:
            _, first, counts = np.unique(rows, axis=0, return_index=True, return_counts=True)
            keep[first[counts % 2 == 1]] = True
        out.append(rows[keep].reshape(-1))
    return out


def _with_repeats(rng, t, N, pattern):
    """t blocks of N bits whose values repeat as `pattern` says, interleaved at random"""
    L = words_per_block(N)
    if pattern == "none" or t == 0:
        return random_blocks(rng, t, N)
    if pattern == "pairs":
        vals = random_blocks(rng, (t + 1) // 2, N).reshape(-1, L)
        idx = np.repeat(np.arange(vals.shape[0]), 2)[:t]
    elif pattern == "single":
        vals = random_blocks(rng, 1, N).reshape(-1, L)
        idx = np.zeros(t, dtype=np.int64)
    else:
        mult = rng.integers(1, 6, size=t)
        idx = np.repeat(np.arange(t), mult)[:t]
        vals = random_blocks(rng, t, N).reshape(-1, L)
    return vals[idx[rng.permutation(t)]].reshape(-1)


def _sizes(dist, rng, n, L):
    if dist == "one":
        return np.ones(n, dtype=np.int64)
    s = rng.integers(0, 9, size=n)
    s[::7] = 0
    if dist == "mixed":                  # elements of several tasks (a task holds about 1024 words or more)
        s[3::11] = rng.integers(40, 90, size=s[3::11].size)
        s[5] = 3 * max(1, 1024 // L) + 7
    return s


def _offsets(sizes):
    off = np.zeros(len(sizes) + 1, dtype=np.uint64)
    off[1:] = np.cumsum(sizes)
    return off


def _check_elements(arr, want):
    assert len(arr) == len(want)
    assert np.array_equal(arr.offsets, _offsets([w.size // arr.ctx.L for w in want]))
    got = arr.to_host()
    for k, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g, w), "element %d differs" % k


def _same(x, y):
    return np.array_equal(x.offsets, y.offsets) and np.array_equal(x.storage.getValues(), y.storage.getValues())


@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("dist", DISTS)
def test_cancel_matches_the_restatement(engine, N, dist):
    L = words_per_block(N)
    rng = np.random.default_rng(N * 7 + DISTS.index(dist))
    ctx = engine.Context(N, 16 if N >= 64 else 4)
    n = 40 if L > 100 else 120
    for pattern in PATTERNS:
        sizes = _sizes(dist, rng, n, L)
        host = [_with_repeats(rng, t, N, pattern if pattern != "single" or k == 5 else "multi")
                for k, t in enumerate(sizes)]
        X = engine.CiphertextArray.from_host(host, ctx)
        want = _cancelled(host, L)
        G = X.cancel()
        _check_elements(G, want)
        if pattern == "none" or dist == "one":
            assert G.offsets[-1] == X.offsets[-1]
        else:
            assert G.offsets[-1] < X.offsets[-1], pattern
        assert _same(G, X.cancel()), pattern                              # two calls, the same words and offsets
        assert _same(G.cancel(), G), pattern                              # idempotent


@pytest.mark.parametrize("N", [1247, 4097, 33000])
def test_near_misses_and_colliding_slots_are_kept(engine, N):
    """Blocks one bit apart (in the first, a middle and the last word) are different values; many distinct blocks in
    small elements share their first slots and must all be kept."""
    L = words_per_block(N)
    rng = np.random.default_rng(5 + N)
    ctx = engine.Context(N, 16)
    b = random_blocks(rng, 1, N)
    near = []
    for w in (0, L // 2, L - 1):
        v = b.copy()
        v[w] ^= BIT
        near.append(v)
    elems = [np.concatenate([b, near[0], near[1], near[2], b, near[0]]), np.concatenate([near[0], b, near[1]]),
             np.concatenate(near + [b])]
    # two to six distinct values in regions of 4 .. 16 slots, each value once or three times
    for _ in range(300):
        k = int(rng.integers(2, 7))
        vals = random_blocks(rng, k, N).reshape(-1, L)
        idx = np.repeat(np.arange(k), rng.choice([1, 3], size=k))
        elems.append(vals[idx[rng.permutation(idx.size)]].reshape(-1))
    X = engine.CiphertextArray.from_host(elems, ctx)
    want = _cancelled(elems, L)
    assert want[0].size == 2 * L and want[1].size == 3 * L and want[2].size == 4 * L
    G = X.cancel()
    _check_elements(G, want)
    assert G.offsets[-1] == sum(w.size for w in want[3:]) // L + 9


def _mix64(x):
    x = x ^ (x >> np.uint64(30))
    x = x * np.uint64(0xbf58476d1ce4e5b9)
    x = x ^ (x >> np.uint64(27))
    x = x * np.uint64(0x94d049bb133111eb)
    return x ^ (x >> np.uint64(31))


def _start_slots(rows, cap):
    """segments.cu's first probe slot of every row (L words) in a region of cap slots: the finaliser of the sum over the
    words of mix64(word + (w + 1) * golden)"""
    w = np.arange(rows.shape[1], dtype=np.uint64) + np.uint64(1)
    with np.errstate(over="ignore"):
        h = _mix64(rows + w * np.uint64(0x9e3779b97f4a7c15)).sum(axis=1, dtype=np.uint64)
        return _mix64(h) & np.uint64(cap - 1)


@pytest.mark.parametrize("N", [191, 1247, 4097, 33000])
def test_blocks_differing_in_one_word_meet_and_stay_apart(engine, N):
    """Equality is decided on all L words.  For each of the first, a middle and the last word, one element holds a base
    block and variants that differ from it in that word only, chosen so that every one of them starts probing at the
    base's slot: each variant is compared with the base and with the variants inserted before it, and only that word
    tells them apart.  Some variants repeat, so the element also cancels.  N = 191 (3 units) and 1247 (10 16-byte units)
    take the group path, where one lane probes and compares; 4097 and 33000 the whole-warp path; a misaligned view of
    the same words takes 8-byte units, which puts N = 1247 (20 units) on the whole-warp path too."""
    import torch
    L = words_per_block(N)
    rng = np.random.default_rng(11 + N)
    ctx = engine.Context(N, 16)
    K = 12
    T = 1 + K + K // 2                                 # base, K variants, every other variant again
    cap = 1
    while cap < 2 * T:
        cap <<= 1
    elems = []
    for w in sorted({0, L // 2, L - 1}):
        b = random_blocks(rng, 1, N).reshape(1, L)
        s0 = _start_slots(b, cap)[0]
        cand = np.repeat(b, 4096, axis=0)
        # any bits of word w: the call compares raw words (pad bits too; the last word of N = 4097 has one valid bit)
        cand[:, w] ^= rng.integers(1, 2**63, size=4096, dtype=np.uint64)
        cand = np.unique(cand[_start_slots(cand, cap) == s0], axis=0)
        cand = cand[~(cand == b).all(axis=1)]
        assert cand.shape[0] >= K, (w, cand.shape[0])
        var = cand[rng.permutation(cand.shape[0])[:K]]
        elems.append(np.concatenate([var[:4], b, var[4:], var[::2]]).reshape(-1))
    want = _cancelled(elems, L)
    assert all(x.size == (1 + K // 2) * L for x in want)
    X = engine.CiphertextArray.from_host(elems, ctx)
    _check_elements(X.cancel(), want)
    flat = np.concatenate(elems)
    t = torch.zeros(flat.size + 1, dtype=torch.int64, device="cuda")
    t[1:] = torch.from_numpy(flat.view(np.int64)).cuda()
    torch.cuda.synchronize()
    view = engine.Ciphertext.view(t.data_ptr() + 8, flat.size // L, ctx, keepalive=t)      # 8 bytes off 16-byte alignment
    _check_elements(engine.CiphertextArray(view, X.offsets.copy()).cancel(), want)


def test_square_and_double_cancel(engine, oracle):
    N = 1247
    L = words_per_block(N)
    rng = np.random.default_rng(17)
    ctx = engine.Context(N, 16)
    sizes = _sizes("rand", rng, 200, L)
    host = [random_blocks(rng, int(t), N) for t in sizes]
    X = engine.CiphertextArray.from_host(host, ctx)
    S = (X * X).cancel()                       # x_i & x_i = x_i first; (i, j) and (j, i) cancel
    _check_elements(S, host)
    D = (X + X).cancel()
    assert D.storage.n_blocks == 0 and not D.offsets.any() and len(D) == len(X)
    c = engine.Ciphertext.from_host(host[1] if sizes[1] else random_blocks(rng, 5, N), ctx)
    assert np.array_equal((c * c).cancel().getValues(), c.getValues())
    assert (c + c).cancel().n_blocks == 0
    assert np.array_equal(c.cancel().getValues(), c.getValues())


def test_decryptions_are_unchanged_under_every_key(engine, oracle):
    N, D = 1247, 16
    L = words_per_block(N)
    rng = np.random.default_rng(23)
    ctx = engine.Context(N, D)
    keys = [random_key(rng, N, D) for _ in range(4)]
    masks = [oracle.key_mask(N, s) for s in keys]
    host = []
    for t in _sizes("mixed", rng, 150, L):
        t = int(t)
        vals = random_blocks(rng, t, N).reshape(-1, L)
        for v in vals:                             # many values satisfied by one of the keys, some by several
            for m in masks:
                if rng.random() < 0.3:
                    v |= m
        idx = np.repeat(np.arange(t), rng.integers(1, 6, size=t))[:t]
        host.append(vals[idx[rng.permutation(t)]].reshape(-1))
    X = engine.CiphertextArray.from_host(host, ctx)
    G = X.cancel()
    _check_elements(G, _cancelled(host, L))
    for s in keys:
        key = engine.SecretKey(ctx, s)
        bits0, counts0 = key.decrypt_array(X)
        bits1, counts1 = key.decrypt_array(G)
        assert np.array_equal(bits0, bits1)
        diff = counts0.astype(np.int64) - counts1.astype(np.int64)
        assert (diff >= 0).all() and (diff % 2 == 0).all()
        assert diff.any()                      # some satisfied blocks did cancel


def test_empty_elements_no_elements_and_a_complete_cancellation(engine):
    N = 1247
    rng = np.random.default_rng(29)
    ctx = engine.Context(N, 16)
    x = random_blocks(rng, 3, N)
    e = np.empty(0, np.uint64)
    X = engine.CiphertextArray.from_host([e, x, e, np.concatenate([x, x]), e], ctx)
    G = X.cancel()
    assert list(G.offsets) == [0, 0, 3, 3, 3, 3]
    _check_elements(G, [e, x, e, e, e])
    # no elements, and elements without blocks: no launch
    for n in (0, 7):
        E = engine.CiphertextArray(engine.Ciphertext.empty(0, ctx), np.zeros(n + 1, dtype=np.uint64))
        engine.sync()
        c0 = engine.launch_count()
        R = E.cancel()
        assert engine.launch_count() - c0 == 0
        assert len(R) == n and R.storage.n_blocks == 0 and not R.offsets.any()
    # everything cancels: a 0-block result with zero offsets, and no write launch
    Z = engine.CiphertextArray.from_host([np.concatenate([x, x]), np.concatenate([x[:2 * 20], x[:2 * 20]])], ctx)
    engine.sync()
    c0 = engine.launch_count()
    R = Z.cancel()
    assert engine.launch_count() - c0 == 2
    assert R.storage.n_blocks == 0 and list(R.offsets) == [0, 0, 0]
    assert engine.Ciphertext.from_host(np.concatenate([x, x]), ctx).cancel().n_blocks == 0


def test_views_lazy_sums_and_a_producer_on_another_stream(engine, oracle):
    import torch
    N = 4097                                                           # odd L = 65
    L = words_per_block(N)
    rng = np.random.default_rng(31)
    ctx = engine.Context(N, 16)
    sizes = _sizes("mixed", rng, 200, L)
    host = [_with_repeats(rng, int(t), N, "multi") for t in sizes]
    flat = np.concatenate(host)
    t = torch.zeros(flat.size + 1, dtype=torch.int64, device="cuda")
    t[1:] = torch.from_numpy(flat.view(np.int64)).cuda()
    torch.cuda.synchronize()
    view = engine.Ciphertext.view(t.data_ptr() + 8, flat.size // L, ctx, keepalive=t)      # 8 bytes off 16-byte alignment
    _check_elements(engine.CiphertextArray(view, _offsets(sizes)).cancel(), _cancelled(host, L))
    # an even L on a misaligned view (8-byte units)
    N2 = 1247
    L2 = words_per_block(N2)
    ctx2 = engine.Context(N2, 16)
    sizes2 = _sizes("rand", rng, 300, L2)
    host2 = [_with_repeats(rng, int(s), N2, "pairs") for s in sizes2]
    flat2 = np.concatenate(host2)
    t2 = torch.zeros(flat2.size + 1, dtype=torch.int64, device="cuda")
    t2[1:] = torch.from_numpy(flat2.view(np.int64)).cuda()
    torch.cuda.synchronize()
    view2 = engine.Ciphertext.view(t2.data_ptr() + 8, flat2.size // L2, ctx2, keepalive=t2)
    _check_elements(engine.CiphertextArray(view2, _offsets(sizes2)).cancel(), _cancelled(host2, L2))

    # a lazy sum (two segments of >= 1 MiB) as the storage of an array, and as a Ciphertext
    half = 7000
    w1 = _with_repeats(rng, half, N2, "multi")
    w2 = np.concatenate([w1[:3000 * L2], random_blocks(rng, half - 3000, N2)])
    rope = engine.Ciphertext.from_host(w1, ctx2).add_lazy(engine.Ciphertext.from_host(w2, ctx2))
    assert rope.segments == 2
    both = np.concatenate([w1, w2])
    off = _offsets([5000, 0, 4000, 5000])
    R = engine.CiphertextArray(rope, off)
    assert rope.segments == 2                  # still lazy when the call receives it
    _check_elements(R.cancel(), _cancelled([both[int(off[k]) * L2:int(off[k + 1]) * L2] for k in range(4)], L2))
    rope2 = engine.Ciphertext.from_host(w1, ctx2).add_lazy(engine.Ciphertext.from_host(w2, ctx2))
    assert np.array_equal(rope2.cancel().getValues(), _cancelled([both], L2)[0])

    # a producer (csgn_mul of a ciphertext by itself) and the cancellation on a caller's stream, with no
    # synchronisation between them
    wa = random_blocks(rng, 300, N2)
    engine.sync()
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        engine.set_stream(st.cuda_stream)
        try:
            a = engine.Ciphertext.from_host(wa, ctx2)
            P = engine.CiphertextArray(a * a, [0, 300 * 300])
            G = P.cancel()
            words = G.storage.getValues().copy()
            goff = G.offsets.copy()
        finally:
            engine.set_stream(0)
    assert list(goff) == [0, 300]
    assert np.array_equal(words, wa)


def test_argument_errors_allocate_nothing(engine):
    """The C ABI's own checks: ctypes calls straight into csgn_seg_cancel, so no Python check runs first."""
    import torch
    from csgn_b200._native import CsgnError, check
    lib = engine._lib()
    N = 1247
    ctx = engine.Context(N, 16)
    rng = np.random.default_rng(3)
    A = engine.CiphertextArray.from_host([random_blocks(rng, 2, N), random_blocks(rng, 1, N)], ctx)
    Vp = ctypes.c_void_p

    def call(buf, off, n):
        out_off = np.empty(n + 1, dtype=np.uint64)
        o = None if off is None else np.ascontiguousarray(off, dtype=np.uint64)
        check(lib.csgn_seg_cancel(buf, None if o is None else o.ctypes.data_as(Vp), n, out_off.ctypes.data_as(Vp),
                                  ctypes.byref(Vp())))
        pytest.fail("the call succeeded")

    h = A.storage._h.value
    cases = [
        (lambda: call(None, [0, 2, 3], 2), -2, "null argument"),
        (lambda: call(h, None, 2), -2, "null offsets"),
        (lambda: call(h, [1, 2, 3], 2), -2, "offsets[0]"),
        (lambda: call(h, [0, 4, 3], 2), -2, "offsets decrease"),
        (lambda: call(h, [0, 1, 2], 2), -5, "the storage holds 3 blocks"),
    ]
    engine.sync()
    free0 = engine.device_info()["hbm_free"]
    for fn, code, text in cases:
        with pytest.raises(CsgnError) as ei:
            fn()
        assert ei.value.code == code and text in str(ei.value), str(ei.value)
    engine.sync()
    assert engine.device_info()["hbm_free"] == free0
    # an element of more than 2^30 blocks (one-word blocks: 8 GiB)
    big = (1 << 30) + 2
    t = torch.zeros(big, dtype=torch.int64, device="cuda")
    ctx64 = engine.Context(64, 4)
    V = engine.Ciphertext.view(t.data_ptr(), big, ctx64, keepalive=t)
    engine.sync()
    free0 = engine.device_info()["hbm_free"]
    with pytest.raises(CsgnError) as ei:
        call(V._h.value, [0, 1, big], 2)
    assert ei.value.code == -2 and "more than the 2^30" in str(ei.value), str(ei.value)
    engine.sync()
    assert engine.device_info()["hbm_free"] == free0
    del V, t
    torch.cuda.empty_cache()


def test_the_same_launches_for_ten_and_ten_thousand_elements(engine):
    N = 1247
    L = words_per_block(N)
    rng = np.random.default_rng(4)
    ctx = engine.Context(N, 16)
    counts = []
    for n in (10, 10000):
        host = [_with_repeats(rng, int(t), N, "multi") for t in np.maximum(_sizes("rand", rng, n, L), 1)]
        X = engine.CiphertextArray.from_host(host, ctx)
        engine.sync()
        c0 = engine.launch_count()
        G = X.cancel()
        counts.append(engine.launch_count() - c0)
        assert G.offsets[-1] > 0
    assert counts == [3, 3]


def _multiplier(engine, X, Y, gate):
    """Product mod 2^n of the bit arrays X[i], Y[i] (bit i of every lane): schoolbook rows, ripple-carry adds, every
    sum and carry one gate(products, terms).  None stands for an all-zero bit (no blocks)."""
    n = len(X)
    acc = [None] * n
    for j in range(n):
        pp = [None] * j + [gate([(X[i], Y[j])], []) for i in range(n - j)]
        c, out = None, []
        for k in range(n):
            ops = [x for x in (acc[k], pp[k], c) if x is not None]
            out.append(gate([], ops) if ops else None)
            prods = [(ops[p], ops[q]) for p in range(len(ops)) for q in range(p + 1, len(ops))]
            c = gate(prods, []) if prods else None
        acc = out
    return acc


def test_5_bit_multiplier_with_cancelled_gates(engine):
    N, D, lanes, bits = 1247, 16, 1024, 5
    rng = np.random.default_rng(41)
    ctx = engine.Context(N, D)
    key = engine.SecretKey(ctx, random_key(rng, N, D))
    xb, yb = rng.integers(0, 1 << bits, lanes), rng.integers(0, 1 << bits, lanes)
    ones = np.arange(0, lanes, 8)                                      # lanes whose inputs all encrypt 1
    xb[ones] = yb[ones] = (1 << bits) - 1
    plain = np.concatenate([np.concatenate([(v >> i) & 1 for i in range(bits)]) for v in (xb, yb)]).astype(np.uint8)
    allb = key.encrypt_array(plain, seed=77)
    rows = [allb.gather(np.arange(r * lanes, (r + 1) * lanes)) for r in range(2 * bits)]
    SP = engine.CiphertextArray.sum_of_products
    P = _multiplier(engine, rows[:bits], rows[bits:], lambda p, t: SP(p, t, compact=True).cancel())
    got = np.zeros(lanes, dtype=np.int64)
    for i in range(bits):
        got |= key.decrypt_array(P[i])[0].astype(np.int64) << i
    assert np.array_equal(got, (xb * yb) % (1 << bits))
    bound = [1, 2, 4, 10, 26]                  # monomials of odd coefficient of product bit i
    for i in range(bits):
        per_lane = np.diff(P[i].offsets.astype(np.int64))
        assert per_lane.max() <= bound[i], (i, per_lane.max())
        assert (per_lane[ones] == bound[i]).all(), (i, per_lane[ones].min())


def test_cpp_cancel_demo():
    exe = os.path.join(ROOT, "tests", "cpp", "bin", "cancel_demo")
    r = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:]
    assert "cancel_demo: 5-bit multiplier over 1024 lanes with cancelled gates: all checks passed" in r.stdout
