"""Sums of products on ciphertext arrays (csgn_seg_mul_sum, CiphertextArray.sum_of_products / sumOfProducts): element
k = A0_k*B0_k + ... + C0_k + ... in one call, every word of every element bit-exact against the oracle and against the
same gate built from csgn_seg_mul and csgn_seg_concat."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle.pyoracle import random_blocks, random_key, words_per_block

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NS = [64, 191, 1247, 4097, 16383, 33000]          # L = 1, 3, 20, 65, 256, 516
DISTS = ["one", "rand", "mixed"]
SHAPES = [(1, 0), (2, 0), (3, 0), (0, 2), (2, 1), (1, 2)]   # (products, terms)

pytestmark = pytest.mark.gpu


def _elements(rng, sizes, N, mask):
    """Random blocks, about half of them with every key bit set (so that counts and products are not all zero)."""
    L = words_per_block(N)
    out = []
    for t in sizes:
        w = random_blocks(rng, int(t), N).reshape(-1, L)
        w[rng.random(int(t)) < 0.5] |= mask
        out.append(w.reshape(-1))
    return out


def _sizes(dist, rng, n):
    if dist == "one":
        return np.ones(n, dtype=np.int64)
    s = rng.integers(0, 9, size=n)
    s[::7] = 0
    if dist == "mixed":                  # with the threshold lowered to 64 blocks: both sides of it
        s[3::11] = rng.integers(40, 90, size=s[3::11].size)
    return s


def _offsets(sizes):
    off = np.zeros(len(sizes) + 1, dtype=np.uint64)
    off[1:] = np.cumsum(sizes)
    return off


def _gate(oracle, L, products, terms):
    """The oracle's words of every element: products first, then terms, each concatenated in order."""
    n = len(products[0][0]) if products else len(terms[0])
    out = []
    for k in range(n):
        parts = [oracle.mul(a[k], b[k], L) for a, b in products if a[k].size and b[k].size] + \
                [c[k] for c in terms if c[k].size]
        w = np.empty(0, np.uint64)
        for p in parts:
            w = oracle.concat(w, p) if w.size else p.copy()
        out.append(w)
    return out


def _check_elements(arr, want):
    assert len(arr) == len(want)
    assert np.array_equal(arr.offsets, _offsets([w.size // arr.ctx.L for w in want]))
    got = arr.to_host()
    for k, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g, w), "element %d differs" % k


def _same(x, y):
    assert np.array_equal(x.offsets, y.offsets)
    assert np.array_equal(x.storage.getValues(), y.storage.getValues())


def _count(oracle, v, N, s):
    return oracle.count_satisfied(v, N, s) if v.size else 0


@pytest.fixture
def low_threshold(monkeypatch):
    """CSGN_SEG_LARGE_BYTES (honoured with CSGN_TUNING, which tests/conftest.py sets) in blocks of L words."""
    def set_blocks(L, blocks):
        monkeypatch.setenv("CSGN_SEG_LARGE_BYTES", str(8 * L * blocks))
    return set_blocks


def _setup(engine, oracle, N, seed):
    D = 16 if N >= 64 else 4
    rng = np.random.default_rng(seed)
    ctx = engine.Context(N, D)
    s = random_key(rng, N, D)
    return rng, ctx, s, oracle.key_mask(N, s), engine.SecretKey(ctx, s)


@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("dist", DISTS)
def test_sum_of_products_matches_the_oracle(engine, oracle, N, dist, low_threshold):
    L = words_per_block(N)
    rng, ctx, s, mask, key = _setup(engine, oracle, N, N * 11 + DISTS.index(dist))
    n = 40 if L > 100 else 120
    low_threshold(L, 64 if dist == "mixed" else 1 << 40)
    host = [_elements(rng, _sizes(dist, rng, n), N, mask) for _ in range(8)]
    arrs = [engine.CiphertextArray.from_host(h, ctx) for h in host]
    for p, q in SHAPES:
        prods = [(arrs[2 * i], arrs[2 * i + 1]) for i in range(p)]
        terms = arrs[6:6 + q]
        G = engine.CiphertextArray.sum_of_products(prods, terms)
        want = _gate(oracle, L, [(host[2 * i], host[2 * i + 1]) for i in range(p)], host[6:6 + q])
        _check_elements(G, want)
        bits, counts = key.decrypt_array(G)
        wc = np.array([_count(oracle, w, N, s) for w in want], dtype=np.uint64)
        assert np.array_equal(counts, wc), (p, q)
        assert np.array_equal(bits, (wc & 1).astype(np.uint8))


@pytest.mark.parametrize("dist", ["rand", "mixed"])
def test_equivalences_with_the_operator_form(engine, oracle, dist, low_threshold):
    N = 1247
    L = words_per_block(N)
    rng, ctx, s, mask, key = _setup(engine, oracle, N, 31 + DISTS.index(dist))
    low_threshold(L, 64 if dist == "mixed" else 1 << 40)
    A0, B0, A1, B1, C = [engine.CiphertextArray.from_host(_elements(rng, _sizes(dist, rng, 150), N, mask), ctx)
                         for _ in range(5)]
    SP = engine.CiphertextArray.sum_of_products
    _same(SP([(A0, B0)]), A0 * B0)
    _same(SP([], [A0, B0]), A0 + B0)
    _same(SP([(A0, B0), (A1, B1)], [C]), A0 * B0 + A1 * B1 + C)


def test_layouts_views_repeats_lazy_sums_and_large_products(engine, oracle):
    import torch
    N = 1247
    L = words_per_block(N)
    rng, ctx, s, mask, key = _setup(engine, oracle, N, 41)
    sizes = _sizes("rand", rng, 200)
    ea = _elements(rng, sizes, N, mask)
    eb = _elements(rng, sizes[::-1], N, mask)
    flat = np.concatenate(ea)
    t = torch.zeros(flat.size + 1, dtype=torch.int64, device="cuda")
    t[1:] = torch.from_numpy(flat.view(np.int64)).cuda()
    torch.cuda.synchronize()
    view = engine.Ciphertext.view(t.data_ptr() + 8, flat.size // L, ctx, keepalive=t)      # 8 bytes off 16-byte alignment
    A = engine.CiphertextArray(view, _offsets(sizes))
    B = engine.CiphertextArray.from_host(eb, ctx)
    SP = engine.CiphertextArray.sum_of_products
    _check_elements(SP([(A, B)], [B, A]), _gate(oracle, L, [(ea, eb)], [eb, ea]))

    # one buffer any number of times: X*X + X, and X*Y + X*X
    _check_elements(SP([(B, B)], [B]), _gate(oracle, L, [(eb, eb)], [eb]))
    _check_elements(SP([(B, A), (B, B)]), _gate(oracle, L, [(eb, ea), (eb, eb)], []))

    # a lazy sum (two segments of >= 1 MiB) as the storage of an array of one-block elements
    half = 7000
    w1, w2 = _elements(rng, [half], N, mask)[0], _elements(rng, [half], N, mask)[0]
    rope = engine.Ciphertext.from_host(w1, ctx).add_lazy(engine.Ciphertext.from_host(w2, ctx))
    assert rope.segments == 2
    R = engine.CiphertextArray(rope, np.arange(2 * half + 1, dtype=np.uint64))
    blocks = [b.copy() for b in np.concatenate([w1, w2]).reshape(-1, L)]
    Rr = engine.CiphertextArray.from_host(blocks[::-1], ctx)
    assert rope.segments == 2                  # still lazy when the gate receives it
    _check_elements(SP([(R, Rr)], [R]), _gate(oracle, L, [(blocks, blocks[::-1])], [blocks]))

    # products above the default 8 MB threshold next to small ones
    big = [1, 300, 0, 3, 2, 270, 1]
    xa, xb = _elements(rng, big, N, mask), _elements(rng, big[::-1], N, mask)
    X, Y = engine.CiphertextArray.from_host(xa, ctx), engine.CiphertextArray.from_host(xb, ctx)
    G = SP([(X, Y), (Y, X)], [X])
    want = _gate(oracle, L, [(xa, xb), (xb, xa)], [xa])
    _check_elements(G, want)
    _, counts = key.decrypt_array(G)
    assert [int(c) for c in counts] == [_count(oracle, w, N, s) for w in want]


def _pipeline(engine, key, ctx, wa, wb, off):
    """A producer csgn_mul and a consuming gate with no synchronisation between them."""
    P = engine.Ciphertext.from_host(wa, ctx) * engine.Ciphertext.from_host(wb, ctx)
    arr = engine.CiphertextArray(P, off)
    G = engine.CiphertextArray.sum_of_products([(arr, arr.gather(np.arange(len(arr))[::-1]))], [arr])
    bits, counts = key.decrypt_array(G)
    return [w.copy() for w in G.to_host()], counts


def test_producer_on_another_stream(engine, oracle):
    import torch
    N = 1247
    L = words_per_block(N)
    rng, ctx, s, mask, key = _setup(engine, oracle, N, 51)
    wa, wb = _elements(rng, [300], N, mask)[0], _elements(rng, [200], N, mask)[0]
    sizes = _sizes("rand", rng, 300 * 200 // 5)
    sizes[-1] += 300 * 200 - sizes.sum()
    off = _offsets(sizes)
    engine.sync()
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        engine.set_stream(st.cuda_stream)
        try:
            words, counts = _pipeline(engine, key, ctx, wa, wb, off)
        finally:
            engine.set_stream(0)
    prod = oracle.mul(wa, wb, L).reshape(-1, L)
    el = [prod[int(off[k]):int(off[k + 1])].reshape(-1) for k in range(len(off) - 1)]
    want = _gate(oracle, L, [(el, el[::-1])], [el])
    assert all(np.array_equal(a, b) for a, b in zip(words, want))
    assert [int(c) for c in counts] == [_count(oracle, w, N, s) for w in want]


def test_argument_errors_allocate_nothing(engine):
    """The C ABI's own checks: ctypes calls straight into csgn_seg_mul_sum, so no Python check runs first."""
    from csgn_b200._native import CsgnError, check
    lib = engine._lib()
    N = 1247
    ctx, ctx2 = engine.Context(N, 16), engine.Context(64, 4)
    rng = np.random.default_rng(3)
    A = engine.CiphertextArray.from_host([random_blocks(rng, 2, N), random_blocks(rng, 1, N)], ctx)
    Z = engine.CiphertextArray.from_host([random_blocks(rng, 1, 64)] * 2, ctx2)
    huge = engine.Ciphertext.view(A.storage.device_ptr(), 1 << 40, ctx)      # views: validation fails before any read
    big = engine.Ciphertext.view(A.storage.device_ptr(), 1 << 31, ctx)
    Vp = ctypes.c_void_p

    def u64(xs):
        return np.ascontiguousarray(np.asarray(xs, dtype=np.uint64))
    keep = []

    def call(prods, terms, n=2, null_out=False):
        """prods: [((buf, off), (buf, off))], terms: [(buf, off)]; buf a Ciphertext or None, off a list or None"""
        def side(items):
            if items is None:
                return None, None
            hs, os_ = [], []
            for buf, off in items:
                hs.append(None if buf is None else buf._h.value)
                o = None if off is None else u64(off)
                keep.append(o)
                os_.append(None if o is None else o.ctypes.data)
            return (Vp * max(1, len(hs)))(*hs), (Vp * max(1, len(os_)))(*os_)
        la, lo = side(None if prods is None else [x for x, _ in prods])
        ra, ro = side(None if prods is None else [y for _, y in prods])
        ca, co = side(terms)
        out_off = np.empty(n + 1, dtype=np.uint64)
        h = Vp()
        check(lib.csgn_seg_mul_sum(la, lo, ra, ro, len(prods or []), ca, co, len(terms or []), n,
                                   None if null_out else out_off.ctypes.data_as(Vp), ctypes.byref(h)))
        pytest.fail("the call succeeded")

    a = (A.storage, [0, 2, 3])
    cases = [
        (lambda: call([(a, (Z.storage, [0, 1, 2]))], []), -5, "words per block"),
        (lambda: call([(a, a)], [(Z.storage, [0, 1, 2])]), -5, "words per block"),
        (lambda: call([(a, (A.storage, [1, 2, 3]))], []), -2, "offsets[0]"),
        (lambda: call([(a, a)], [(A.storage, [0, 3, 2])]), -2, "offsets decrease"),
        (lambda: call([(a, (A.storage, [0, 1, 2]))], []), -5, "storage holds"),
        (lambda: call([], [a, (A.storage, [0, 1, 1])]), -5, "storage holds"),
        (lambda: call([(a, (A.storage, None))], []), -2, "null offsets"),
        (lambda: call([], []), -2, "no products and no terms"),
        (lambda: call(None, None), -2, "no products and no terms"),
        (lambda: call([((None, [0, 2, 3]), a)], []), -2, "null left operand 0"),
        (lambda: call([(a, a)], [a, (None, [0, 1, 2])]), -2, "null term 1"),
        (lambda: check(lib.csgn_seg_mul_sum(None, None, None, None, 1, None, None, 0, 2,
                                            np.empty(3, np.uint64).ctypes.data_as(Vp), ctypes.byref(Vp()))), -2,
         "null product arrays"),
        (lambda: check(lib.csgn_seg_mul_sum(None, None, None, None, 0, None, None, 1, 2,
                                            np.empty(3, np.uint64).ctypes.data_as(Vp), ctypes.byref(Vp()))), -2,
         "null term arrays"),
        (lambda: call([(a, a)], [], null_out=True), -2, "null argument"),
        (lambda: call([((huge, [0, 1 << 40]), (huge, [0, 1 << 40]))], [], n=1), -2, "overflows"),
        (lambda: call([((big, [0, 1 << 31]), (big, [0, 1 << 31]))], [], n=1), -2, "output block count overflows"),
        (lambda: call([((big, [0, 1 << 31]), (big, [0, 1 << 31]))] * 4, [], n=1), -2, "output block count overflows"),
    ]
    engine.sync()
    free0 = engine.device_info()["hbm_free"]
    for fn, code, text in cases:
        with pytest.raises(CsgnError) as ei:
            fn()
        assert ei.value.code == code and text in str(ei.value), str(ei.value)
    # the Python method refuses mismatched element counts and contexts before the call
    SP = engine.CiphertextArray.sum_of_products
    for bad in (lambda: SP([(A, A)], [engine.CiphertextArray(A.storage, [0, 3])]), lambda: SP([(A, A)], [Z]),
                lambda: SP([], [])):
        with pytest.raises(ValueError):
            bad()
    engine.sync()
    assert engine.device_info()["hbm_free"] == free0


def test_two_launches_for_ten_thousand_elements(engine):
    N, n = 1247, 10000
    rng = np.random.default_rng(4)
    ctx = engine.Context(N, 16)
    key = engine.SecretKey(ctx, random_key(rng, N, 16))
    X, Y, C = [key.encrypt_array(rng.integers(0, 2, n), seed=i) for i in (1, 2, 3)]
    T = X + Y
    engine.sync()
    c0 = engine.launch_count()
    G = engine.CiphertextArray.sum_of_products([(X, Y), (T, C)], [C])
    assert engine.launch_count() - c0 <= 2
    assert len(G) == n


def _bit_rows(key, xb, yb, lanes, bits):
    plain = np.concatenate([np.concatenate([(v >> i) & 1 for i in range(bits)]) for v in (xb, yb)]).astype(np.uint8)
    allb = key.encrypt_array(plain, seed=99)
    return [allb.gather(np.arange(r * lanes, (r + 1) * lanes)) for r in range(2 * bits)]


def test_simd_adder_with_one_call_per_carry(engine):
    N, D, lanes = 1247, 16, 1024
    rng = np.random.default_rng(8)
    ctx = engine.Context(N, D)
    key = engine.SecretKey(ctx, random_key(rng, N, D))
    xb, yb = rng.integers(0, 256, lanes), rng.integers(0, 256, lanes)
    rows = _bit_rows(key, xb, yb, lanes, 8)
    SP = engine.CiphertextArray.sum_of_products
    X, Y = rows[0], rows[8]
    S, C, Cops = [X + Y], SP([(X, Y)]), X * Y
    _same(C, Cops)
    for i in range(1, 8):
        X, Y = rows[i], rows[8 + i]
        T = X + Y
        S.append(T + C)
        C, Cops = SP([(X, Y), (T, C)]), X * Y + T * Cops
        _same(C, Cops)
    got = np.zeros(lanes, dtype=np.int64)
    for i in range(8):
        got |= key.decrypt_array(S[i])[0].astype(np.int64) << i
    assert np.array_equal(got, (xb + yb) % 256)
    assert np.array_equal(key.decrypt_array(C)[0], (xb + yb) >> 8)


def test_majority_and_multiplexer(engine):
    N, D, lanes = 1247, 16, 1024
    rng = np.random.default_rng(9)
    ctx = engine.Context(N, D)
    key = engine.SecretKey(ctx, random_key(rng, N, D))
    x, y, z = (rng.integers(0, 2, lanes) for _ in range(3))
    X, Y, Z = (key.encrypt_array(v, seed=10 + i) for i, v in enumerate((x, y, z)))
    SP = engine.CiphertextArray.sum_of_products
    maj = SP([(X, Y), (X, Z), (Y, Z)])
    assert np.array_equal(key.decrypt_array(maj)[0], ((x + y + z) >= 2).astype(np.uint8))
    s, a, b = x, y, z
    mux = SP([(X, Y), (X, Z)], [Z])                                   # s*a + s*b + b = s ? a : b
    assert np.array_equal(key.decrypt_array(mux)[0], np.where(s == 1, a, b).astype(np.uint8))
    orr = SP([(X, Y)], [X, Y])                                        # x*y + x + y = x OR y
    assert np.array_equal(key.decrypt_array(orr)[0], (x | y).astype(np.uint8))


def test_cpp_gates_demo():
    exe = os.path.join(ROOT, "tests", "cpp", "bin", "gates_demo")
    r = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:]
    assert "gates_demo: 8-bit adder over 1024 lanes with one sumOfProducts call per carry: all checks passed" in r.stdout
