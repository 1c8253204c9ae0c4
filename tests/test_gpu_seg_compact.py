"""Compacting gates on ciphertext arrays (csgn_seg_mul_sum_compact; CiphertextArray.sum_of_products(compact=True),
.compact(), Ciphertext.compact(); CiphertextArray::compactSumOfProducts in C++): element k is the stable subsequence
of the uncompacted gate's element k made of the blocks with at least min_bits set bits.  Checked word for word against
the oracle's gate filtered by popcount in numpy, and, with min_bits = D, the satisfied-block count of every element
against the uncompacted result."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle.pyoracle import random_blocks, random_key, words_per_block

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NS = [64, 191, 1247, 4097, 16383, 33000]          # L = 1, 3, 20, 65, 256, 516
DISTS = ["one", "rand", "mixed"]
SHAPES = [(2, 0), (0, 1), (2, 1)]                 # (products, terms): products only, compaction on its own, both

pytestmark = pytest.mark.gpu


def _popcounts(w, L):
    """set bits of every block of the words w (pad bits included)"""
    return np.unpackbits(np.ascontiguousarray(w).reshape(-1, L).view(np.uint8), axis=1).sum(axis=1)


def _filtered(elements, L, min_bits):
    """the numpy restatement: every element without its blocks of fewer than min_bits set bits, in order"""
    return [w.reshape(-1, L)[_popcounts(w, L) >= min_bits].reshape(-1) for w in elements]


def _elements(rng, sizes, N, D, mask):
    """Blocks of every density: about D set bits (on both sides of it), a few times D, or half of N; a third carry
    every key bit (so that counts are not all zero)."""
    L = words_per_block(N)
    k_mid = max(0, int(np.log2(N / D)))           # AND of k random blocks: about N / 2^(k+1) set bits
    out = []
    for t in sizes:
        t = int(t)
        w = random_blocks(rng, t, N).reshape(-1, L)
        for i, k in enumerate(rng.choice([0, k_mid - 2, k_mid - 1, k_mid, k_mid + 1], size=t)):
            for _ in range(max(0, int(k))):
                w[i] &= random_blocks(rng, 1, N)
        w[rng.random(t) < 0.3] |= mask
        out.append(w.reshape(-1))
    return out


def _sizes(dist, rng, n):
    if dist == "one":
        return np.ones(n, dtype=np.int64)
    s = rng.integers(0, 9, size=n)
    s[::7] = 0
    if dist == "mixed":                  # large elements, which the uncompacted gate sends to other kernels
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


def _count(oracle, v, N, s):
    return oracle.count_satisfied(v, N, s) if v.size else 0


def _setup(engine, oracle, N, seed):
    D = 16 if N >= 64 else 4
    rng = np.random.default_rng(seed)
    ctx = engine.Context(N, D)
    s = random_key(rng, N, D)
    return rng, ctx, s, oracle.key_mask(N, s), engine.SecretKey(ctx, s)


def _abi(engine, products, terms, min_bits):
    """csgn_seg_mul_sum_compact straight through ctypes with any min_bits"""
    from csgn_b200._native import check
    Vp = ctypes.c_void_p
    arrays = [x for pr in products for x in pr] + list(terms)
    n, ctx = len(arrays[0]), arrays[0].ctx
    h = lambda xs: engine.handle_array([x.storage for x in xs]) if xs else None                 # noqa: E731
    o = lambda xs: (Vp * len(xs))(*[x.offsets.ctypes.data for x in xs]) if xs else None        # noqa: E731
    left, right = [x for x, _ in products], [y for _, y in products]
    out_off = np.empty(n + 1, dtype=np.uint64)
    out = Vp()
    check(engine._lib().csgn_seg_mul_sum_compact(h(left), o(left), h(right), o(right), len(products), h(terms),
                                                 o(terms), len(terms), n, min_bits, out_off.ctypes.data_as(Vp),
                                                 ctypes.byref(out)))
    return engine.CiphertextArray(engine.Ciphertext(out, ctx), out_off)


@pytest.fixture
def low_threshold(monkeypatch):
    """CSGN_SEG_LARGE_BYTES (honoured with CSGN_TUNING, which tests/conftest.py sets) in blocks of L words."""
    def set_blocks(L, blocks):
        monkeypatch.setenv("CSGN_SEG_LARGE_BYTES", str(8 * L * blocks))
    return set_blocks


@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("dist", DISTS)
def test_compacted_gate_matches_the_filtered_oracle(engine, oracle, N, dist, low_threshold):
    L = words_per_block(N)
    rng, ctx, s, mask, key = _setup(engine, oracle, N, N * 13 + DISTS.index(dist))
    D = ctx.D
    n = 40 if L > 100 else 120
    low_threshold(L, 64 if dist == "mixed" else 1 << 40)
    host = [_elements(rng, _sizes(dist, rng, n), N, D, mask) for _ in range(6)]
    arrs = [engine.CiphertextArray.from_host(h, ctx) for h in host]
    SP = engine.CiphertextArray.sum_of_products
    for p, q in SHAPES:
        prods = [(arrs[2 * i], arrs[2 * i + 1]) for i in range(p)]
        terms = arrs[4:4 + q]
        full = _gate(oracle, L, [(host[2 * i], host[2 * i + 1]) for i in range(p)], host[4:4 + q])
        want = _filtered(full, L, D)
        G = SP(prods, terms, compact=True) if p else terms[0].compact()
        _check_elements(G, want)
        assert sum(w.size for w in want) < sum(w.size for w in full), (p, q)     # the filter drops blocks here
        # the satisfied-block count of every element is that of the uncompacted gate
        _, counts = key.decrypt_array(G)
        _, full_counts = key.decrypt_array(SP(prods, terms))
        assert np.array_equal(counts, full_counts), (p, q)
        assert [int(c) for c in counts] == [_count(oracle, w, N, s) for w in full], (p, q)


@pytest.mark.parametrize("N", [64, 1247])
def test_min_bits_through_the_c_abi(engine, oracle, N):
    L = words_per_block(N)
    rng, ctx, s, mask, key = _setup(engine, oracle, N, 61 + N)
    sizes = _sizes("rand", rng, 150)
    ea, eb, ec = (_elements(rng, sizes, N, ctx.D, mask) for _ in range(3))
    ec[5] = np.full(3 * L, ~np.uint64(0), dtype=np.uint64)             # all ones: 64 L set bits, pad bits included
    A, B, C = (engine.CiphertextArray.from_host(e, ctx) for e in (ea, eb, ec))
    full = _gate(oracle, L, [(ea, eb)], [ec])
    for min_bits in (1, ctx.D, 64 * L):
        want = _filtered(full, L, min_bits)
        G = _abi(engine, [(A, B)], [C], min_bits)
        _check_elements(G, want)
    assert G.offsets[-1] == 3                                          # only the three all-ones blocks are left


def test_blocks_on_either_side_of_the_threshold(engine, oracle):
    N, D = 1247, 16
    L = words_per_block(N)
    rng, ctx, s, mask, key = _setup(engine, oracle, N, 71)
    blocks, keep = [], []
    for bits in (D - 1, D, D + 1, 0, D, D - 1, 1, 64 * L - 33):
        pos = rng.choice(N, size=min(bits, N), replace=False)
        w = np.zeros(L, dtype=np.uint64)
        for p in pos:
            w[p // 64] |= np.uint64(1) << np.uint64(p % 64)
        blocks.append(w)
        keep.append(min(bits, N) >= D)
    elems = [np.concatenate(blocks[:3]), np.concatenate(blocks[3:4]), np.concatenate(blocks[4:])]
    X = engine.CiphertextArray.from_host(elems, ctx)
    want = [np.concatenate([b for b, k in zip(blocks[i:j], keep[i:j]) if k] or [np.empty(0, np.uint64)])
            for i, j in ((0, 3), (3, 4), (4, 8))]
    _check_elements(X.compact(), want)
    # the same blocks as a product with an all-ones block (pad bits zero), and as a single Ciphertext
    pad = np.full(L, ~np.uint64(0), dtype=np.uint64)
    if N % 64:
        pad[-1] = (np.uint64(1) << np.uint64(N % 64)) - np.uint64(1)
    P = engine.CiphertextArray.from_host([pad] * 3, ctx)
    _check_elements(engine.CiphertextArray.sum_of_products([(P, X)], compact=True), want)
    c = engine.Ciphertext.from_host(np.concatenate(blocks), ctx)
    assert np.array_equal(c.compact().getValues(), np.concatenate(want))
    assert c.n_blocks == len(blocks)                                   # the input is unchanged


def test_layouts_views_repeats_lazy_sums_streams_and_large_products(engine, oracle):
    import torch
    N = 4097                                                           # odd L = 65
    L = words_per_block(N)
    rng, ctx, s, mask, key = _setup(engine, oracle, N, 81)
    D = ctx.D
    sizes = _sizes("rand", rng, 200)
    ea = _elements(rng, sizes, N, D, mask)
    eb = _elements(rng, sizes[::-1], N, D, mask)
    flat = np.concatenate(ea)
    t = torch.zeros(flat.size + 1, dtype=torch.int64, device="cuda")
    t[1:] = torch.from_numpy(flat.view(np.int64)).cuda()
    torch.cuda.synchronize()
    view = engine.Ciphertext.view(t.data_ptr() + 8, flat.size // L, ctx, keepalive=t)      # 8 bytes off 16-byte alignment
    A = engine.CiphertextArray(view, _offsets(sizes))
    B = engine.CiphertextArray.from_host(eb, ctx)
    SP = engine.CiphertextArray.sum_of_products
    _check_elements(SP([(A, B)], [B, A], compact=True), _filtered(_gate(oracle, L, [(ea, eb)], [eb, ea]), L, D))
    # one buffer any number of times
    _check_elements(SP([(B, B)], [B], compact=True), _filtered(_gate(oracle, L, [(eb, eb)], [eb]), L, D))
    _check_elements(SP([(B, A), (B, B)], compact=True), _filtered(_gate(oracle, L, [(eb, ea), (eb, eb)], []), L, D))

    # a lazy sum (two segments of >= 1 MiB) as the storage of an array of one-block elements, and as a Ciphertext
    N2 = 1247
    L2 = words_per_block(N2)
    ctx2 = engine.Context(N2, 16)
    mask2 = oracle.key_mask(N2, random_key(rng, N2, 16))
    half = 7000
    w1, w2 = (_elements(rng, [half], N2, 16, mask2)[0] for _ in range(2))
    rope = engine.Ciphertext.from_host(w1, ctx2).add_lazy(engine.Ciphertext.from_host(w2, ctx2))
    assert rope.segments == 2
    R = engine.CiphertextArray(rope, np.arange(2 * half + 1, dtype=np.uint64))
    blocks = [b.copy() for b in np.concatenate([w1, w2]).reshape(-1, L2)]
    Rr = engine.CiphertextArray.from_host(blocks[::-1], ctx2)
    assert rope.segments == 2                  # still lazy when the gate receives it
    _check_elements(SP([(R, Rr)], [R], compact=True), _filtered(_gate(oracle, L2, [(blocks, blocks[::-1])], [blocks]),
                                                                L2, 16))
    rope2 = engine.Ciphertext.from_host(w1, ctx2).add_lazy(engine.Ciphertext.from_host(w2, ctx2))
    assert np.array_equal(rope2.compact().getValues(), _filtered([np.concatenate([w1, w2])], L2, 16)[0])

    # products above 8 MB (which the uncompacted gate writes with launch_mul) next to small ones
    big = [1, 300, 0, 3, 2, 270, 1]
    xa, xb = _elements(rng, big, N2, 16, mask2), _elements(rng, big[::-1], N2, 16, mask2)
    X, Y = engine.CiphertextArray.from_host(xa, ctx2), engine.CiphertextArray.from_host(xb, ctx2)
    assert 300 * 270 * L2 * 8 > 8 << 20
    G = SP([(X, Y), (Y, X)], [X], compact=True)
    _check_elements(G, _filtered(_gate(oracle, L2, [(xa, xb), (xb, xa)], [xa]), L2, 16))

    # a producer csgn_mul and a consuming compacting gate on a caller's stream, with no synchronisation between them
    wa, wb = _elements(rng, [300], N2, 16, mask2)[0], _elements(rng, [200], N2, 16, mask2)[0]
    psizes = _sizes("rand", rng, 300 * 200 // 5)
    psizes[-1] += 300 * 200 - psizes.sum()
    off = _offsets(psizes)
    engine.sync()
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        engine.set_stream(st.cuda_stream)
        try:
            P = engine.Ciphertext.from_host(wa, ctx2) * engine.Ciphertext.from_host(wb, ctx2)
            arr = engine.CiphertextArray(P, off)
            G = SP([(arr, arr.gather(np.arange(len(arr))[::-1]))], [arr], compact=True)
            words = [w.copy() for w in G.to_host()]
            goff = G.offsets.copy()
        finally:
            engine.set_stream(0)
    prod = oracle.mul(wa, wb, L2).reshape(-1, L2)
    el = [prod[int(off[k]):int(off[k + 1])].reshape(-1) for k in range(len(off) - 1)]
    want = _filtered(_gate(oracle, L2, [(el, el[::-1])], [el]), L2, 16)
    assert np.array_equal(goff, _offsets([w.size // L2 for w in want]))
    assert all(np.array_equal(a, b) for a, b in zip(words, want))


def test_dead_elements_and_an_empty_result(engine, oracle):
    N = 1247
    L = words_per_block(N)
    rng, ctx, s, mask, key = _setup(engine, oracle, N, 91)
    sparse = random_blocks(rng, 1, N)
    for _ in range(8):
        sparse &= random_blocks(rng, 1, N)                             # about 2 set bits
    dense = random_blocks(rng, 1, N) | mask
    A = engine.CiphertextArray.from_host([sparse, np.concatenate([dense, sparse]), sparse, np.empty(0, np.uint64),
                                          np.concatenate([sparse, dense])], ctx)
    G = A.compact()
    assert list(G.offsets) == [0, 0, 1, 1, 1, 2]
    _check_elements(G, [np.empty(0, np.uint64), dense, np.empty(0, np.uint64), np.empty(0, np.uint64), dense])
    bits, counts = key.decrypt_array(G)
    assert list(counts) == [0, 1, 0, 0, 1] and list(bits) == [0, 1, 0, 0, 1]
    # nothing survives: a 0-block result with all-zero offsets
    Z = engine.CiphertextArray.from_host([sparse] * 4, ctx)
    E = engine.CiphertextArray.sum_of_products([(Z, Z)], [Z], compact=True)
    assert E.storage.n_blocks == 0 and list(E.offsets) == [0] * 5
    bits, counts = key.decrypt_array(E)
    assert list(counts) == [0] * 4
    assert engine.Ciphertext.from_host(sparse, ctx).compact().n_blocks == 0


def test_argument_errors_allocate_nothing(engine):
    """The C ABI's own checks: ctypes calls straight into csgn_seg_mul_sum_compact, so no Python check runs first."""
    from csgn_b200._native import CsgnError, check
    lib = engine._lib()
    N = 1247
    L = words_per_block(N)
    ctx, ctx2 = engine.Context(N, 16), engine.Context(64, 4)
    rng = np.random.default_rng(3)
    A = engine.CiphertextArray.from_host([random_blocks(rng, 2, N), random_blocks(rng, 1, N)], ctx)
    Z = engine.CiphertextArray.from_host([random_blocks(rng, 1, 64)] * 2, ctx2)
    Vp = ctypes.c_void_p
    keep = []

    def call(prods, terms, min_bits=16, n=2):
        def side(items):
            hs = [x.storage._h.value for x in items]
            os_ = [np.ascontiguousarray(o, dtype=np.uint64) for o in [x.offsets for x in items]]
            keep.extend(os_)
            return (Vp * max(1, len(hs)))(*hs), (Vp * max(1, len(os_)))(*[o.ctypes.data for o in os_])
        la, lo = side([x for x, _ in prods])
        ra, ro = side([y for _, y in prods])
        ca, co = side(terms)
        out_off = np.empty(n + 1, dtype=np.uint64)
        check(lib.csgn_seg_mul_sum_compact(la, lo, ra, ro, len(prods), ca, co, len(terms), n, min_bits,
                                           out_off.ctypes.data_as(Vp), ctypes.byref(Vp())))
        pytest.fail("the call succeeded")

    bad_off = engine.CiphertextArray(A.storage, [0, 4, 3])
    cases = [
        (lambda: call([(A, A)], [], min_bits=0), -2, "min_bits = 0"),
        (lambda: call([(A, A)], [], min_bits=64 * L + 1), -2, "min_bits = %d" % (64 * L + 1)),
        (lambda: call([], [A], min_bits=1 << 31), -2, "min_bits"),
        (lambda: call([], [], min_bits=16), -2, "no products and no terms"),
        (lambda: call([(A, Z)], [], min_bits=16), -5, "words per block"),
        (lambda: call([(A, A)], [bad_off], min_bits=16), -2, "offsets decrease"),
    ]
    engine.sync()
    free0 = engine.device_info()["hbm_free"]
    for fn, code, text in cases:
        with pytest.raises(CsgnError) as ei:
            fn()
        assert ei.value.code == code and text in str(ei.value), str(ei.value)
    SP = engine.CiphertextArray.sum_of_products
    for bad in (lambda: SP([(A, A)], [engine.CiphertextArray(A.storage, [0, 3])], compact=True),
                lambda: SP([(A, A)], [Z], compact=True), lambda: SP([], [], compact=True)):
        with pytest.raises(ValueError):
            bad()
    engine.sync()
    assert engine.device_info()["hbm_free"] == free0


def test_two_launches_for_ten_thousand_elements_and_none_for_empty_ones(engine):
    N, n = 1247, 10000
    rng = np.random.default_rng(4)
    ctx = engine.Context(N, 16)
    key = engine.SecretKey(ctx, random_key(rng, N, 16))
    X, Y, C = [key.encrypt_array(rng.integers(0, 2, n), seed=i) for i in (1, 2, 3)]
    T = X + Y
    engine.sync()
    c0 = engine.launch_count()
    G = engine.CiphertextArray.sum_of_products([(X, Y), (T, C)], [C], compact=True)
    assert engine.launch_count() - c0 == 2
    assert len(G) == n
    E = engine.CiphertextArray(engine.Ciphertext.empty(0, ctx), np.zeros(n + 1, dtype=np.uint64))
    engine.sync()
    c0 = engine.launch_count()
    R = engine.CiphertextArray.sum_of_products([(E, E)], [E], compact=True)
    assert engine.launch_count() - c0 == 0
    assert R.storage.n_blocks == 0 and not R.offsets.any() and len(R) == n


def test_32_bit_simd_adder_compacting_every_carry(engine):
    N, D, lanes, bits = 1247, 16, 1024, 32
    rng = np.random.default_rng(12)
    ctx = engine.Context(N, D)
    key = engine.SecretKey(ctx, random_key(rng, N, D))
    xb, yb = rng.integers(0, 1 << bits, lanes), rng.integers(0, 1 << bits, lanes)
    plain = np.concatenate([np.concatenate([(v >> i) & 1 for i in range(bits)]) for v in (xb, yb)]).astype(np.uint8)
    allb = key.encrypt_array(plain, seed=123)
    rows = [allb.gather(np.arange(r * lanes, (r + 1) * lanes)) for r in range(2 * bits)]
    SP = engine.CiphertextArray.sum_of_products
    X, Y = rows[0], rows[bits]
    S, C = [X + Y], SP([(X, Y)], compact=True)
    held = [int(C.offsets[-1])]
    for i in range(1, bits):
        X, Y = rows[i], rows[bits + i]
        T = X + Y
        S.append(T + C)
        C = SP([(X, Y), (T, C)], compact=True)
        held.append(int(C.offsets[-1]))
    assert max(held) < 512 * lanes, held                               # uncompacted: 2^(i+1) - 1 blocks per lane
    got = np.zeros(lanes, dtype=np.int64)
    for i in range(bits):
        got |= key.decrypt_array(S[i])[0].astype(np.int64) << i
    assert np.array_equal(got, (xb + yb) % (1 << bits))
    assert np.array_equal(key.decrypt_array(C)[0], (xb + yb) >> bits)


def test_cpp_compact_demo():
    exe = os.path.join(ROOT, "tests", "cpp", "bin", "compact_demo")
    r = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:]
    assert "compact_demo: 32-bit adder over 1024 lanes with compactSumOfProducts carries: all checks passed" in r.stdout
