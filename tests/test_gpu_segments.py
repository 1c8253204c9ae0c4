"""Ciphertext arrays (include/csgn.h, "ciphertext arrays"; csgn_b200/csrc/segments.cu, capi_seg.cu): every element of
every result, bit-exact against the oracle applied element by element."""
import os
import subprocess

import numpy as np
import pytest

from oracle.pyoracle import random_blocks, random_key, words_per_block

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NS = [64, 191, 1247, 4097, 16383, 33000]          # L = 1, 3, 20, 65, 256, 516
DISTS = ["one", "rand", "mixed"]

pytestmark = pytest.mark.gpu


def _elements(rng, sizes, N, mask):
    """Random blocks, about half of them with every key bit set (so that counts and products are not all zero)."""
    L = words_per_block(N)
    out = []
    for t in sizes:
        w = random_blocks(rng, int(t), N).reshape(-1, L)
        sat = rng.random(int(t)) < 0.5
        w[sat] |= mask
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


def _check_elements(arr, want):
    assert len(arr) == len(want)
    got = arr.to_host()
    for k, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g, w), "element %d differs" % k


def _count(oracle, v, N, s):
    return oracle.count_satisfied(v, N, s) if v.size else 0


@pytest.fixture
def low_threshold(monkeypatch):
    monkeypatch.setenv("CSGN_SEG_LARGE_BYTES", "0")

    def set_blocks(L, blocks):
        monkeypatch.setenv("CSGN_SEG_LARGE_BYTES", str(8 * L * blocks))
    return set_blocks


@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("dist", DISTS)
def test_array_operations_match_the_oracle(engine, oracle, N, dist, low_threshold):
    L = words_per_block(N)
    D = 16 if N >= 64 else 4
    rng = np.random.default_rng(N * 7 + DISTS.index(dist))
    n = 60 if L > 100 else 150
    if dist == "mixed":
        low_threshold(L, 64)
    else:
        low_threshold(L, 1 << 40)
    ctx = engine.Context(N, D)
    s = random_key(rng, N, D)
    mask = oracle.key_mask(N, s)
    key = engine.SecretKey(ctx, s)
    ea = _elements(rng, _sizes(dist, rng, n), N, mask)
    eb = _elements(rng, _sizes(dist, rng, n), N, mask)
    A, B = engine.CiphertextArray.from_host(ea, ctx), engine.CiphertextArray.from_host(eb, ctx)

    P = A * B
    want_p = [oracle.mul(a, b, L) if a.size and b.size else np.empty(0, np.uint64) for a, b in zip(ea, eb)]
    assert np.array_equal(P.offsets, _offsets([w.size // L for w in want_p]))
    _check_elements(P, want_p)

    S = A + B
    _check_elements(S, [oracle.concat(a, b) for a, b in zip(ea, eb)])

    for idx in (rng.integers(0, n, size=n + 9), np.arange(n)[::-1], np.zeros(0, dtype=np.int64)):
        G = A.gather(idx)
        _check_elements(G, [ea[int(i)] for i in idx])

    parts = [engine.Ciphertext.from_host(e, ctx) for e in ea if e.size]
    K = engine.CiphertextArray.pack(parts)
    _check_elements(K, [e for e in ea if e.size])

    for arr, want in ((A, ea), (P, want_p)):
        bits, counts = key.decrypt_array(arr)
        wc = np.array([_count(oracle, w, N, s) for w in want], dtype=np.uint64)
        assert np.array_equal(counts, wc)
        assert np.array_equal(bits, (wc & 1).astype(np.uint8))


def test_large_elements_at_the_default_threshold(engine, oracle):
    """Products above the built-in threshold (8 MB) run on the single-ciphertext kernels, next to small ones."""
    N, D = 1247, 16
    L = words_per_block(N)
    rng = np.random.default_rng(5)
    ctx = engine.Context(N, D)
    s = random_key(rng, N, D)
    key = engine.SecretKey(ctx, s)
    sizes = [1, 300, 0, 3, 2, 270, 1]
    ea = _elements(rng, sizes, N, oracle.key_mask(N, s))
    eb = _elements(rng, sizes[::-1], N, oracle.key_mask(N, s))
    A, B = engine.CiphertextArray.from_host(ea, ctx), engine.CiphertextArray.from_host(eb, ctx)
    P = A * B
    want = [oracle.mul(a, b, L) if a.size and b.size else np.empty(0, np.uint64) for a, b in zip(ea, eb)]
    _check_elements(P, want)
    _, counts = key.decrypt_array(P)
    assert [int(c) for c in counts] == [_count(oracle, w, N, s) for w in want]


def test_misaligned_storage_and_lazy_sum(engine, oracle):
    import torch
    N, D = 1247, 16
    L = words_per_block(N)
    rng = np.random.default_rng(11)
    ctx = engine.Context(N, D)
    s = random_key(rng, N, D)
    key = engine.SecretKey(ctx, s)
    mask = oracle.key_mask(N, s)
    sizes = _sizes("rand", rng, 200)
    ea = _elements(rng, sizes, N, mask)
    flat = np.concatenate(ea)
    t = torch.zeros(flat.size + 1, dtype=torch.int64, device="cuda")
    t[1:] = torch.from_numpy(flat.view(np.int64)).cuda()
    torch.cuda.synchronize()
    view = engine.Ciphertext.view(t.data_ptr() + 8, flat.size // L, ctx, keepalive=t)      # 8 bytes off 16-byte alignment
    A = engine.CiphertextArray(view, _offsets(sizes))
    B = engine.CiphertextArray.from_host(ea[::-1], ctx)
    _check_elements(A * B, [oracle.mul(a, b, L) if a.size and b.size else np.empty(0, np.uint64)
                            for a, b in zip(ea, ea[::-1])])
    _check_elements(A + B, [oracle.concat(a, b) for a, b in zip(ea, ea[::-1])])
    _check_elements(A.gather([5, 5, 0]), [ea[5], ea[5], ea[0]])
    _, counts = key.decrypt_array(A)
    assert [int(c) for c in counts] == [_count(oracle, w, N, s) for w in ea]

    # a lazy sum (two segments of >= 1 MiB) as the storage of an array of one-block elements
    half = 7000
    w1, w2 = _elements(rng, [half], N, mask)[0], _elements(rng, [half], N, mask)[0]
    rope = engine.Ciphertext.from_host(w1, ctx).add_lazy(engine.Ciphertext.from_host(w2, ctx))
    assert rope.segments == 2
    R = engine.CiphertextArray(rope, np.arange(2 * half + 1, dtype=np.uint64))
    blocks = np.concatenate([w1, w2]).reshape(-1, L)
    _, counts = key.decrypt_array(R)
    assert [int(c) for c in counts] == [_count(oracle, b, N, s) for b in blocks]
    idx = np.arange(0, 2 * half, 97)
    _check_elements(R.gather(idx) * R.gather(idx[::-1]), [oracle.mul(blocks[i], blocks[j], L) for i, j in zip(idx, idx[::-1])])


def test_argument_errors_allocate_nothing(engine):
    from csgn_b200._native import CsgnError
    N = 1247
    ctx, ctx2 = engine.Context(N, 16), engine.Context(64, 4)
    rng = np.random.default_rng(3)
    A = engine.CiphertextArray.from_host([random_blocks(rng, 2, N), random_blocks(rng, 1, N)], ctx)
    Z = engine.CiphertextArray.from_host([random_blocks(rng, 1, 64)] * 2, ctx2)
    key = engine.SecretKey(ctx, random_key(rng, N, 16))
    engine.sync()
    free0 = engine.device_info()["hbm_free"]
    cases = [
        (lambda: engine.CiphertextArray(A.storage, [1, 2, 3]) * A, -2, "offsets[0]"),
        (lambda: engine.CiphertextArray(A.storage, [0, 3, 2, 3]) + engine.CiphertextArray(A.storage, [0, 1, 2, 3]), -2,
         "offsets decrease"),
        (lambda: A * engine.CiphertextArray(A.storage, [0, 1, 2]), -5, "storage holds"),
        (lambda: engine.CiphertextArray(A.storage, [0, 2]) + engine.CiphertextArray(A.storage, [0, 3]), -5, "storage holds"),
        (lambda: A * Z, -5, "words per block"),
        (lambda: A.gather([0, 2]), -2, "idx[1] = 2"),
        (lambda: key.decrypt_array(Z), -5, "words per block"),
        (lambda: key.decrypt_array(engine.CiphertextArray(A.storage, [0, 1])), -5, "storage holds"),
    ]
    for fn, code, text in cases:
        with pytest.raises(CsgnError) as ei:
            fn()
        assert ei.value.code == code and text in str(ei.value), str(ei.value)
    engine.sync()
    assert engine.device_info()["hbm_free"] == free0


def test_one_launch_per_call_for_ten_thousand_elements(engine):
    N, n = 1247, 10000
    rng = np.random.default_rng(4)
    ctx = engine.Context(N, 16)
    key = engine.SecretKey(ctx, random_key(rng, N, 16))
    A, B = key.encrypt_array(rng.integers(0, 2, n), seed=1), key.encrypt_array(rng.integers(0, 2, n), seed=2)
    engine.sync()
    for op in (lambda: A * B, lambda: A + B, lambda: key.decrypt_array(A)):
        c0 = engine.launch_count()
        op()
        assert engine.launch_count() - c0 <= 2
    # against one launch per item for the batch entry points
    a, b = [A.element(k) for k in range(64)], [B.element(k) for k in range(64)]
    c0 = engine.launch_count()
    engine.mul_batch(a, b)
    assert engine.launch_count() - c0 >= 64


def _adder_arrays(engine, key, xb, yb, lanes):
    """8-bit ripple-carry adder, SIMD over the lanes: s_i = x_i + y_i + c, c' = x_i*y_i + (x_i + y_i)*c."""
    bits = np.concatenate([np.concatenate([(xb >> i) & 1 for i in range(8)]),
                           np.concatenate([(yb >> i) & 1 for i in range(8)])]).astype(np.uint8)
    allb = key.encrypt_array(bits, seed=99)
    row = lambda r: allb.gather(np.arange(r * lanes, (r + 1) * lanes))      # noqa: E731
    X, Y = row(0), row(8)
    S, C = [X + Y], X * Y
    for i in range(1, 8):
        X, Y = row(i), row(8 + i)
        T = X + Y
        S.append(T + C)
        C = X * Y + T * C
    return allb, S, C


def test_simd_ripple_carry_adder(engine):
    N, D, lanes = 1247, 16, 1024
    rng = np.random.default_rng(8)
    ctx = engine.Context(N, D)
    key = engine.SecretKey(ctx, random_key(rng, N, D))
    xb, yb = rng.integers(0, 256, lanes), rng.integers(0, 256, lanes)
    allb, S, C = _adder_arrays(engine, key, xb, yb, lanes)
    got = np.zeros(lanes, dtype=np.int64)
    for i in range(8):
        got |= key.decrypt_array(S[i])[0].astype(np.int64) << i
    carry = key.decrypt_array(C)[0]
    assert np.array_equal(got, (xb + yb) % 256)
    assert np.array_equal(carry, (xb + yb) >> 8)
    for l in rng.choice(lanes, 16, replace=False):
        l = int(l)
        x = [allb.element(i * lanes + l) for i in range(8)]
        y = [allb.element((8 + i) * lanes + l) for i in range(8)]
        s, c = x[0] + y[0], x[0] * y[0]
        assert np.array_equal(s.getValues(), S[0].element(l).getValues())
        for i in range(1, 8):
            t = x[i] + y[i]
            s = t + c
            c = x[i] * y[i] + t * c
            assert np.array_equal(s.getValues(), S[i].element(l).getValues())
        assert np.array_equal(c.getValues(), C.element(l).getValues())


def _pipeline(engine, key, ctx, wa, wb, off):
    """A producer csgn_mul and consuming array calls with no synchronisation between them."""
    P = engine.Ciphertext.from_host(wa, ctx) * engine.Ciphertext.from_host(wb, ctx)
    arr = engine.CiphertextArray(P, off)
    Q = arr * arr.gather(np.arange(len(arr))[::-1])
    R = Q + arr
    bits, counts = key.decrypt_array(R)
    return [w.copy() for w in R.to_host()], counts


def test_ordering_with_producers_lanes_and_streams(engine, oracle):
    import torch
    N, D = 1247, 16
    rng = np.random.default_rng(21)
    ctx = engine.Context(N, D)
    s = random_key(rng, N, D)
    key = engine.SecretKey(ctx, s)
    mask = oracle.key_mask(N, s)
    wa, wb = _elements(rng, [300], N, mask)[0], _elements(rng, [200], N, mask)[0]
    sizes = _sizes("rand", rng, 300 * 200 // 5)
    sizes[-1] += 300 * 200 - sizes.sum()
    off = _offsets(sizes)
    engine.sync()
    ref_words, ref_counts = _pipeline(engine, key, ctx, wa, wb, off)
    prod = oracle.mul(wa, wb, words_per_block(N)).reshape(-1, words_per_block(N))
    engine.set_auto_lanes(True)
    try:
        words, counts = _pipeline(engine, key, ctx, wa, wb, off)
    finally:
        engine.set_auto_lanes(False)
    assert np.array_equal(counts, ref_counts) and all(np.array_equal(a, b) for a, b in zip(words, ref_words))
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        engine.set_stream(st.cuda_stream)
        try:
            words, counts = _pipeline(engine, key, ctx, wa, wb, off)
        finally:
            engine.set_stream(0)
    assert np.array_equal(counts, ref_counts) and all(np.array_equal(a, b) for a, b in zip(words, ref_words))
    # and against the oracle, element by element
    L = words_per_block(N)
    el = [prod[int(off[k]):int(off[k + 1])].reshape(-1) for k in range(len(off) - 1)]
    want = [oracle.concat(oracle.mul(a, b, L) if a.size and b.size else np.empty(0, np.uint64), a)
            for a, b in zip(el, el[::-1])]
    assert all(np.array_equal(a, b) for a, b in zip(ref_words, want))
    assert [int(c) for c in ref_counts] == [_count(oracle, w, N, s) for w in want]


def test_cpp_array_demo():
    exe = os.path.join(ROOT, "tests", "cpp", "bin", "array_demo")
    r = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:]
    assert "array_demo: 8-bit adder over 1024 lanes on CiphertextArray: all checks passed" in r.stdout
