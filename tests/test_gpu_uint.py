"""Encrypted integers on the GPU (csgn_encrypt_uint, csgn_decrypt_uint[_async]; SecretKey.encrypt_uint / decrypt_uint,
UIntCircuit, EncryptedUInt in Python; certFHE::UIntCircuit and EncryptedUInt in C++).

Encryption is checked word for word against csgn_encrypt_batch of the bit planes laid one after another and against the
oracle; decryption against the per-plane decrypt_array assembled on the host; whole expressions against numpy."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle.pyoracle import random_key, words_per_block

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
Vp = ctypes.c_void_p

pytestmark = pytest.mark.gpu


def _key(engine, N, D, seed):
    rng = np.random.default_rng(seed)
    s = random_key(rng, N, D)
    ctx = engine.Context(N, D)
    return rng, ctx, s, engine.SecretKey(ctx, s)


def _values(rng, n, W):
    hi = (1 << W) - 1
    return rng.integers(0, hi, size=n, dtype=np.uint64, endpoint=True)


def _planes_bits(values, W):
    """bit planes laid one after another: entry j*n + k = bit j of values[k]"""
    return np.concatenate([(values >> np.uint64(j)) & np.uint64(1) for j in range(W)]).astype(np.uint8)


def _assemble(key, x):
    """the per-plane decrypt_array of x put together on the host"""
    out = np.zeros(len(x), dtype=np.uint64)
    for j, p in enumerate(x.planes):
        out |= key.decrypt_array(p)[0].astype(np.uint64) << np.uint64(j)
    return out


def _words(x):
    return np.concatenate([p.storage.getValues() for p in x.planes])


# -- encryption -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [64, 191, 1247, 4097])          # L = 1, 3, 20, 65: the three kernel forms
@pytest.mark.parametrize("W", [1, 7, 32, 64])
def test_encrypt_matches_batch_and_oracle(engine, oracle, N, W):
    rng, ctx, s, key = _key(engine, N, 8, N + W)
    for n, first in [(0, 0), (1, 0), (1000, 0), (4096, 12345)]:
        v = _values(rng, n, W)
        x = key.encrypt_uint(v, W, seed=77, first_block=first)
        assert x.width == W and len(x) == n
        assert all(list(p.offsets) == list(range(n + 1)) for p in x.planes)
        if n == 0:
            assert all(p.storage.n_blocks == 0 for p in x.planes)
            continue
        bits = _planes_bits(v, W)
        want = key.encrypt_batch(bits, seed=77, first_block=first).getValues()
        assert np.array_equal(_words(x), want), "n=%d" % n
        if n * W <= 8000:
            assert np.array_equal(want, oracle.encrypt_batch(bits, N, s, 77, first))
        assert np.array_equal(key.decrypt_uint(x), v)


def test_one_launch_each_and_free_in_any_order(engine):
    rng, ctx, s, key = _key(engine, 1247, 16, 5)
    v = _values(rng, 4096, 32)
    engine.sync()
    c0 = engine.launch_count()
    x = key.encrypt_uint(v, 32, seed=1)
    assert engine.launch_count() - c0 == 1
    c0 = engine.launch_count()
    assert np.array_equal(key.decrypt_uint(x), v)
    assert engine.launch_count() - c0 == 1
    planes = list(x.planes)
    del x
    order = rng.permutation(32)
    for i, j in enumerate(order):
        planes[j] = None                                    # frees that handle of the shared allocation
        if i % 8 == 0:
            left = [k for k in range(32) if planes[k] is not None]
            for k in left[:2]:
                assert np.array_equal(key.decrypt_array(planes[k])[0], ((v >> np.uint64(k)) & np.uint64(1)).astype(np.uint8))
    engine.sync()


def test_values_that_do_not_fit_are_rejected(engine):
    from csgn_b200._native import CsgnError
    rng, ctx, s, key = _key(engine, 1247, 16, 6)
    engine.sync()
    free0 = engine.device_info()["hbm_free"]
    for v, W in [([0, 256], 8), ([1 << 63], 63), ([2], 1), ([0], 0), ([0], 65)]:
        with pytest.raises(CsgnError) as ei:
            key.encrypt_uint(np.array(v, dtype=np.uint64), W, seed=1)
        assert ei.value.code == -2, str(ei.value)
    engine.sync()
    assert engine.device_info()["hbm_free"] == free0
    assert np.array_equal(key.decrypt_uint(key.encrypt_uint(np.array([2**64 - 1], dtype=np.uint64), 64, seed=2)),
                          [2**64 - 1])


# -- decryption -------------------------------------------------------------------------------------------------------
def _circuit_outputs(engine, key, ctx, rng, n=600, cancel=True):
    """planes of different sizes with empty elements: a * b, a + b, a - b, a & b and a << 2 (whose low planes are the
    zero input) of 6-bit operands"""
    W = 6
    a, b = _values(rng, n, W), _values(rng, n, W)
    a[::5] = 0
    b[::5] = 0
    A, B = key.encrypt_uint(a, W, seed=10), key.encrypt_uint(b, W, seed=11, first_block=1 << 20)
    c = engine.UIntCircuit(W, 2)
    x, y = c.inputs
    outs = c.evaluate([A, B], [c.mul(x, y), c.add(x, y), c.sub(x, y), c.and_(x, y), c.shl(x, 2)], cancel=cancel)
    m = np.uint64(63)
    return outs, [(a * b) & m, (a + b) & m, (a - b) & m, a & b, (a << np.uint64(2)) & m]


def test_decrypt_equals_per_plane_decrypt(engine):
    rng, ctx, s, key = _key(engine, 1247, 16, 7)
    outs, want = _circuit_outputs(engine, key, ctx, rng)
    assert outs[-1].planes[0].storage.n_blocks == 0
    for x, w in zip(outs, want):
        got = key.decrypt_uint(x)
        assert np.array_equal(got, _assemble(key, x))
        assert np.array_equal(got, w)
    engine.sync()
    c0 = engine.launch_count()
    key.decrypt_uint(outs[0])
    assert engine.launch_count() - c0 == 1


@pytest.mark.parametrize("N", [191, 1247])                    # odd L on 8-byte units, even L on 16-byte units
def test_decrypt_large_elements(engine, monkeypatch, N):
    rng, ctx, s, key = _key(engine, N, 8, 8)
    outs, want = _circuit_outputs(engine, key, ctx, rng, n=300)
    L = words_per_block(N)
    monkeypatch.setenv("CSGN_SEG_LARGE_BYTES", str(8 * L * 4))     # elements of 4 blocks or more: one fold each
    for x, w in zip(outs, want):
        big = sum(p.blocks(k) >= 4 for p in x.planes for k in range(len(x)))
        engine.sync()
        c0 = engine.launch_count()
        got = key.decrypt_uint(x)
        launched = engine.launch_count() - c0
        assert np.array_equal(got, w)
        assert np.array_equal(got, _assemble(key, x))
        if big:
            assert launched >= big + 1
    monkeypatch.setenv("CSGN_SEG_LARGE_BYTES", "0")                # every element on its own
    assert np.array_equal(key.decrypt_uint(outs[0]), want[0])


def test_decrypt_async_and_other_stream(engine):
    import torch
    rng, ctx, s, key = _key(engine, 1247, 16, 9)
    v = _values(rng, 5000, 20)
    x = key.encrypt_uint(v, 20, seed=3)
    d = torch.full((5000,), -1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()                               # the fill runs on torch's stream, the decrypt on the library's
    key.decrypt_uint_async(x, d.data_ptr())
    engine.sync()
    assert np.array_equal(d.cpu().numpy().view(np.uint64), v)
    # producer (encrypt + circuit) and consumer on a caller's stream, no synchronisation in between
    engine.sync()
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        engine.set_stream(st.cuda_stream)
        try:
            a, b = _values(rng, 4096, 16), _values(rng, 4096, 16)
            A, B = key.encrypt_uint(a, 16, seed=4), key.encrypt_uint(b, 16, seed=5)
            S = A + B
            out = torch.empty(4096, dtype=torch.int64, device="cuda")
            key.decrypt_uint_async(S, out.data_ptr())
            got = out.cpu().numpy().view(np.uint64).copy()
        finally:
            engine.set_stream(0)
    assert np.array_equal(got, (a + b) & np.uint64(0xFFFF))


def test_argument_errors_allocate_nothing(engine):
    from csgn_b200._native import CsgnError, check
    lib = engine._lib()
    rng, ctx, s, key = _key(engine, 1247, 16, 10)
    x = key.encrypt_uint(_values(rng, 10, 4), 4, seed=1)
    other = engine.SecretKey(engine.Context(64, 4), random_key(rng, 64, 4))
    planes = (Vp * 4)(*[p.storage._h for p in x.planes])
    offs = (Vp * 4)(*[p.offsets.ctypes.data for p in x.planes])
    bad = np.array([0, 1, 3, 2] + list(range(4, 11)), dtype=np.uint64)
    bad_offs = (Vp * 4)(*([bad.ctypes.data] + [p.offsets.ctypes.data for p in x.planes[1:]]))
    null_planes = (Vp * 4)(*([None] + [p.storage._h for p in x.planes[1:]]))
    vals = np.zeros(10, dtype=np.uint64)
    vp = vals.ctypes.data_as(Vp)
    out = (Vp * 4)()
    cases = [
        (lambda: lib.csgn_decrypt_uint(None, offs, 4, 10, key._h, vp), -2),
        (lambda: lib.csgn_decrypt_uint(planes, None, 4, 10, key._h, vp), -2),
        (lambda: lib.csgn_decrypt_uint(planes, offs, 4, 10, None, vp), -2),
        (lambda: lib.csgn_decrypt_uint(planes, offs, 4, 10, key._h, None), -2),
        (lambda: lib.csgn_decrypt_uint(planes, offs, 0, 10, key._h, vp), -2),
        (lambda: lib.csgn_decrypt_uint(planes, offs, 65, 10, key._h, vp), -2),
        (lambda: lib.csgn_decrypt_uint(null_planes, offs, 4, 10, key._h, vp), -2),
        (lambda: lib.csgn_decrypt_uint(planes, bad_offs, 4, 10, key._h, vp), -2),
        (lambda: lib.csgn_decrypt_uint(planes, offs, 4, 9, key._h, vp), -5),
        (lambda: lib.csgn_decrypt_uint(planes, offs, 4, 10, other._h, vp), -5),
        (lambda: lib.csgn_decrypt_uint_async(planes, offs, 4, 10, key._h, None), -2),
        (lambda: lib.csgn_encrypt_uint(None, vp, 10, 4, 0, 1, out), -2),
        (lambda: lib.csgn_encrypt_uint(key._h, None, 10, 4, 0, 1, out), -2),
        (lambda: lib.csgn_encrypt_uint(key._h, vp, 10, 4, 0, 1, None), -2),
    ]
    engine.sync()
    free0 = engine.device_info()["hbm_free"]
    for i, (fn, code) in enumerate(cases):
        rc = fn()
        assert rc == code, "case %d: %d (%s)" % (i, rc, lib.csgn_last_error())
    engine.sync()
    assert engine.device_info()["hbm_free"] == free0
    # n == 0: empty planes, no launch
    e = key.encrypt_uint(np.zeros(0, dtype=np.uint64), 3, seed=1)
    engine.sync()
    c0 = engine.launch_count()
    assert key.decrypt_uint(e).size == 0
    assert engine.launch_count() - c0 == 0


# -- whole expressions ------------------------------------------------------------------------------------------------
BINARY = {
    "add": lambda a, b, m: (a + b) & m, "sub": lambda a, b, m: (a - b) & m, "mul": lambda a, b, m: (a * b) & m,
    "lt": lambda a, b, m: (a < b).astype(np.uint64), "gt": lambda a, b, m: (a > b).astype(np.uint64),
    "ne": lambda a, b, m: (a != b).astype(np.uint64), "eq": lambda a, b, m: (a == b).astype(np.uint64),
    "le": lambda a, b, m: (a <= b).astype(np.uint64), "ge": lambda a, b, m: (a >= b).astype(np.uint64),
    "min": lambda a, b, m: np.minimum(a, b), "max": lambda a, b, m: np.maximum(a, b),
    "and_": lambda a, b, m: a & b, "xor": lambda a, b, m: a ^ b, "or_": lambda a, b, m: a | b,
}
NEEDS_ONE = {"eq", "le", "ge"}


# Operations whose results stay small at any width run at 8 and 32 bits.  The others hold, per lane, about 3^W blocks
# (the monomials of their algebraic normal form that compaction keeps; lt and ne of two W-bit operands have 3^W - 1), so
# 32-bit ones do not fit in device memory: they run at 8 bits.
_ANY_WIDTH = {"add", "and_", "xor", "or_"}


def _cases():
    for op in sorted(BINARY):
        if op == "mul":
            # without cancellation a multiplier's products repeat monomials along many paths and its gates grow into
            # the thousands of blocks per lane; a 4-bit one keeps that path covered at a size that stays small
            yield from [("mul", 8, True), ("mul", 12, True), ("mul", 4, False)]
            continue
        for W in ((8, 32) if op in _ANY_WIDTH else (8,)):
            for cancel in (True, False):
                yield op, W, cancel


@pytest.mark.parametrize("op,W,cancel", list(_cases()))
def test_every_operation_end_to_end(engine, op, W, cancel):
    rng, ctx, s, key = _key(engine, 1247, 16, W * 100 + len(op))
    n = 4096
    a, b = _values(rng, n, W), _values(rng, n, W)
    b[:64] = a[:64]
    A, B = key.encrypt_uint(a, W, seed=1), key.encrypt_uint(b, W, seed=2, first_block=n * W)
    one = key.encrypt_array(np.ones(n, dtype=np.uint8), seed=3) if op in NEEDS_ONE else None
    c = engine.UIntCircuit(W, 2, one=one is not None)
    r = getattr(c, op)(*c.inputs)
    (x,) = c.evaluate([A, B], [r], cancel=cancel, one=one)
    got = key.decrypt_uint(x)
    m = np.uint64((1 << W) - 1)
    assert np.array_equal(got, BINARY[op](a, b, m)), "%s W=%d cancel=%s (%d fallback lanes)" % (
        op, W, cancel, c.last_fallback)


def test_unary_and_select(engine):
    rng, ctx, s, key = _key(engine, 1247, 16, 11)
    n, W = 4096, 8
    a, b, sel = _values(rng, n, W), _values(rng, n, W), _values(rng, n, 1)
    A, B, S = key.encrypt_uint(a, W, seed=1), key.encrypt_uint(b, W, seed=2, first_block=1 << 30), \
        key.encrypt_uint(sel, 1, seed=3, first_block=1 << 31)
    one = key.encrypt_array(np.ones(n, dtype=np.uint8), seed=4)
    c = engine.UIntCircuit(W, 3, one=True)
    x, y, z = c.inputs
    rs = [c.neg(x), c.invert(x), c.shl(x, 3), c.shr(x, 2), c.select(z[:1], x, y)]
    outs = c.evaluate([A, B, S], rs, cancel=True, one=one)
    m = np.uint64(255)
    want = [(0 - a) & m, ~a & m, (a << np.uint64(3)) & m, a >> np.uint64(2), np.where(sel == 1, a, b)]
    for o, w in zip(outs, want):
        assert np.array_equal(key.decrypt_uint(o), w)
    with pytest.raises(ValueError):
        engine.UIntCircuit(W, 1).invert(x)


def test_composite_expression_in_one_call(engine):
    """min(a + b, c) - a and lt(a + b, c), one csgn_seg_circuit call.  Cancelled, a 5-bit result bit holds at most 2963
    blocks per lane (its algebraic normal form); uncancelled, the netlist's bound passes 10^11 blocks at 4 bits."""
    rng, ctx, s, key = _key(engine, 1247, 16, 12)
    n, W = 4096, 5
    a, b, cc = (_values(rng, n, W) for _ in range(3))
    X = [key.encrypt_uint(v, W, seed=20 + i, first_block=i << 24) for i, v in enumerate((a, b, cc))]
    c = engine.UIntCircuit(W, 3)
    x, y, z = c.inputs
    sm = c.add(x, y)
    r1, r2 = c.evaluate(X, [c.sub(c.min(sm, z), x), c.lt(sm, z)], cancel=True)
    m = np.uint64((1 << W) - 1)
    assert np.array_equal(key.decrypt_uint(r1), (np.minimum((a + b) & m, cc) - a) & m)
    assert np.array_equal(key.decrypt_uint(r2), (((a + b) & m) < cc).astype(np.uint64))


def test_eager_operators(engine):
    rng, ctx, s, key = _key(engine, 1247, 16, 13)
    n, W = 4096, 8
    a, b = _values(rng, n, W), _values(rng, n, W)
    A, B = key.encrypt_uint(a, W, seed=1), key.encrypt_uint(b, W, seed=2, first_block=1 << 30)
    m = np.uint64(255)
    D = lambda x: key.decrypt_uint(x)                                          # noqa: E731
    assert np.array_equal(D(A + B), (a + b) & m)
    assert np.array_equal(D(A - B), (a - b) & m)
    assert np.array_equal(D(A * B), (a * b) & m)
    lt = A < B
    assert lt.width == 1 and np.array_equal(D(lt), (a < b).astype(np.uint64))
    assert np.array_equal(D(A > B), (a > b).astype(np.uint64))
    assert np.array_equal(D(A & B), a & b)
    assert np.array_equal(D(A ^ B), a ^ b)
    assert np.array_equal(D(A | B), a | b)
    assert np.array_equal(D(engine.EncryptedUInt.select(lt, A, B)), np.minimum(a, b))
    # mixed widths: the 1-bit comparison zero-extended
    assert np.array_equal(D(A + lt), (a + (a < b)) & m)


def test_cpp_uint_demo():
    exe = os.path.join(ROOT, "tests", "cpp", "bin", "uint_demo")
    r = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:]
    assert "uint_demo: all checks passed" in r.stdout
