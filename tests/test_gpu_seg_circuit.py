"""Circuits over ciphertext arrays (csgn_seg_circuit; Circuit in Python, certFHE::Circuit in C++): every output of the
one-call circuit equals, word for word and offset for offset, what the gate-by-gate loop over the existing array calls
gives in the same test (sum_of_products, compacted to min_bits, cancelled after every gate)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle.pyoracle import random_blocks, random_key, words_per_block

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NS = [1, 191, 1247, 4096, 4097, 16383]     # L = 1, 3, 20 (10 16-byte units), 64 (32 units), 65 (odd), 256 (128 units)
DISTS = ["uniform", "skewed", "empty"]
Vp = ctypes.c_void_p

pytestmark = pytest.mark.gpu


# -- netlists: lists of (products, terms) over wire ids; wires 0 .. n_inputs - 1 are the inputs --------------------
def adder(bits):
    """inputs x_0 .. x_{bits-1}, y_0 ..; outputs the sum bits and the final carry"""
    g, outs = [], []
    w = 2 * bits

    def gate(p, t):
        nonlocal w
        g.append((p, t))
        w += 1
        return w - 1
    outs.append(gate([], [0, bits]))
    c = gate([(0, bits)], [])
    for i in range(1, bits):
        t = gate([], [i, bits + i])
        outs.append(gate([], [t, c]))
        c = gate([(i, bits + i), (t, c)], [])
    return 2 * bits, g, outs + [c]


def multiplier(bits):
    """x * y mod 2^bits, schoolbook rows added with ripple carries"""
    g = []
    w = 2 * bits

    def gate(p, t):
        nonlocal w
        g.append((p, t))
        w += 1
        return w - 1
    acc = [None] * bits
    for j in range(bits):
        pp = [None] * j + [gate([(i, bits + j)], []) for i in range(bits - j)]
        c, out = None, []
        for k in range(bits):
            ops = [x for x in (acc[k], pp[k], c) if x is not None]
            out.append(gate([], ops) if ops else None)
            prods = [(ops[p], ops[q]) for p in range(len(ops)) for q in range(p + 1, len(ops))]
            c = gate(prods, []) if prods else None
        acc = out
    return 2 * bits, g, acc


def majority_mux():
    """inputs a, b, s: majority(a, b, s) = ab + as + bs and mux(s, a, b) = sa + sb + b, and the output a itself"""
    g = [([(0, 1), (0, 2), (1, 2)], []), ([(2, 0), (2, 1)], [1])]
    return 3, g, [3, 4, 0]


def random_netlist(rng, n_inputs, n_gates, most=1500):
    """seeded gates over earlier wires, with x*x, a + a and wires read many times.  A product whose worst-case size
    (inputs of up to 5 blocks, no compaction) would pass `most` blocks per lane becomes a term."""
    g, size = [], [5] * n_inputs
    for k in range(n_gates):
        w = n_inputs + k
        pick = lambda: int(rng.integers(max(0, w - 6), w)) if rng.random() < 0.7 else int(rng.integers(0, w))  # noqa
        p = [(pick(), pick()) for _ in range(int(rng.integers(0, 3)))]
        t = [pick() for _ in range(int(rng.integers(0 if p else 1, 3)))]
        if k % 5 == 1:
            x = pick()
            p.append((x, x))                       # x * x
        if k % 7 == 2:
            t += [t[0]] if t else [pick(), pick()]  # a + a
        total = 0
        for u, v in list(p):
            if total + size[u] * size[v] > most:
                p.remove((u, v))
                t.append(u)
            else:
                total += size[u] * size[v]
        if sum(size[x] for x in t) + total > most:
            t = t[:1] if not p else []
        if not p and not t:
            t = [0]
        size.append(total + sum(size[x] for x in t))
        g.append((p, t))
    outs = sorted({n_inputs + n_gates - 1, n_inputs + n_gates // 2, 0, int(rng.integers(n_inputs, n_inputs + n_gates))})
    return n_inputs, g, outs


# -- inputs ---------------------------------------------------------------------------------------------------------
def _sizes(dist, rng, n):
    if dist == "uniform":
        return np.full(n, 2, dtype=np.int64)
    if dist == "skewed":
        s = np.ones(n, dtype=np.int64)
        s[rng.random(n) < 0.2] = 4
        return s
    s = rng.integers(0, 3, size=n)
    s[rng.random(n) < 0.6] = 0
    return s


def _blocks(rng, t, N):
    """t blocks of mixed density: some dense, some with a handful of set bits, so compaction keeps some and drops some"""
    L = words_per_block(N)
    w = random_blocks(rng, t, N).reshape(-1, L)
    for r in range(t):
        for _ in range(int(rng.choice([0, 1, 2, 4]))):
            w[r] &= random_blocks(rng, 1, N)
    return w.reshape(-1)


def _inputs(engine, rng, ctx, n_inputs, n, dist):
    return [engine.CiphertextArray.from_host([_blocks(rng, int(t), ctx.N) for t in _sizes(dist, rng, n)], ctx)
            for _ in range(n_inputs)]


# -- the gate-by-gate loop through the existing calls -----------------------------------------------------------------
def _gate(engine, products, terms, min_bits):
    """csgn_seg_mul_sum (min_bits 0) or csgn_seg_mul_sum_compact(min_bits) over the arrays given"""
    if min_bits == 0:
        return engine.CiphertextArray.sum_of_products(products, terms)
    arrays = [x for pr in products for x in pr] + list(terms)
    n, ctx = len(arrays[0]), arrays[0].ctx
    h = lambda xs: engine.handle_array([x.storage for x in xs]) if xs else None                    # noqa: E731
    o = lambda xs: (Vp * len(xs))(*[x.offsets.ctypes.data for x in xs]) if xs else None            # noqa: E731
    left, right = [x for x, _ in products], [y for _, y in products]
    out_off = np.empty(n + 1, dtype=np.uint64)
    out = Vp()
    from csgn_b200._native import check
    check(engine._lib().csgn_seg_mul_sum_compact(h(left), o(left), h(right), o(right), len(products), h(terms),
                                                  o(terms), len(terms), n, min_bits, out_off.ctypes.data_as(Vp),
                                                  ctypes.byref(out)))
    return engine.CiphertextArray(engine.Ciphertext(out, ctx), out_off)


def _gate_by_gate(engine, inputs, gates, outputs, min_bits, cancel):
    wires = list(inputs)
    for p, t in gates:
        x = _gate(engine, [(wires[u], wires[v]) for u, v in p], [wires[w] for w in t], min_bits)
        wires.append(x.cancel() if cancel else x)
    return [wires[w] for w in outputs]


def _circuit(engine, n_inputs, gates):
    C = engine.Circuit(n_inputs)
    for k, (p, t) in enumerate(gates):
        assert C.gate(p, t) == n_inputs + k
    return C


def _assert_same(got, want):
    assert len(got) == len(want)
    for j, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g.offsets, w.offsets), "output %d: offsets differ" % j
        assert np.array_equal(g.storage.getValues(), w.storage.getValues()), "output %d: words differ" % j


def _check(engine, inputs, net, min_bits, cancel, lane_capacity=0):
    n_inputs, gates, outs = net
    C = _circuit(engine, n_inputs, gates)
    got = C.evaluate(inputs, outs, min_bits=min_bits, cancel=cancel, lane_capacity=lane_capacity)
    _assert_same(got, _gate_by_gate(engine, inputs, gates, outs, min_bits, cancel))
    return C.last_fallback, got


def _ctx(engine, N):
    return engine.Context(N, min(16, N))


# -- equivalence ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("dist", DISTS)
def test_circuits_equal_the_gate_by_gate_loop(engine, N, dist):
    rng = np.random.default_rng(N * 3 + DISTS.index(dist))
    ctx = _ctx(engine, N)
    n = 24 if N > 4000 else 64
    nets = [adder(3), multiplier(3), majority_mux(), random_netlist(rng, 3, 14)]
    for net in nets:
        inputs = _inputs(engine, rng, ctx, net[0], n, dist)
        for min_bits in (0, 1, ctx.D):
            for cancel in (False, True):
                _check(engine, inputs, net, min_bits, cancel)


@pytest.mark.parametrize("seed", range(6))
def test_random_netlists(engine, seed):
    rng = np.random.default_rng(100 + seed)
    N = [191, 1247, 4097][seed % 3]
    ctx = _ctx(engine, N)
    net = random_netlist(rng, 2 + seed % 3, 20 + 5 * seed)
    inputs = _inputs(engine, rng, ctx, net[0], 80, DISTS[seed % 3])
    for min_bits, cancel in ((ctx.D, True), (ctx.D, False), (1, True), (0, True)):
        _check(engine, inputs, net, min_bits, cancel)


def test_square_and_double_inside_a_circuit(engine):
    """x*x cancels to x and a + a to nothing, inside the one call"""
    rng = np.random.default_rng(7)
    ctx = _ctx(engine, 1247)
    X = _inputs(engine, rng, ctx, 1, 100, "skewed")[0]
    net = (1, [([(0, 0)], []), ([], [0, 0]), ([(1, 1)], [2])], [1, 2, 3])
    _, got = _check(engine, [X], net, 0, True)
    assert np.array_equal(got[0].offsets, X.offsets)
    assert got[1].storage.n_blocks == 0


# -- capacity and fallback ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("cancel", [False, True])
def test_fallback_lanes_give_the_same_result(engine, cancel):
    rng = np.random.default_rng(11)
    ctx = _ctx(engine, 1247)
    n = 200
    net = adder(3)
    inputs = _inputs(engine, rng, ctx, net[0], n, "skewed")
    inputs = [engine.CiphertextArray.from_host([np.concatenate([_blocks(rng, 1, ctx.N), e]) for e in x.to_host()], ctx)
              for x in inputs]                                         # no empty lane
    fb, ref = _check(engine, inputs, net, 0, cancel)
    assert fb == 0                                                     # roomy
    fb, _ = _check(engine, inputs, net, 0, cancel, lane_capacity=1)
    assert fb == n                                                     # tiny
    partial = []
    for cap in (8, 16, 32, 64, 128, 256, 512, 1024):
        fb, got = _check(engine, inputs, net, 0, cancel, lane_capacity=cap)
        _assert_same(got, ref)
        partial.append(0 < fb < n)
    assert any(partial), "no middling capacity split the lanes"


# -- decryption -------------------------------------------------------------------------------------------------------
def test_decryptions_equal_the_plaintext_circuits(engine):
    N, D, n, bits = 1247, 16, 512, 5
    rng = np.random.default_rng(13)
    ctx = engine.Context(N, D)
    for kk in range(3):
        key = engine.SecretKey(ctx, random_key(rng, N, D))
        x, y = rng.integers(0, 1 << bits, n), rng.integers(0, 1 << bits, n)
        x[::9] = y[::9] = (1 << bits) - 1
        plain = np.concatenate([(v >> i) & 1 for v in (x, y) for i in range(bits)]).astype(np.uint8)
        allb = key.encrypt_array(plain, seed=31 + kk)
        rows = [allb.gather(np.arange(r * n, (r + 1) * n)) for r in range(2 * bits)]

        def word(arrs):
            v = np.zeros(n, dtype=np.int64)
            for i, a in enumerate(arrs):
                v |= key.decrypt_array(a)[0].astype(np.int64) << i
            return v
        for net, want, cancel in ((adder(bits), x + y, False), (multiplier(bits), (x * y) % (1 << bits), True)):
            C = _circuit(engine, *net[:2])
            assert np.array_equal(word(C.evaluate(rows, net[2], cancel=cancel)), want)
            assert np.array_equal(word(C.evaluate(rows, net[2], min_bits=0, cancel=cancel)), want)
        a, b, s = rows[0], rows[1], rows[bits]
        C = _circuit(engine, *majority_mux()[:2])
        maj, mux, same = C.evaluate([a, b, s], majority_mux()[2])
        xa, xb, xs = x & 1, (x >> 1) & 1, y & 1
        assert np.array_equal(key.decrypt_array(maj)[0], (xa & xb) | (xa & xs) | (xb & xs))
        assert np.array_equal(key.decrypt_array(mux)[0], np.where(xs == 1, xa, xb))
        assert np.array_equal(key.decrypt_array(same)[0], xa)


# -- argument errors ----------------------------------------------------------------------------------------------
def test_argument_errors_allocate_nothing(engine):
    """The C ABI's own checks: ctypes calls straight into csgn_seg_circuit, so no Python check runs first."""
    from csgn_b200._native import CsgnError, check
    lib = engine._lib()
    rng = np.random.default_rng(3)
    ctx = _ctx(engine, 1247)
    A = engine.CiphertextArray.from_host([random_blocks(rng, 2, 1247), random_blocks(rng, 1, 1247)], ctx)
    B = engine.CiphertextArray.from_host([random_blocks(rng, 1, 1247), random_blocks(rng, 1, 1247)], ctx)
    ctx2 = _ctx(engine, 191)
    W = engine.CiphertextArray.from_host([random_blocks(rng, 1, 191), random_blocks(rng, 1, 191)], ctx2)

    def call(arrays, offs, gates, n_gates, outputs, min_bits=16, gates_len=None):
        g = np.asarray(gates, dtype=np.uint32)
        o = np.asarray(outputs, dtype=np.uint32)
        offs = [np.ascontiguousarray(x, dtype=np.uint64) for x in offs]
        out_off = [np.empty(3, dtype=np.uint64) for _ in outputs]
        out = (Vp * max(1, len(outputs)))()
        check(lib.csgn_seg_circuit(engine.handle_array([x.storage for x in arrays]),
                                   (Vp * len(offs))(*[x.ctypes.data for x in offs]), len(arrays), 2,
                                   g.ctypes.data_as(Vp), g.size if gates_len is None else gates_len, n_gates,
                                   o.ctypes.data_as(Vp), o.size, min_bits, 0, 0,
                                   (Vp * max(1, len(outputs)))(*[x.ctypes.data for x in out_off]), out, None))
        pytest.fail("the call succeeded")

    ok = [A.offsets, B.offsets]
    cases = [
        (lambda: call([A, B], ok, [1, 0, 0, 2], 1, [2]), "reads wire 2"),                # an operand at its own wire
        (lambda: call([A, B], ok, [1, 0, 0, 5], 1, [2]), "reads wire 5"),                # a forward reference
        (lambda: call([A, B], ok, [0, 0], 1, [2]), "no products and no terms"),
        (lambda: call([A, B], ok, [1, 0, 0, 1], 1, [2], gates_len=3), "gates_len = 3 ends inside gate 0"),
        (lambda: call([A, B], ok, [1, 0, 0, 1, 7], 1, [2]), "gates_len = 5, the 1 gates encode 4"),
        (lambda: call([A, B], ok, [1, 0, 0, 1], 2, [2]), "ends inside gate 1"),
        (lambda: call([A, B], ok, [1, 0, 0, 1], 1, [3]), "output 0 names wire 3"),
        (lambda: call([A, W], [A.offsets, W.offsets], [1, 0, 0, 1], 1, [2]), "words per block differ"),
        (lambda: call([A, B], [A.offsets, [0, 1, 3]], [1, 0, 0, 1], 1, [2]), "input 1: offsets[2] = 3"),
        (lambda: call([A, B], [[1, 2, 3], B.offsets], [1, 0, 0, 1], 1, [2]), "input 0: offsets[0]"),
        (lambda: call([A, B], [[0, 3, 2], B.offsets], [1, 0, 0, 1], 1, [2]), "input 0: offsets decrease"),
        (lambda: call([A, B], ok, [1, 0, 0, 1], 1, [2], min_bits=64 * 20 + 1), "min_bits = 1281 outside"),
        (lambda: call([A, B], ok, [1, 0, 0, 1], 1, []), "at least one output"),
    ]
    engine.sync()
    free0 = engine.device_info()["hbm_free"]
    for fn, text in cases:
        with pytest.raises(CsgnError) as ei:
            fn()
        assert text in str(ei.value), str(ei.value)
    engine.sync()
    assert engine.device_info()["hbm_free"] == free0
    with pytest.raises(ValueError):
        engine.Circuit(2).gate([(0, 2)])
    C = engine.Circuit(2)
    C.gate([], [0])
    with pytest.raises(ValueError):
        C.evaluate([A, W], [2])                                        # arrays of two contexts


def test_no_lanes_empty_lanes_and_input_outputs(engine):
    ctx = _ctx(engine, 1247)
    net = adder(2)
    C = _circuit(engine, *net[:2])
    E = [engine.CiphertextArray(engine.Ciphertext.empty(0, ctx), np.zeros(n + 1, dtype=np.uint64))
         for n in (0, 0, 0, 0)]
    for R in C.evaluate(E, net[2] + [0]):
        assert len(R) == 0 and R.storage.n_blocks == 0
    E = [engine.CiphertextArray(engine.Ciphertext.empty(0, ctx), np.zeros(6, dtype=np.uint64)) for _ in range(4)]
    for R in C.evaluate(E, net[2], cancel=True):
        assert len(R) == 5 and R.storage.n_blocks == 0 and not R.offsets.any()
    rng = np.random.default_rng(5)
    X = _inputs(engine, rng, ctx, 4, 30, "empty")
    _check(engine, X, (4, net[1], [3, 1, 3]), ctx.D, True)            # outputs that are inputs only: no gate output
    _check(engine, X, (4, net[1], [3] + net[2] + [0]), ctx.D, True)


# -- launch bound ---------------------------------------------------------------------------------------------------
def test_launches_do_not_grow_with_lanes_or_gates(engine):
    rng = np.random.default_rng(9)
    ctx = _ctx(engine, 1247)
    counts = []
    for bits in (4, 8):
        net = adder(bits)
        C = _circuit(engine, *net[:2])
        outs = net[2][-3:]                                             # the same number of outputs
        for n in (10, 10000):
            key = engine.SecretKey(ctx, random_key(rng, ctx.N, ctx.D))
            allb = key.encrypt_array(rng.integers(0, 2, net[0] * n).astype(np.uint8), seed=n + bits)
            inputs = [allb.gather(np.arange(r * n, (r + 1) * n)) for r in range(net[0])]
            engine.sync()
            c0 = engine.launch_count()
            C.evaluate(inputs, outs)
            counts.append(engine.launch_count() - c0)
            assert C.last_fallback == 0
    assert counts == [1 + 3] * 4, counts


def test_cpp_circuit_demo():
    exe = os.path.join(ROOT, "tests", "cpp", "bin", "circuit_demo")
    r = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:]
    assert "circuit_demo: 16-bit adder and 5-bit multiplier over 1024 lanes as circuits: all checks passed" in r.stdout
