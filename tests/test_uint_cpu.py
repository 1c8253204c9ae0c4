"""Integer netlists (UIntCircuit) on plaintext bits, without a GPU: the flat netlist is evaluated over GF(2) (every gate
an XOR of ANDs) and compared with numpy integer arithmetic mod 2^W.  The C++ builder (certFHE::UIntCircuit) must emit
the same netlists, wire for wire."""
import itertools
import os
import subprocess

import numpy as np
import pytest

from csgn_b200.engine import UIntCircuit

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# op -> (operands, builder, numpy reference over uint64 lanes, needs `one`)
BINARY = {
    "add": (lambda c, a, b: c.add(a, b), lambda a, b, m: (a + b) & m, False),
    "sub": (lambda c, a, b: c.sub(a, b), lambda a, b, m: (a - b) & m, False),
    "mul": (lambda c, a, b: c.mul(a, b), lambda a, b, m: (a * b) & m, False),
    "lt": (lambda c, a, b: c.lt(a, b), lambda a, b, m: (a < b).astype(np.uint64), False),
    "gt": (lambda c, a, b: c.gt(a, b), lambda a, b, m: (a > b).astype(np.uint64), False),
    "ne": (lambda c, a, b: c.ne(a, b), lambda a, b, m: (a != b).astype(np.uint64), False),
    "eq": (lambda c, a, b: c.eq(a, b), lambda a, b, m: (a == b).astype(np.uint64), True),
    "le": (lambda c, a, b: c.le(a, b), lambda a, b, m: (a <= b).astype(np.uint64), True),
    "ge": (lambda c, a, b: c.ge(a, b), lambda a, b, m: (a >= b).astype(np.uint64), True),
    "min": (lambda c, a, b: c.min(a, b), lambda a, b, m: np.minimum(a, b), False),
    "max": (lambda c, a, b: c.max(a, b), lambda a, b, m: np.maximum(a, b), False),
    "and": (lambda c, a, b: c.and_(a, b), lambda a, b, m: a & b, False),
    "xor": (lambda c, a, b: c.xor(a, b), lambda a, b, m: a ^ b, False),
    "or": (lambda c, a, b: c.or_(a, b), lambda a, b, m: a | b, False),
}
UNARY = {
    "neg": (lambda c, a: c.neg(a), lambda a, m: (0 - a) & m, False),
    "invert": (lambda c, a: c.invert(a), lambda a, m: ~a & m, True),
    "shl3": (lambda c, a: c.shl(a, 3), lambda a, m: (a << np.uint64(3)) & m, False),
    "shr2": (lambda c, a: c.shr(a, 2), lambda a, m: a >> np.uint64(2), False),
}


def run_netlist(circ, operands, width):
    """Evaluate the flat netlist over GF(2), lane by lane with numpy bool vectors; the inputs are the bit planes of
    `operands` (uint64 arrays), then `one`, then the zero wire."""
    n_inputs, gates = circ.netlist()
    n = operands[0].size
    wires = []
    for v in operands:
        wires += [((v >> np.uint64(j)) & np.uint64(1)).astype(bool) for j in range(width)]
    if circ.one is not None:
        wires.append(np.ones(n, dtype=bool))
    wires.append(np.zeros(n, dtype=bool))
    assert len(wires) == n_inputs
    i = 0
    while i < len(gates):
        p, q = gates[i], gates[i + 1]
        i += 2
        acc = np.zeros(n, dtype=bool)
        for _ in range(p):
            acc ^= wires[gates[i]] & wires[gates[i + 1]]
            i += 2
        for _ in range(q):
            acc ^= wires[gates[i]]
            i += 1
        wires.append(acc)
    return wires


def value(wires, result):
    out = np.zeros(wires[0].size, dtype=np.uint64)
    for j, w in enumerate(result):
        out |= wires[w].astype(np.uint64) << np.uint64(j)
    return out


def mask(w):
    return np.uint64((1 << w) - 1) if w < 64 else np.uint64(0xFFFFFFFFFFFFFFFF)


def check_binary(op, wa, wb, a, b):
    build, ref, needs_one = BINARY[op]
    W = max(wa, wb)
    c = UIntCircuit(W, 2, one=needs_one)
    r = build(c, c.inputs[0][:wa], c.inputs[1][:wb])
    got = value(run_netlist(c, [a, b], W), r)
    with np.errstate(over="ignore"):
        want = ref(a, b, mask(W))
    np.testing.assert_array_equal(got, want, err_msg="%s at %d x %d bits" % (op, wa, wb))


def exhaustive(wa, wb):
    a, b = zip(*itertools.product(range(1 << wa), range(1 << wb)))
    return np.array(a, dtype=np.uint64), np.array(b, dtype=np.uint64)


@pytest.mark.parametrize("op", sorted(BINARY))
@pytest.mark.parametrize("W", [1, 2, 3, 4, 5])
def test_binary_exhaustive(op, W):
    check_binary(op, W, W, *exhaustive(W, W))


@pytest.mark.parametrize("op", sorted(BINARY))
@pytest.mark.parametrize("wa,wb", [(1, 4), (5, 2), (3, 5)])
def test_binary_mixed_widths(op, wa, wb):
    check_binary(op, wa, wb, *exhaustive(wa, wb))


@pytest.mark.parametrize("op", sorted(BINARY))
@pytest.mark.parametrize("W", [16, 32, 64])
def test_binary_random(op, W):
    rng = np.random.default_rng(1000 + W)
    hi = np.uint64((1 << W) - 1) if W < 64 else np.uint64(0xFFFFFFFFFFFFFFFF)
    a = rng.integers(0, hi, size=10_000, dtype=np.uint64, endpoint=True)
    b = rng.integers(0, hi, size=10_000, dtype=np.uint64, endpoint=True)
    b[:100] = a[:100]                     # equal pairs for eq / le / ge
    check_binary(op, W, W, a, b)


@pytest.mark.parametrize("op", sorted(UNARY))
@pytest.mark.parametrize("W", [1, 3, 5, 16, 64])
def test_unary(op, W):
    build, ref, needs_one = UNARY[op]
    c = UIntCircuit(W, 1, one=needs_one)
    r = build(c, c.inputs[0])
    rng = np.random.default_rng(W)
    a = np.arange(1 << W, dtype=np.uint64) if W <= 5 else rng.integers(0, mask(W), size=10_000, dtype=np.uint64,
                                                                        endpoint=True)
    got = value(run_netlist(c, [a], W), r)
    with np.errstate(over="ignore"):
        np.testing.assert_array_equal(got, ref(a, mask(W)))


@pytest.mark.parametrize("W", [1, 4, 5])
def test_select(W):
    c = UIntCircuit(W, 3)
    r = c.select(c.inputs[0][:1], c.inputs[1], c.inputs[2])
    s, x, y = zip(*itertools.product(range(2), range(1 << W), range(1 << W)))
    s, x, y = (np.array(v, dtype=np.uint64) for v in (s, x, y))
    np.testing.assert_array_equal(value(run_netlist(c, [s, x, y], W), r), np.where(s == 1, x, y))


def test_composite():
    """min(a + b, c) - a and lt(a + b, c) in one netlist"""
    W = 4
    c = UIntCircuit(W, 3)
    a, b, cc = c.inputs
    s = c.add(a, b)
    r1, r2 = c.sub(c.min(s, cc), a), c.lt(s, cc)
    x, y, z = zip(*itertools.product(range(16), range(16), range(16)))
    x, y, z = (np.array(v, dtype=np.uint64) for v in (x, y, z))
    wires = run_netlist(c, [x, y, z], W)
    m = np.uint64(15)
    np.testing.assert_array_equal(value(wires, r1), (np.minimum((x + y) & m, z) - x) & m)
    np.testing.assert_array_equal(value(wires, r2), (((x + y) & m) < z).astype(np.uint64))


def test_borrow_formula():
    """a*b + (a + b)*r + b + r equals (not a and b) or (not (a xor b) and r) over every (a, b, r)"""
    for a, b, r in itertools.product((0, 1), repeat=3):
        assert (a & b) ^ ((a ^ b) & r) ^ b ^ r == int((not a and b) or (not (a ^ b) and r))


@pytest.mark.parametrize("op", ["eq", "le", "ge"])
def test_not_needs_one(op):
    c = UIntCircuit(4, 2)
    with pytest.raises(ValueError, match="one"):
        BINARY[op][0](c, *c.inputs)
    with pytest.raises(ValueError, match="one"):
        UIntCircuit(4, 1).invert(c.inputs[0])


def test_shifts_add_no_gate():
    c = UIntCircuit(8, 1)
    r = c.shr(c.shl(c.inputs[0], 3), 1)
    assert c.netlist()[1] == [] and c.circuit.n_gates == 0
    a = np.arange(256, dtype=np.uint64)
    np.testing.assert_array_equal(value(run_netlist(c, [a], 8), r), ((a << np.uint64(3)) & np.uint64(255)) >> np.uint64(1))


def test_bad_arguments():
    with pytest.raises(ValueError):
        UIntCircuit(0, 1)
    with pytest.raises(ValueError):
        UIntCircuit(65, 1)
    c = UIntCircuit(4, 3)
    with pytest.raises(ValueError):
        c.select(c.inputs[0][:2], c.inputs[1], c.inputs[2])
    with pytest.raises(ValueError):
        c.shl(c.inputs[0], -1)


# -- the C++ builder emits the same netlists -------------------------------------------------------------------------
def python_netlists(W=8):
    """The text uint_netlists prints: one line per op, 'op n_inputs g0 g1 ...'."""
    lines = []
    for op in sorted(BINARY):
        c = UIntCircuit(W, 2, one=BINARY[op][2])
        r = BINARY[op][0](c, *c.inputs)
        n, g = c.netlist()
        lines.append(" ".join(map(str, [op, n] + g + ["->"] + r)))
    for op in sorted(UNARY):
        c = UIntCircuit(W, 1, one=UNARY[op][2])
        r = UNARY[op][0](c, c.inputs[0])
        n, g = c.netlist()
        lines.append(" ".join(map(str, [op, n] + g + ["->"] + r)))
    c = UIntCircuit(W, 3)
    r = c.select(c.inputs[0][:1], c.inputs[1], c.inputs[2])
    n, g = c.netlist()
    lines.append(" ".join(map(str, ["select", n] + g + ["->"] + r)))
    return lines


def test_cpp_netlists_match_python():
    exe = os.path.join(ROOT, "tests", "cpp", "bin", "uint_netlists")
    if not os.path.exists(exe):
        from csgn_b200 import build as b
        b.build_all()
    out = subprocess.run([exe, "8"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stdout + out.stderr
    got = out.stdout.strip().splitlines()
    want = python_netlists(8)
    assert [l.split()[0] for l in got] == [l.split()[0] for l in want]
    for g, w in zip(got, want):
        assert g == w, "C++ and Python netlists differ for %s" % w.split()[0]
