"""Ciphertext arrays, circuits and encrypted integers at every lane layout of their kernels.

A warp lays its 32 lanes over a block of U units; units are 16 bytes when L is even and the storage is 16-byte aligned,
8 bytes otherwise.  The grouped multiply (segments.cu seg_mul_kernel in its plain, count and write-live modes, and
circuit.cu gate_eval) takes 32 // U blocks per warp step below 32 units, with 32 - (32 // U) U idle lanes, and from 32
units on strides the lanes over one block with a ragged last step when 32 does not divide U.  Decrypt
(seg_decrypt_kernel and its bit-plane form) and cancellation (seg_cancel_insert/write_kernel, circuit.cu
cancel_in_place) use groups of G lanes, G the power of two >= U up to 32, and the whole warp probes when G = 32.

The shapes here reach every U from 1 to 33 in 16-byte units, every odd U up to 65 and the even U from 2 to 64 in 8-byte
units (views 8 bytes off alignment), and blocks of 64 to 257 units.  Each test id names its case's unit width, U, blocks
per multiply step and group width G.

Every result is compared, word for word and offset for offset, with a host reference built from the oracle and the
numpy restatements of the array suites."""
import os
import re

import numpy as np
import pytest

from oracle.pyoracle import random_key, srand, words_per_block
from test_gpu_seg_cancel import _cancelled
from test_gpu_seg_circuit import adder, multiplier
from test_gpu_seg_compact import _abi, _elements, _filtered
from test_gpu_seg_gates import _check_elements, _gate, _offsets
from test_gpu_uint import _planes_bits, _values, _words

ALIGNED = list(range(1, 67)) + [127, 128, 130, 257, 258]
MISALIGNED = [2, 4, 8, 16, 30, 32, 34, 62, 64]            # even L on 8-byte units
SHAPES = [(L, False) for L in ALIGNED] + [(L, True) for L in MISALIGNED]
N_ELEMS = 40
NETS = [adder(3), multiplier(3)]
CAPACITIES = list(range(2, 33)) + [48, 64, 96, 128, 192, 256]
# kCircuitCancelBlocks (csrc/kernels.cuh): a lane whose gate output to cancel holds more blocks falls back
with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "csgn_b200", "csrc",
                       "kernels.cuh")) as _f:
    CANCEL_BLOCKS = int(re.search(r"kCircuitCancelBlocks = (\d+);", _f.read()).group(1))


def _layout(L, off8):
    """(unit bytes, U, blocks per warp step of the multiply, group width G of decrypt and cancellation) that the
    launchers in segments.cu, capi_seg.cu and capi_circuit.cu choose for blocks of L words"""
    unit = 16 if L % 2 == 0 and not off8 else 8
    U = L * 8 // unit
    G = 1
    while G < min(U, 32):
        G *= 2
    return unit, U, 32 // U if U < 32 else 1, G


def _shape_id(shape):
    L, off8 = shape
    unit, U, per_step, G = _layout(L, off8)
    return "L%d-%s-%dB-U%d-step%d-G%d" % (L, "off8" if off8 else "aligned", unit, U, per_step, G)


def _encrypt_form(L):
    """encrypt.cu's kernel for fresh blocks of L words in a new (aligned) buffer"""
    return "warp" if L >= 64 else "units" if L % 2 == 0 else "lane"


def _setup(engine, oracle, L, seed):
    """N = 64 L - (7 L mod 64), so the pad bits vary with L (none at L = 64 and 128); D = min(16, N // 2)"""
    N = 64 * L - (7 * L) % 64
    D = min(16, N // 2)
    rng = np.random.default_rng(seed)
    s = random_key(rng, N, D)
    ctx = engine.Context(N, D)
    assert ctx.L == L
    return rng, ctx, s, oracle.key_mask(N, s), engine.SecretKey(ctx, s)


def _array(engine, ctx, elements, off8):
    """The host elements as a CiphertextArray: a fresh buffer, or with off8 a view 8 bytes off 16-byte alignment,
    which puts every kernel on 8-byte units."""
    if not off8:
        return engine.CiphertextArray.from_host(elements, ctx)
    import torch
    flat = np.concatenate(elements)
    t = torch.zeros(flat.size + 1, dtype=torch.int64, device="cuda")
    t[1:] = torch.from_numpy(flat.view(np.int64)).cuda()
    torch.cuda.synchronize()
    view = engine.Ciphertext.view(t.data_ptr() + 8, flat.size // ctx.L, ctx, keepalive=t)
    return engine.CiphertextArray(view, _offsets([e.size // ctx.L for e in elements]))


def _repeated(rng, w, L):
    """the blocks of w with about a third of them replaced by copies of other blocks of w"""
    rows = w.reshape(-1, L)
    idx = np.arange(rows.shape[0])
    dup = rng.random(idx.size) < 0.35
    idx[dup] = rng.integers(0, max(1, idx.size), size=int(dup.sum()))
    return rows[idx].reshape(-1)


def _edge_blocks(rng, N, L, bits_list):
    """one block of exactly b set bits for every b in bits_list (pad bits only when b > N)"""
    out = []
    for bits in bits_list:
        b = np.zeros(64 * L, dtype=np.uint8)
        b[rng.choice(N if bits <= N else 64 * L, size=bits, replace=False)] = 1
        out.append(np.packbits(b).view(np.uint64))
    return np.concatenate(out)


def _sizes(rng, n=N_ELEMS):
    """empty, one-block and 2-8-block elements"""
    s = rng.integers(2, 9, size=n)
    s[rng.random(n) < 0.3] = 1
    s[::7] = 0
    return s


def _operands(rng, N, D, mask):
    """Host elements of A0, B0, A1, B1 and C: blocks of every density around D, values repeated inside elements.
    Element 3 of B0 and element 10 of A1 hold more than 1024 / L blocks (a task holds 1024 words here), so decrypt and
    cancellation split them, and the compacting gate cuts the row A0_3 x B0_3 into column ranges.  Element 1 of A0 and
    B0 starts with an all-ones block, and element 5 of C holds blocks of exactly 0, 1, D - 1, D, D + 1, 64 L - 1 and
    64 L set bits: both sides of every min_bits used."""
    L = words_per_block(N)
    big = 1024 // L + 2
    sizes = [_sizes(rng) for _ in range(5)]
    sizes[0][3], sizes[1][3] = 2, big
    sizes[2][10], sizes[3][10] = big, 1
    sizes[0][1], sizes[1][1] = 2, 3
    host = [[_repeated(rng, e, L) for e in _elements(rng, sz, N, D, mask)] for sz in sizes]
    for x in host[:2]:
        x[1][:L] = ~np.uint64(0)
    host[4][5] = _edge_blocks(rng, N, L, (0, 1, D - 1, D, D + 1, 64 * L - 1, 64 * L))
    return host


def _counts(oracle, elements, N, s):
    return np.array([oracle.count_satisfied(w, N, s) if w.size else 0 for w in elements], dtype=np.uint64)


# -- the grouped multiply, compaction, cancellation and decrypt -------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=_shape_id)
def test_gates_compaction_cancellation_and_decrypt(engine, oracle, shape):
    L, off8 = shape
    rng, ctx, s, mask, key = _setup(engine, oracle, L, 8 * L + off8)
    N, D = ctx.N, ctx.D
    host = _operands(rng, N, D, mask)
    a0, b0, a1, b1, c = host
    A0, B0, A1, B1, C = (_array(engine, ctx, h, off8) for h in host)

    _check_elements(A0 * B0, _gate(oracle, L, [(a0, b0)], []))
    full = _gate(oracle, L, [(a0, b0), (a1, b1)], [c])
    G = engine.CiphertextArray.sum_of_products([(A0, B0), (A1, B1)], [C])
    _check_elements(G, full)

    for min_bits in (1, D, 64 * L):
        want = _filtered(full, L, min_bits)
        assert 0 < sum(w.size for w in want) < sum(w.size for w in full), min_bits     # some blocks kept, some dropped
        _check_elements(_abi(engine, [(A0, B0), (A1, B1)], [C], min_bits), want)

    for arr, elems in ((B0, b0), (A1, a1), (G, full)):
        want = _cancelled(elems, L)
        assert sum(w.size for w in want) < sum(w.size for w in elems)
        _check_elements(arr.cancel(), want)

    # A0 on aligned and on misaligned storage
    for arr, elems in ((A0, a0), (_array(engine, ctx, a0, not off8), a0), (B0, b0), (G, full)):
        bits, counts = key.decrypt_array(arr)
        wc = _counts(oracle, elems, N, s)
        assert wc.any()
        assert np.array_equal(counts, wc)
        assert np.array_equal(bits, (wc & 1).astype(np.uint8))


# -- circuits ---------------------------------------------------------------------------------------------------------
def _host_circuit(oracle, L, net, inputs, min_bits, cancel):
    """Every wire of the netlist over every lane (inputs: per input wire, the host elements of its lanes): per gate the
    oracle's gate, without its blocks of fewer than min_bits set bits, and with cancel its repeated blocks cancelled.
    Also the blocks of every gate before cancellation."""
    wires, pre = list(inputs), []
    for p, t in net[1]:
        w = _filtered(_gate(oracle, L, [(wires[u], wires[v]) for u, v in p], [wires[x] for x in t]), L, min_bits)
        pre.append([e.size // L for e in w])
        wires.append(_cancelled(w, L) if cancel else w)
    return wires, pre


def _value(oracle, outputs, lane, N, s):
    """the integer whose bit j is the decryption of output j of the lane (an empty element decrypts to 0)"""
    return sum((oracle.decrypt(o[lane], N, s) if o[lane].size else 0) << j for j, o in enumerate(outputs))


def _arena(net, sizes, pre, cancel, caps):
    """csgn_seg_circuit's lane arena replayed from the reference's wire sizes at every lane capacity in caps: per
    capacity and lane, whether the lane falls back to the gate-by-gate path, and whether slide_down moved one of its
    live wires.  This restates the arena policy: circuit.cu run_lane (slide the live wires down when a gate's
    uncompacted bound does not fit above the top, fall back when it still does not fit or when a gate output to cancel
    exceeds kCircuitCancelBlocks) and the free list of capi_circuit.cu (a gate wire dies after its last reader, an
    output never).  A change to that policy has to be made here too, or the fallback counts below stop matching."""
    n_in, gates, outs = net
    last = list(range(len(gates)))                     # gate wires die after their last reader, outputs never
    for g, (p, t) in enumerate(gates):
        for w in [x for pr in p for x in pr] + list(t):
            if w >= n_in:
                last[w - n_in] = g
    for w in outs:
        if w >= n_in:
            last[w - n_in] = -1
    n = len(sizes[0])
    bounds = [[sum(sizes[u][k] * sizes[v][k] for u, v in p) + sum(sizes[x][k] for x in t) for k in range(n)]
              for p, t in gates]                       # every gate's output before compaction
    out = []
    for cap in caps:
        fallback, moved = np.zeros(n, dtype=bool), np.zeros(n, dtype=bool)
        for k in range(n):
            top, at = 0, {}                            # live gate wire -> its first block in the lane's slice
            for g in range(len(gates)):
                if bounds[g][k] > cap - top:
                    top = 0
                    for w in sorted(at):
                        moved[k] |= at[w] != top
                        at[w] = top
                        top += sizes[w][k]
                    if bounds[g][k] > cap - top:
                        fallback[k] = True
                        break
                if cancel and pre[g][k] > CANCEL_BLOCKS:
                    fallback[k] = True
                    break
                at[n_in + g] = top
                top += sizes[n_in + g][k]
                for w in [w for w in at if last[w - n_in] == g]:
                    del at[w]
        out.append((fallback, moved))
    return out


def _capacities(net, sizes, pre, cancel):
    """[(lane capacity, lanes that fall back)]: the default capacity (roomy), and the capacity at which the most lanes
    slide their wires down and still fit"""
    (roomy, _), *rest = _arena(net, sizes, pre, cancel, [1 << 40] + CAPACITIES)
    i = max(range(len(rest)), key=lambda i: (rest[i][1] & ~rest[i][0]).sum())
    fallback, moved = rest[i]
    assert (moved & ~fallback).any()
    return [(0, int(roomy.sum())), (CAPACITIES[i], int(fallback.sum()))]


def _circuit_inputs(rng, N, D, mask, n_in):
    """lanes of 0-3 blocks of every density, with repeats; lane 1 of input 0 holds blocks of exactly D - 1, D and D + 1
    set bits"""
    L = words_per_block(N)
    out = []
    for _ in range(n_in):
        sz = rng.integers(0, 4, size=N_ELEMS)
        sz[rng.random(N_ELEMS) < 0.3] = 0
        out.append([_repeated(rng, e, L) for e in _elements(rng, sz, N, D, mask)])
    out[0][1] = _edge_blocks(rng, N, L, (D - 1, D, D + 1))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=_shape_id)
def test_circuits_and_integer_decrypt(engine, oracle, shape, monkeypatch):
    L, off8 = shape
    rng, ctx, s, mask, key = _setup(engine, oracle, L, 9 * L + off8)
    N, D = ctx.N, ctx.D
    for net in NETS:
        n_in, gates, outs = net
        host = _circuit_inputs(rng, N, D, mask, n_in)
        inputs = [_array(engine, ctx, h, off8) for h in host]
        circ = engine.Circuit(n_in)
        for p, t in gates:
            circ.gate(p, t)
        for min_bits in (0, D):
            for cancel in (False, True):
                wires, pre = _host_circuit(oracle, L, net, host, min_bits, cancel)
                want = [wires[w] for w in outs]
                sizes = [[e.size // L for e in w] for w in wires]
                for lane_capacity, fallback in _capacities(net, sizes, pre, cancel):
                    got = circ.evaluate(inputs, outs, min_bits=min_bits, cancel=cancel, lane_capacity=lane_capacity)
                    for g, w in zip(got, want):
                        _check_elements(g, w)
                    assert circ.last_fallback == fallback, (min_bits, cancel, lane_capacity)
                if min_bits == 0 and not cancel:                    # the largest planes, for the integer decrypt
                    planes, values = got, [_value(oracle, want, k, N, s) for k in range(N_ELEMS)]
        if L % 2 == 0 and not off8:                        # one misaligned input: 8-byte units in the circuit kernel
            inputs[0] = _array(engine, ctx, host[0], True)
            wires, _ = _host_circuit(oracle, L, net, host, D, True)
            for g, w in zip(circ.evaluate(inputs, outs, min_bits=D, cancel=True), [wires[w] for w in outs]):
                _check_elements(g, w)

        # the integer decrypt of the uncompacted outputs: planes of different sizes, with empty elements
        elems = [p.to_host() for p in planes]
        assert any(e.size == 0 for p in elems for e in p)
        assert np.array_equal(key.decrypt_uint(engine.EncryptedUInt(planes)), values)
        # elements of 4 blocks or more counted on their own and folded in by seg_uint_pack_kernel
        assert any(e.size >= 4 * L for p in elems for e in p) and any(0 < e.size < 4 * L for p in elems for e in p)
        monkeypatch.setenv("CSGN_SEG_LARGE_BYTES", str(8 * L * 4))
        assert np.array_equal(key.decrypt_uint(engine.EncryptedUInt(planes)), values)
        monkeypatch.delenv("CSGN_SEG_LARGE_BYTES")
        # the largest plane as a misaligned view: every plane on 8-byte units
        j = max(range(len(planes)), key=lambda i: planes[i].storage.n_blocks)
        mixed = list(planes)
        mixed[j] = _array(engine, ctx, elems[j], True)
        assert np.array_equal(key.decrypt_uint(engine.EncryptedUInt(mixed)), values)


# -- encrypted integers ---------------------------------------------------------------------------------------------
def _runs(n, W, most=2000):
    """block ranges of the W planes of n lanes to check against the oracle: all of them when there are at most `most`,
    else the first 256, the last 64 and the two blocks at every plane boundary (j n - 1 and j n)"""
    total = n * W
    if total <= most:
        return [(0, total)]
    return [(0, 256), (total - 64, total)] + [(j * n - 1, j * n + 1) for j in range(1, W)]


# A fresh buffer is always aligned, so the kernel depends on L alone: the shapes with misaligned views add nothing here.
@pytest.mark.gpu
@pytest.mark.parametrize("L", ALIGNED, ids=lambda L: "L%d-%s" % (L, _encrypt_form(L)))
def test_integer_encrypt_and_decrypt(engine, oracle, L):
    rng, ctx, s, mask, key = _setup(engine, oracle, L, 10 * L)
    N = ctx.N
    for W in (1, 64):
        for n in (1, 33, 1000):
            v = _values(rng, n, W)
            seed, first = 1000 * L + n, int(rng.integers(0, 1 << 40))
            x = key.encrypt_uint(v, W, seed=seed, first_block=first)
            bits = _planes_bits(v, W)
            words = _words(x)
            assert np.array_equal(words, key.encrypt_batch(bits, seed=seed, first_block=first).getValues()), (W, n)
            for a, b in _runs(n, W):
                assert np.array_equal(words[a * L:b * L], oracle.encrypt_batch(bits[a:b], N, s, seed, first + a)), \
                    (W, n, a)
                assert [oracle.count_satisfied(words[i * L:(i + 1) * L], N, s) & 1 for i in range(a, b)] == \
                    list(bits[a:b]), (W, n, a)
            assert np.array_equal(key.decrypt_uint(x), v), (W, n)


# -- without a GPU --------------------------------------------------------------------------------------------------
def test_host_circuit_reference_adds_and_multiplies(oracle):
    """The circuit reference above over fresh oracle encryptions of every pair of 3-bit operands: the adder's outputs
    decrypt to x + y and the multiplier's to x y mod 8, with and without compaction and cancellation."""
    N, D = 191, 16
    L = words_per_block(N)
    s = random_key(np.random.default_rng(5), N, D)
    srand(5)
    xs, ys = np.repeat(np.arange(8), 8), np.tile(np.arange(8), 8)
    inputs = [[oracle.encrypt(int(v >> i) & 1, N, D, s) for v in vals] for vals in (xs, ys) for i in range(3)]
    for (n_in, gates, outs), want in zip(NETS, (xs + ys, (xs * ys) % 8)):
        for min_bits, cancel in ((0, False), (0, True), (D, False), (D, True)):
            wires, _ = _host_circuit(oracle, L, (n_in, gates, outs), inputs, min_bits, cancel)
            got = [_value(oracle, [wires[w] for w in outs], k, N, s) for k in range(xs.size)]
            assert got == list(want), (len(gates), min_bits, cancel)


def test_the_shapes_reach_every_lane_layout():
    lay = [_layout(L, off8) for L, off8 in SHAPES]
    assert {U for unit, U, _, _ in lay if unit == 16} >= set(range(1, 34)) | {64, 65, 129}
    assert {U for unit, U, _, _ in lay if unit == 8} >= set(range(1, 66, 2)) | set(MISALIGNED) | {127, 257}
    for width in (8, 16):
        Us = {U for unit, U, _, _ in lay if unit == width}
        assert {G for unit, _, _, G in lay if unit == width} == {1, 2, 4, 8, 16, 32}
        assert any(U < 32 and 32 % U == 0 for U in Us)                # G U = 32: no idle lane
        assert any(U < 32 and 32 % U for U in Us)                     # idle lanes
        assert 32 in Us
        assert any(U > 32 and U % 32 == 0 for U in Us)                # strided, no ragged step
        assert any(U > 32 and U % 32 == 1 for U in Us)                # a one-lane ragged step
        assert any(16 < U < 32 for U in Us)                           # one block per step and the whole-warp probe
