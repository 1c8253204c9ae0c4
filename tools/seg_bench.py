"""Ciphertext arrays against per-ciphertext calls, on one GPU, in one run (include/csgn.h, "ciphertext arrays").

  small   n one-block products and decrypts at Context(1247,16): csgn_seg_mul / csgn_seg_decrypt against
          csgn_mul_batch / csgn_decrypt_batch on n handles -- time and kernel launches per call
  mixed   operand elements of 1-64 blocks (log-uniform), >= 1 GB of product: write rate of csgn_seg_mul next to csgn_mul of
          one product of the same size, read rate of csgn_seg_decrypt next to csgn_decrypt_count on the same storage,
          both as a fraction of a device-to-device copy (torch) of the same bytes measured in the same run
  adder   the 8-bit ripple-carry adder over 4096 lanes, end to end (encrypt, circuit, decrypt) on arrays and with
          per-element Ciphertext calls (csgn_mul_batch for the products)
  gates   the carry step C' = X*Y + T*C of a 12-bit ripple-carry adder over 4096 lanes (carry 2^i - 1 blocks per lane,
          ~2.7 GB at the last step) as three calls (csgn_seg_mul twice, csgn_seg_concat) and as one csgn_seg_mul_sum:
          time and launches per step, output bytes per second as a fraction of a device-to-device copy of the same
          bytes; then the whole 12-bit adder (circuit and decrypt) both ways
  compact the carry gate with compaction (csgn_seg_mul_sum_compact, min_bits = D: only blocks that some key could
          satisfy are kept): the 12-bit adder over 4096 lanes with plain and with compacting carry gates, the 32-bit adder
          compacted (uncompacted its last carry would hold 2^32 - 1 blocks per lane), and compact() on its own over the
          uncompacted 12-bit carry -- time, bytes written by the carry gates, and blocks held per lane after every gate
  cancel  cancellation (csgn_seg_cancel: per element, the first occurrence of every block value that occurs an odd
          number of times): cancel() on its own over 4096 elements of 100 blocks with repeated values (time, blocks
          per second, input bytes per second against a device-to-device copy), and the 6-bit multiplier (product mod
          64) over 1024 lanes, random and all-ones, with every gate compacted, with and without cancellation -- time
          and blocks per lane after every gate (without cancellation only where every gate stays under 40 GB and half
          the free device memory)
  sweep   elements whose product is 64 KB .. 64 MB, ~1 GB per call: the grouped kernel against one launch_mul per
          element (CSGN_SEG_LARGE_BYTES), which sets the large-element threshold of capi_seg.cu

Under CSGN_LIBRARY=<older libcsgn.so> (an A/B run) sections that need entry points the older build lacks are skipped.
Timing: CUDA events, recorded on the stream the library runs on, around enough calls to fill >= 1 s after a warm-up call; inputs of the mixed and sweep runs are
larger than the 126 MB L2.  Usage: python tools/seg_bench.py [--out FILE] [--quick]"""
import argparse
import ctypes
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("CSGN_TUNING", "1")      # CSGN_SEG_LARGE_BYTES is honoured only with it

import torch  # noqa: E402

from csgn_b200 import engine as eng  # noqa: E402
from oracle.pyoracle import pad_mask  # noqa: E402

LINES = []


def log(s):
    print(s, flush=True)
    LINES.append(s)


def timed(fn, min_s=1.0, min_reps=3):
    """seconds per call: one warm-up call, then enough calls for >= min_s between two CUDA events"""
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    one = max(time.perf_counter() - t0, 1e-6)
    reps = max(min_reps, int(np.ceil(min_s / one)))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps, reps


def launches(fn):
    c0 = eng.launch_count()
    fn()
    return eng.launch_count() - c0


def gpu_header():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    log("gpu: %s" % q.stdout.strip().splitlines()[0] if q.returncode == 0 else "gpu: nvidia-smi unavailable")
    log("torch %s, %s, %s" % (torch.__version__, eng.version(), os.environ.get("CSGN_LIBRARY", "libcsgn.so of this tree")))


def one_block_operands(n, ctx, rng):
    """n one-block csgn_bufs from one upload (csgn_buf_upload_batch), and the same words as one array"""
    L = ctx.L
    words = np.ascontiguousarray(rng.integers(0, 2**63, size=n * L, dtype=np.uint64))
    ub = eng.UploadBatch([words.ctypes.data + 8 * L * k for k in range(n)], [1] * n, ctx)
    handles = ub.upload()
    eng.sync()
    return words, handles


def small(ctx, key, rng, sizes):
    lib = eng._lib()
    for n in sizes:
        wa, ha = one_block_operands(n, ctx, rng)
        wb, hb = one_block_operands(n, ctx, rng)
        off = np.arange(n + 1, dtype=np.uint64)
        A = eng.CiphertextArray(eng.Ciphertext.from_host(wa, ctx), off)
        B = eng.CiphertextArray(eng.Ciphertext.from_host(wb, ctx), off)
        res = {}
        res["seg_mul"] = timed(lambda: A * B), launches(lambda: A * B)
        res["seg_decrypt"] = timed(lambda: key.decrypt_array(A)), launches(lambda: key.decrypt_array(A))

        out = (ctypes.c_void_p * n)()

        def batch_mul():
            eng.mul_batch_arrays(ha, hb, out)
            eng.free_handles(out)
        bits, counts = (ctypes.c_uint8 * n)(), (ctypes.c_uint64 * n)()

        def batch_dec():
            eng.check(lib.csgn_decrypt_batch(ha, n, key._h, bits, counts))
        res["mul_batch"] = timed(batch_mul), launches(batch_mul)
        res["decrypt_batch"] = timed(batch_dec), launches(batch_dec)
        for k, ((t, reps), nl) in res.items():
            log("small n=%-6d %-14s %10.1f us/call  %6d launches/call  (%d calls)" % (n, k, t * 1e6, nl, reps))
        log("small n=%-6d speed-up: multiply %.1fx, decrypt %.1fx" % (
            n, res["mul_batch"][0][0] / res["seg_mul"][0][0], res["decrypt_batch"][0][0] / res["seg_decrypt"][0][0]))
        eng.free_handles(ha)
        eng.free_handles(hb)


def copy_rate(nbytes):
    src = torch.empty(nbytes // 8, dtype=torch.int64, device="cuda")
    dst = torch.empty_like(src)
    t, _ = timed(lambda: dst.copy_(src))
    del src, dst
    torch.cuda.empty_cache()
    return nbytes / t


def log_uniform_sizes(rng, n, hi=64):
    return np.minimum(hi, np.floor(np.exp(rng.uniform(0, np.log(hi + 1), n)))).astype(np.int64)


def mixed(ctx, key, rng, target_bytes):
    L = ctx.L
    n = 1024
    while True:
        t1, t2 = log_uniform_sizes(rng, n), log_uniform_sizes(rng, n)
        if int((t1 * t2).sum()) * L * 8 >= target_bytes:
            break
        n *= 2
    prod_blocks = int((t1 * t2).sum())
    pbytes = prod_blocks * L * 8
    a = torch.randint(-2**62, 2**62, (int(t1.sum()) * L,), dtype=torch.int64, device="cuda")
    b = torch.randint(-2**62, 2**62, (int(t2.sum()) * L,), dtype=torch.int64, device="cuda")
    A = eng.CiphertextArray(eng.Ciphertext.from_tensor(a, ctx), np.concatenate([[0], np.cumsum(t1)]))
    B = eng.CiphertextArray(eng.Ciphertext.from_tensor(b, ctx), np.concatenate([[0], np.cumsum(t2)]))
    log("mixed: %d elements, operand blocks 1-64 log-uniform, product %d blocks = %.2f GB" % (n, prod_blocks, pbytes / 1e9))
    cp = copy_rate(pbytes)
    log("mixed: device-to-device copy of %.2f GB: %.0f GB/s (bytes copied per second)" % (pbytes / 1e9, cp / 1e9))
    keep = []

    def seg_mul():
        keep[:] = [A * B]
    t_seg, _ = timed(seg_mul)
    keep.clear()
    # one product of the same size
    s1 = int(np.sqrt(prod_blocks))
    s2 = (prod_blocks + s1 - 1) // s1
    x = eng.Ciphertext.from_tensor(torch.randint(-2**62, 2**62, (s1 * L,), dtype=torch.int64, device="cuda"), ctx)
    y = eng.Ciphertext.from_tensor(torch.randint(-2**62, 2**62, (s2 * L,), dtype=torch.int64, device="cuda"), ctx)
    one = []

    def one_mul():
        one[:] = [x * y]
    t_one, _ = timed(one_mul)
    one_bytes = s1 * s2 * L * 8
    r_seg, r_one = pbytes / t_seg, one_bytes / t_one
    log("mixed: seg_mul  %8.2f ms  %6.0f GB/s written  %.2f of copy | csgn_mul %dx%d %8.2f ms  %6.0f GB/s  %.2f of copy"
        " | seg / single %.2f" % (t_seg * 1e3, r_seg / 1e9, r_seg / cp, s1, s2, t_one * 1e3, r_one / 1e9, r_one / cp,
                                  r_seg / r_one))
    one.clear()
    P = A * B
    counts = torch.zeros(n, dtype=torch.int64, device="cuda")
    t_sd, _ = timed(lambda: key.decrypt_array_count_async(P, counts.data_ptr()))
    total = torch.zeros(1, dtype=torch.int64, device="cuda")
    t_d, _ = timed(lambda: key.count_satisfied_async(P.storage, total.data_ptr()))
    r_sd, r_d = pbytes / t_sd, pbytes / t_d
    log("mixed: seg_decrypt %8.2f ms  %6.0f GB/s read  %.2f of copy | csgn_decrypt_count same storage %8.2f ms  %6.0f GB/s"
        "  %.2f of copy | seg / single %.2f" % (t_sd * 1e3, r_sd / 1e9, r_sd / cp, t_d * 1e3, r_d / 1e9, r_d / cp,
                                                 r_sd / r_d))
    del P, A, B, a, b, x, y
    torch.cuda.empty_cache()


def adder(ctx, key, rng, lanes):
    xb, yb = rng.integers(0, 256, lanes), rng.integers(0, 256, lanes)
    bits = np.concatenate([np.concatenate([(xb >> i) & 1 for i in range(8)]),
                           np.concatenate([(yb >> i) & 1 for i in range(8)])]).astype(np.uint8)

    def on_arrays():
        allb = key.encrypt_array(bits, seed=5)
        row = lambda r: allb.gather(np.arange(r * lanes, (r + 1) * lanes))    # noqa: E731
        X, Y = row(0), row(8)
        S, C = [X + Y], X * Y
        for i in range(1, 8):
            X, Y = row(i), row(8 + i)
            T = X + Y
            S.append(T + C)
            C = X * Y + T * C
        out = [key.decrypt_array(s)[0] for s in S] + [key.decrypt_array(C)[0]]
        return out

    def per_element():
        allb = key.encrypt_array(bits, seed=5)
        el = [allb.element(k) for k in range(16 * lanes)]
        x = [el[i * lanes:(i + 1) * lanes] for i in range(8)]
        y = [el[(8 + i) * lanes:(9 + i) * lanes] for i in range(8)]
        S = [[a + b for a, b in zip(x[0], y[0])]]
        C = eng.mul_batch(x[0], y[0])
        for i in range(1, 8):
            T = [a + b for a, b in zip(x[i], y[i])]
            S.append([t + c for t, c in zip(T, C)])
            XY, TC = eng.mul_batch(x[i], y[i]), eng.mul_batch(T, C)
            C = [p + q for p, q in zip(XY, TC)]
        return [np.array(key.decrypt_batch(s)[0], dtype=np.uint8) for s in S] + [np.array(key.decrypt_batch(C)[0], np.uint8)]

    got = on_arrays()
    val = sum(got[i].astype(np.int64) << i for i in range(8))
    assert np.array_equal(val, (xb + yb) % 256) and np.array_equal(got[8], (xb + yb) >> 8), "adder on arrays is wrong"
    ref = per_element()
    assert all(np.array_equal(p, q) for p, q in zip(got, ref)), "the two adders disagree"
    t_arr, r1 = timed(on_arrays, min_s=2.0, min_reps=2)
    l_arr = launches(on_arrays)
    t_el, r2 = timed(per_element, min_s=2.0, min_reps=2)
    l_el = launches(per_element)
    log("adder: 8-bit, %d lanes, Context(%d,%d): arrays %8.2f ms (%d launches) | per-element calls %8.2f ms (%d launches)"
        " | speed-up %.1fx" % (lanes, ctx.N, ctx.D, t_arr * 1e3, l_arr, t_el * 1e3, l_el, t_el / t_arr))


def gates(ctx, key, rng, lanes, bits):
    SP = eng.CiphertextArray.sum_of_products
    xb, yb = rng.integers(0, 1 << bits, lanes), rng.integers(0, 1 << bits, lanes)
    plain = np.concatenate([np.concatenate([(v >> i) & 1 for i in range(bits)]) for v in (xb, yb)]).astype(np.uint8)
    allb = key.encrypt_array(plain, seed=7)
    rows = [allb.gather(np.arange(r * lanes, (r + 1) * lanes)) for r in range(2 * bits)]
    T = [rows[i] + rows[bits + i] for i in range(bits)]

    def adder(one_call):
        C = rows[0] * rows[bits]
        S = [T[0]]
        for i in range(1, bits):
            S.append(T[i] + C)
            C = SP([(rows[i], rows[bits + i]), (T[i], C)]) if one_call else rows[i] * rows[bits + i] + T[i] * C
        return S, C

    def decrypted(S, C):
        return [key.decrypt_array(s)[0] for s in S] + [key.decrypt_array(C)[0]]

    S3, C3 = adder(False)
    S1, C1 = adder(True)
    assert np.array_equal(C1.offsets, C3.offsets), "carry offsets differ"
    assert C1.storage.checksum() == C3.storage.checksum(), "carry words differ"
    got = decrypted(S1, C1)
    assert all(np.array_equal(p, q) for p, q in zip(decrypted(S3, C3), got)), "the two adders disagree"
    val = sum(got[i].astype(np.int64) << i for i in range(bits))
    assert np.array_equal(val, (xb + yb) % (1 << bits)) and np.array_equal(got[bits], (xb + yb) >> bits), "adder wrong"
    # the last carry step: C' = X*Y + T*C with the carry of bit bits-2
    C = rows[0] * rows[bits]
    for i in range(1, bits - 1):
        C = SP([(rows[i], rows[bits + i]), (T[i], C)])
    X, Y, Tl = rows[bits - 1], rows[2 * bits - 1], T[bits - 1]
    out_bytes = C1.storage.n_blocks * ctx.L * 8
    del S3, C3, S1
    torch.cuda.empty_cache()
    cp = copy_rate(out_bytes)
    keep = []

    def three():
        keep[:] = [X * Y + Tl * C]

    def one():
        keep[:] = [SP([(X, Y), (Tl, C)])]
    assert SP([(X, Y), (Tl, C)]).storage.checksum() == C1.storage.checksum()
    del C1
    res = {}
    for name, fn in (("three calls", three), ("one call", one), ("three calls", three), ("one call", one)):
        t, _ = timed(fn)
        res.setdefault(name, []).append(t)
        res[name + " launches"] = launches(fn)
        keep.clear()
    log("gates: carry step %d of a %d-bit adder, %d lanes, Context(%d,%d): carry in %d -> out %d blocks per lane, "
        "output %.2f GB; device-to-device copy of the same bytes %.0f GB/s" % (
            bits - 1, bits, lanes, ctx.N, ctx.D, (1 << (bits - 1)) - 1, (1 << bits) - 1, out_bytes / 1e9, cp / 1e9))
    for name in ("three calls", "one call"):
        t = min(res[name])
        log("gates: carry step, %-11s %8.3f ms (runs %s)  %d launches  %6.0f GB/s of output  %.2f of copy" % (
            name, t * 1e3, " / ".join("%.3f" % (x * 1e3) for x in res[name]), res[name + " launches"],
            out_bytes / t / 1e9, out_bytes / t / cp))
    log("gates: carry step, three calls / one call %.2fx" % (min(res["three calls"]) / min(res["one call"])))
    del C
    torch.cuda.empty_cache()
    whole = {}
    for name, flag in (("three calls", False), ("one call", True), ("three calls", False), ("one call", True)):
        def run():
            decrypted(*adder(flag))
        t, _ = timed(run, min_s=2.0, min_reps=2)
        whole.setdefault(name, []).append(t)
        whole[name + " launches"] = launches(run)
        torch.cuda.empty_cache()
    log("gates: whole %d-bit adder (circuit + decrypt of %d arrays), %d lanes: three-call carries %8.2f ms (%d launches) | "
        "one-call carries %8.2f ms (%d launches) | %.2fx" % (
            bits, bits + 1, lanes, min(whole["three calls"]) * 1e3, whole["three calls launches"],
            min(whole["one call"]) * 1e3, whole["one call launches"], min(whole["three calls"]) / min(whole["one call"])))


def compact_adder(ctx, key, rng, lanes, bits, compact):
    """-> (run, check): run() computes the carries of a `bits`-bit adder over `lanes` lanes (carry gates compacting or
    not) and returns (sum arrays, last carry, blocks per lane after every carry gate, bytes the carry gates wrote)"""
    SP = eng.CiphertextArray.sum_of_products
    xb, yb = rng.integers(0, 1 << bits, lanes), rng.integers(0, 1 << bits, lanes)
    plain = np.concatenate([np.concatenate([(v >> i) & 1 for i in range(bits)]) for v in (xb, yb)]).astype(np.uint8)
    allb = key.encrypt_array(plain, seed=11)
    rows = [allb.gather(np.arange(r * lanes, (r + 1) * lanes)) for r in range(2 * bits)]
    T = [rows[i] + rows[bits + i] for i in range(bits)]
    word_bytes = ctx.L * 8

    def run():
        C = SP([(rows[0], rows[bits])], compact=compact)
        S, held, written = [T[0]], [C.storage.n_blocks / lanes], C.storage.n_blocks * word_bytes
        for i in range(1, bits):
            S.append(T[i] + C)
            C = SP([(rows[i], rows[bits + i]), (T[i], C)], compact=compact)
            held.append(C.storage.n_blocks / lanes)
            written += C.storage.n_blocks * word_bytes
        return S, C, held, written

    def check(S, C):
        got = [key.decrypt_array(x)[0] for x in S] + [key.decrypt_array(C)[0]]
        val = sum(got[i].astype(np.int64) << i for i in range(bits))
        assert np.array_equal(val, (xb + yb) % (1 << bits)) and np.array_equal(got[bits], (xb + yb) >> bits), \
            "%d-bit adder wrong" % bits
    return run, check


def compaction(ctx, key, rng, lanes):
    keep = []
    for bits, modes in ((12, (False, True)), (32, (True,))):
        for compact in modes:
            run, check = compact_adder(ctx, key, np.random.default_rng(bits), lanes, bits, compact)
            S, C, held, written = run()
            check(S, C)
            del S, C
            torch.cuda.empty_cache()

            def carries():
                keep[:] = [run()]
            t, reps = timed(carries, min_s=2.0, min_reps=2)
            keep.clear()
            torch.cuda.empty_cache()
            log("compact: %d-bit adder carries, %d lanes, Context(%d,%d), %s: %8.2f ms (%d runs)  %.3f GB written by "
                "the carry gates" % (bits, lanes, ctx.N, ctx.D, "compacting gates" if compact else "plain gates   ",
                                     t * 1e3, reps, written / 1e9))
            log("compact: %d-bit %s blocks per lane after each carry gate: %s" % (
                bits, "compacted" if compact else "plain    ", " ".join("%.1f" % h for h in held)))
    # compact() on its own over the uncompacted 12-bit carry
    run, _ = compact_adder(ctx, key, np.random.default_rng(12), lanes, 12, False)
    _, C, _, _ = run()
    small = C.compact()

    def compact_once():
        keep[:] = [C.compact()]
    t, reps = timed(compact_once)
    keep.clear()
    log("compact: compact() of the uncompacted 12-bit carry (%.2f GB, %.1f blocks per lane) -> %.1f blocks per lane: "
        "%8.3f ms (%d calls)  %.3f GB written  %.0f GB/s read" % (
            C.storage.n_blocks * ctx.L * 8 / 1e9, C.storage.n_blocks / lanes, small.storage.n_blocks / lanes, t * 1e3,
            reps, small.storage.n_blocks * ctx.L * 8 / 1e9, C.storage.n_blocks * ctx.L * 8 / t / 1e9))
    del C, small
    torch.cuda.empty_cache()


class TooLarge(Exception):
    pass


def multiplier(X, Y, gate):
    """Product mod 2^n of the bit arrays X[i], Y[i]: schoolbook rows, ripple-carry adds, every sum and carry one
    gate(products, terms); None is an all-zero bit"""
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


def cancellation(ctx, key, rng, n_elems, lanes, bits, budget_bytes):
    L = ctx.L
    # cancel() alone: about 100 blocks per element drawn from 70 values each, so most values repeat
    per, vals_per = 100, 70
    vals = torch.randint(-2**62, 2**62, (n_elems, vals_per, L), dtype=torch.int64, device="cuda")
    idx = torch.randint(0, vals_per, (n_elems, per), device="cuda")
    vals[:, :, L - 1] &= int(np.int64(np.uint64(pad_mask(ctx.N))))           # pad bits zero, as the library leaves them
    words = torch.gather(vals, 1, idx.unsqueeze(-1).expand(-1, -1, L)).reshape(-1).contiguous()
    X = eng.CiphertextArray(eng.Ciphertext.from_tensor(words, ctx), np.arange(n_elems + 1, dtype=np.uint64) * per)
    blocks, nbytes = n_elems * per, n_elems * per * L * 8
    cp = copy_rate(nbytes)
    keep = []

    def once():
        keep[:] = [X.cancel()]
    t, reps = timed(once)
    kept = keep[0].storage.n_blocks
    nl = launches(once)
    keep.clear()
    log("cancel: cancel() of %d elements x %d blocks (%d values each), Context(%d,%d), %.1f MB in (less than the 126 MB "
        "L2: repeated calls may read it from there): "
        "%8.3f ms (%d calls, %d launches)  %.0f M blocks/s  %.0f GB/s of input  %.2f of a device copy of the same bytes "
        "(%.0f GB/s)  %d of %d blocks kept" % (n_elems, per, vals_per, ctx.N, ctx.D, nbytes / 1e6, t * 1e3, reps, nl,
                                             blocks / t / 1e6, nbytes / t / 1e9, nbytes / t / cp, cp / 1e9, kept,
                                             blocks))
    del X, vals, idx, words
    torch.cuda.empty_cache()

    # the n-bit multiplier over `lanes` lanes, every gate compacted, with and without cancellation
    SP = eng.CiphertextArray.sum_of_products
    for lanes_kind in ("random", "all-ones"):
        r = np.random.default_rng(bits)
        if lanes_kind == "random":
            xb, yb = r.integers(0, 1 << bits, lanes), r.integers(0, 1 << bits, lanes)
        else:
            xb = yb = np.full(lanes, (1 << bits) - 1)
        plain = np.concatenate([np.concatenate([(v >> i) & 1 for i in range(bits)]) for v in (xb, yb)]).astype(np.uint8)
        allb = key.encrypt_array(plain, seed=13)
        rows = [allb.gather(np.arange(q * lanes, (q + 1) * lanes)) for q in range(2 * bits)]
        for cancel in (True, False):
            held = []

            def gate(products, terms):
                out = sum(int(np.dot(np.diff(a.offsets.astype(np.int64)), np.diff(b.offsets.astype(np.int64))))
                          for a, b in products) + sum(int(c.offsets[-1]) for c in terms)
                # the gate's product blocks, and the result before compaction in the worst case, next to what is held
                limit = min(budget_bytes, eng.device_info()["hbm_free"] // 2)
                if out * L * 8 > limit:
                    raise TooLarge("a gate of %.1f GB before compaction, %.1f GB allowed" % (out * L * 8 / 1e9,
                                                                                          limit / 1e9))
                g = SP(products, terms, compact=True)
                if cancel:
                    g = g.cancel()
                held.append(g.storage.n_blocks / lanes)
                return g

            def run():
                held.clear()
                return multiplier(rows[:bits], rows[bits:], gate)
            name = "compact + cancel" if cancel else "compact alone   "
            try:
                P = run()
            except TooLarge as e:
                log("cancel: %d-bit multiplier, %d %s lanes, %s: does not fit (%s)" % (bits, lanes, lanes_kind, name, e))
                torch.cuda.empty_cache()
                continue
            got = sum(key.decrypt_array(P[i])[0].astype(np.int64) << i for i in range(bits))
            assert np.array_equal(got, (xb * yb) % (1 << bits)), "%d-bit multiplier wrong" % bits
            out_bits = [P[i].storage.n_blocks / lanes for i in range(bits)]
            del P
            torch.cuda.empty_cache()

            def circuit():
                keep[:] = [run()]
            t, reps = timed(circuit, min_s=2.0, min_reps=2)
            keep.clear()
            torch.cuda.empty_cache()
            log("cancel: %d-bit multiplier (product mod 2^%d), %d %s lanes, Context(%d,%d), %s: %8.2f ms (%d runs), "
                "%d gates, at most %.1f blocks per lane after a gate; output bits %s blocks per lane" % (
                    bits, bits, lanes, lanes_kind, ctx.N, ctx.D, name, t * 1e3, reps, len(held), max(held),
                    " ".join("%.1f" % h for h in out_bits)))
            log("cancel: %d-bit %s lanes, %s, blocks per lane after each gate: %s" % (
                bits, lanes_kind, name.strip(), " ".join("%.1f" % h for h in held)))


def sweep(ctx, total_bytes, sizes_kb):
    L = ctx.L
    for kb in sizes_kb:
        t = max(1, int(round(np.sqrt(kb * 1024 / (8 * L)))))
        pbytes = t * t * L * 8
        n = max(1, total_bytes // pbytes)
        a = torch.randint(-2**62, 2**62, (n * t * L,), dtype=torch.int64, device="cuda")
        off = np.arange(n + 1, dtype=np.uint64) * t
        A = eng.CiphertextArray(eng.Ciphertext.from_tensor(a, ctx), off)
        keep = []
        res = {}
        for mode, knob in (("grouped", str(1 << 50)), ("per-element", "0")):
            os.environ["CSGN_SEG_LARGE_BYTES"] = knob

            def run():
                keep[:] = [A * A]
            tt, _ = timed(run)
            res[mode] = (tt, launches(run))
            keep.clear()
        os.environ.pop("CSGN_SEG_LARGE_BYTES", None)
        g, p = res["grouped"], res["per-element"]
        log("sweep: product %6.0f KB (%4dx%-4d blocks) x %5d elements = %.2f GB: grouped %7.0f GB/s (%d launches) | "
            "per-element launch_mul %7.0f GB/s (%d launches) | grouped / per-element %.2f" % (
                pbytes / 1024, t, t, n, n * pbytes / 1e9, n * pbytes / g[0] / 1e9, g[1], n * pbytes / p[0] / 1e9, p[1],
                p[0] / g[0]))
        del A, a
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--quick", action="store_true", help="small sizes (a check of the script, not a measurement)")
    ap.add_argument("--only", default="small,mixed,adder,gates,compact,cancel,sweep")
    args = ap.parse_args()
    torch.cuda.set_device(0)
    eng.init(0)
    # One NON-default torch stream for the library's work, torch's copies and the timing events.  (torch's default
    # stream has the handle 0, and csgn_set_stream(0) selects the library's own non-blocking stream, which events
    # recorded on torch's default stream would not wait for.)
    st = torch.cuda.Stream()
    torch.cuda.set_stream(st)
    eng.set_stream(st.cuda_stream)
    gpu_header()
    rng = np.random.default_rng(1)
    ctx = eng.Context(1247, 16)
    key = eng.SecretKey(ctx, rng.permutation(1247)[:16].astype(np.uint64))
    only = args.only.split(",")
    if "small" in only:
        small(ctx, key, rng, [100, 1000] if args.quick else [1000, 10000, 100000])
    if "mixed" in only:
        mixed(ctx, key, rng, (64 << 20) if args.quick else (1 << 30))
    if "adder" in only:
        adder(ctx, key, rng, 256 if args.quick else 4096)
    if "gates" in only:
        if hasattr(eng._lib(), "csgn_seg_mul_sum"):
            gates(ctx, key, rng, 256 if args.quick else 4096, 8 if args.quick else 12)
        else:
            log("gates: skipped, %s has no csgn_seg_mul_sum" % os.environ.get("CSGN_LIBRARY", "this build"))
    if "compact" in only:
        if hasattr(eng._lib(), "csgn_seg_mul_sum_compact"):
            compaction(ctx, key, rng, 256 if args.quick else 4096)
        else:
            log("compact: skipped, %s has no csgn_seg_mul_sum_compact" % os.environ.get("CSGN_LIBRARY", "this build"))
    if "cancel" in only:
        if hasattr(eng._lib(), "csgn_seg_cancel"):
            cancellation(ctx, key, rng, 256 if args.quick else 4096, 128 if args.quick else 1024, 4 if args.quick else 6,
                         40 << 30)
        else:
            log("cancel: skipped, %s has no csgn_seg_cancel" % os.environ.get("CSGN_LIBRARY", "this build"))
    if "sweep" in only:
        sweep(ctx, (64 << 20) if args.quick else (1 << 30),
              [64, 256] if args.quick else [64, 256, 1024, 4096, 16384, 65536])
    eng.set_stream(0)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
