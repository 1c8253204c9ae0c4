"""Encrypted integers on one GPU, in one run (include/csgn.h, "encrypted integers"), at Context(1247,16) over 4096 and
65536 lanes:

  encrypt  csgn_encrypt_uint of 32-bit values (one launch, no host synchronisation) against 32 encrypt_array calls, one
           per bit plane (csgn_encrypt_batch, one launch and one host synchronisation each)
  decrypt  csgn_decrypt_uint of the 32 planes (one launch, one synchronisation) against 32 decrypt_array calls and the
           assembly of the bits on the host
  e2e      encrypt_uint of the operands -> one UIntCircuit.evaluate (compacted and cancelled) -> decrypt_uint, for the
           32-bit add, the 8-bit min (lt + select) and the 8-bit mul: time, lanes per second, kernel launches per call.
           A cancelled result holds the monomials of its algebraic normal form, which for comparisons and products grow
           about threefold per bit (3^W - 1 for lt), so min and mul run at 8 bits; add stays small at any width

The two arms of a comparison alternate call by call in the same run and each reports its median; every timed call ends
in a device synchronisation (host clock).  Every result is checked against numpy before it is timed.
Usage: python tools/uint_bench.py [--out FILE] [--quick]"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from csgn_b200 import engine as eng  # noqa: E402
from oracle.pyoracle import random_key  # noqa: E402

LINES = []


def log(s):
    print(s, flush=True)
    LINES.append(s)


def gpu_header():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    log("gpu (name, power limit, SM clock, max SM clock): %s" % (q.stdout.strip().splitlines()[0] if q.returncode == 0
                                                                 else "nvidia-smi unavailable"))
    log("torch %s, %s" % (torch.__version__, eng.version()))


def call_s(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def launches(fn):
    c0 = eng.launch_count()
    fn()
    return eng.launch_count() - c0


def alternate(arms, reps, budget_s):
    """median seconds per call of every arm, the arms called in turn after one warm-up call each"""
    for fn in arms:
        fn()
    times = [[] for _ in arms]
    t_end = time.perf_counter() + budget_s
    r = 0
    while r < reps or (r < 3 * reps and time.perf_counter() < t_end):
        for i, fn in enumerate(arms):
            times[i].append(call_s(fn))
        r += 1
    return [float(np.median(t)) for t in times], r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true")
    args = ap.parse_args()
    eng.init(0)
    gpu_header()
    N, D = 1247, 16
    rng = np.random.default_rng(2026)
    ctx = eng.Context(N, D)
    key = eng.SecretKey(ctx, random_key(rng, N, D))
    reps = 3 if args.quick else 10
    budget = 2.0 if args.quick else 10.0
    for n in ([4096] if args.quick else [4096, 65536]):
        log("")
        log("== %d lanes ==" % n)
        W = 32
        v = rng.integers(0, 1 << W, size=n, dtype=np.uint64)
        planes = [((v >> np.uint64(j)) & np.uint64(1)).astype(np.uint8) for j in range(W)]

        def enc_uint():
            return key.encrypt_uint(v, W, seed=1)

        def enc_planes():
            return [key.encrypt_array(planes[j], seed=1, first_block=j * n) for j in range(W)]

        x = enc_uint()
        assert np.array_equal(key.decrypt_uint(x), v)
        assert all(np.array_equal(a.storage.getValues(), p.storage.getValues()) for a, p in zip(x.planes, enc_planes()))
        (t_u, t_p), r = alternate([enc_uint, enc_planes], reps, budget)
        log("encrypt %d-bit: encrypt_uint %.3f ms (%d launch), 32 x encrypt_array %.3f ms (%d launches, 32 host "
            "synchronisations): %.2fx  [%d alternations]"
            % (W, t_u * 1e3, launches(enc_uint), t_p * 1e3, launches(enc_planes), t_p / t_u, r))

        def dec_uint():
            return key.decrypt_uint(x)

        def dec_planes():
            out = np.zeros(n, dtype=np.uint64)
            for j, p in enumerate(x.planes):
                out |= key.decrypt_array(p)[0].astype(np.uint64) << np.uint64(j)
            return out

        assert np.array_equal(dec_uint(), v) and np.array_equal(dec_planes(), v)
        (t_u, t_p), r = alternate([dec_uint, dec_planes], reps, budget)
        log("decrypt %d-bit: decrypt_uint %.3f ms (%d launch), 32 x decrypt_array + host assembly %.3f ms (%d launches, "
            "32 host synchronisations): %.2fx  [%d alternations]"
            % (W, t_u * 1e3, launches(dec_uint), t_p * 1e3, launches(dec_planes), t_p / t_u, r))

        for name, W, ref in [("add", 32, lambda a, b, m: (a + b) & m), ("min", 8, lambda a, b, m: np.minimum(a, b)),
                             ("mul", 8, lambda a, b, m: (a * b) & m)]:
            a = rng.integers(0, 1 << W, size=n, dtype=np.uint64)
            b = rng.integers(0, 1 << W, size=n, dtype=np.uint64)
            c = eng.UIntCircuit(W, 2)
            res = getattr(c, name)(*c.inputs)
            fallback = []

            def e2e():
                A, B = key.encrypt_uint(a, W, seed=2), key.encrypt_uint(b, W, seed=3, first_block=n * W)
                (r_,) = c.evaluate([A, B], [res], cancel=True)
                fallback.append(c.last_fallback)
                return key.decrypt_uint(r_)

            try:
                got = e2e()
            except eng.CsgnError as err:
                log("e2e %s %d-bit: does not fit (%s)" % (name, W, err))
                continue
            assert np.array_equal(got, ref(a, b, np.uint64((1 << W) - 1))), name
            (t,), r = alternate([e2e], max(3, reps // 2), budget)
            log("e2e %s %d-bit (%d gates, compacted and cancelled): %.3f ms, %.3g lanes/s, %d launches per call, "
                "%d fallback lanes  [%d calls]"
                % (name, W, c.circuit.n_gates, t * 1e3, n / t, launches(e2e), max(fallback), r))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
