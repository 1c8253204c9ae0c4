#!/usr/bin/env python
"""bench.py -- the headline measurement of BASELINE.json on B200.

Metric: output blocks/s of the ciphertext hot path -- multiply (all-pairs AND of T1 x T2 blocks) followed by
decrypt of the product -- at Context(1247,16), 1000 x 1000 -> 1,000,000 output blocks per ciphertext pair
(BASELINE.json configs[1]).

A step is one pass over a batch of `pairs` independent ciphertext pairs.  For every pair the product is WRITTEN to
HBM (the caller keeps it) and decrypted:
  --mode fused (default)   one kernel per pair writes the product and evaluates the decrypt predicate on the product
                           words while they are in registers (csgn_mul_count_batch_async): one pass over HBM;
  --mode two-pass          [multiply pair 0..P-1] then [decrypt product 0..P-1] (csgn_mul_into_batch +
                           csgn_decrypt_count_batch_async): every product is written and, P-1 products later, read
                           back.  Always measured as well and reported under "two_pass".
Either way a step moves P x 160 MB of products (far more than the 126 MB L2): the kernels run against HBM.

  value          device-resident operands and outputs, no host traffic in the timed region
  e2e            the same batch through the public C ABI from pinned HOST operands: csgn_buf_upload x 2P ->
                 csgn_mul_count_batch_async (products allocated by the library) -> one D2H of the P counts per step,
                 read and checked on the host every step
  e2e_cpp        the same through the certFHE C++ drop-in API (tools/cpp_e2e.cpp): Ciphertext(V,Bitlen,len,ctx) from
                 host arrays -> operator* -> SecretKey::decrypt, a plain loop over the pairs
  roofline       the dominant kernel: 160 B written per output block / its CUDA-event time, against MEASURED_PEAKS.json
  two_pass       the round-1 definition of the step (separate multiply and decrypt kernels) on the same buffers
  sustained      the same step loop run for >= 3 s: value, SM clock, board power, throttle reasons under sustained load
  other_workloads  BASELINE.json configs[3], [4]: the 10^6 x 125 chain product (20 GB per GPU; 10^9 blocks at 8 GPUs)
                 and Context(16383,64) at 300x300 and 2000x2000, each kernel against the same roofline
  other_kernels  permute and add on the products the bench holds
  precheck       before anything is timed: a small sharded multiply / fused multiply->decrypt / decrypt / permute
                 compared WORD FOR WORD with a numpy restatement written here (no import from oracle/), on every rank
  cpu_baseline   the unmodified reference (oracle/_ref) or the oracle port, 1 thread, on the full 1000x1000 pair

Every count the timed loops produce is compared with the host-known truth: the satisfied blocks of each operand are
counted in numpy from the host copies, and count(a*b) = sum over ranks of count(a_shard) * count(b).

N > 1 (torchrun, one process per GPU): weak scaling.  The left operand of every pair has 1000*N blocks and is
sharded by contiguous block range (csgn_shard_range); the right operand is replicated; every rank multiplies and
folds its own 1M-block shard.  The per-pair satisfied-block counts are summed ACROSS GPUs BY THE KERNEL ITSELF: its
last CTA stores the count into every rank's mailbox over NVLink and the launch closing the batch collects the sums
(csrc/peer.cuh) -- no NCCL call in the step.  `--exchange nccl` keeps the separate all-reduce it replaces.

`--impl reference` times the reference's own CPU implementation (public operator* and SecretKey::decrypt) on the
host cores, one replica thread per core, each on the full 1000 x 1000 pair.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (N, D, T1, T2, description)
    "cfg2": (1247, 16, 1000, 1000, "Context(1247,16): 1000x1000 -> 1M output blocks, multiply then decrypt"),
    "cfg5": (16383, 64, 300, 300, "Context(16383,64): 300x300 -> 90k output blocks, multiply then decrypt"),
    # BASELINE.json configs[3]: deep product chain (a*b)*d; per GPU 1000 x 1000 x chain_d blocks, the left
    # operand sharded by block range, b and d replicated, decrypt finished by a one-word exchange.
    # chain_d = 125 gives 1.25e8 blocks = 20 GB per GPU, 1e9 blocks at 8 GPUs.
    "cfg4": (1247, 16, 1000, 1000, "Context(1247,16): chain (a*b)*d, 1000 x 1000 x chain_d blocks per GPU, decrypt + exchange"),
}
METRIC = "ctxt-mul+decrypt output blocks/s"
UNIT = "blocks/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", default="fused", choices=["fused", "two-pass"],
                    help="fused: one kernel per pair writes the product and folds it (default); two-pass: multiply, then decrypt")
    ap.add_argument("--pairs", type=int, default=16, help="independent ciphertext pairs per step")
    ap.add_argument("--chain-d", type=int, default=125, help="cfg4: blocks of the third operand (125 -> 20 GB/GPU)")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N>1: decrypt's cross-GPU sum inside the fold kernel over NVLink mailboxes (peer) "
                         "or as a separate NCCL all-reduce (nccl, the baseline it replaces)")
    ap.add_argument("--collect", default="lagged", choices=["lagged", "same-step"],
                    help="peer exchange: the launch closing step k collects step k-1's sums (never waits for a slower "
                         "rank; the last step's sums are collected before the timed region ends) or its own step's")
    ap.add_argument("--t1", type=int, default=0, help="blocks of the left operand (overrides the workload's; with --scaling "
                                                      "strong: of the WHOLE left operand, sharded over the ranks)")
    ap.add_argument("--t2", type=int, default=0, help="blocks of the right operand (overrides the workload's)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N>1: weak = every rank multiplies t1 x t2 (default, the headline); strong = the t1 blocks of the "
                         "left operand are split over the ranks (SURVEY 8d, the cfg5 sweep)")
    ap.add_argument("--sustain-s", type=float, default=3.0, help="seconds of the sustained run (0: skip)")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the side measurements: other_kernels, other_workloads, two_pass, sustained, e2e_cpp")
    ap.add_argument("--no-other-workloads", action="store_true")
    ap.add_argument("--no-precheck", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned to DIR/<name>.npy (float64): "
                         "counts (satisfied blocks per pair), product_blocks (a fixed, seeded sample of block indices of "
                         "the products, pair-major) and product_words (those blocks' words, [..., 0] = high and [..., 1] = "
                         "low 32 bits); one file set per rank, suffixed _rank<r>, when N > 1")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path (--impl ours)")
    return args


def words_per_block(N):
    return N // 64 + (1 if N % 64 else 0)


def seeded_blocks(rng, T, N):
    L = words_per_block(N)
    w = rng.integers(0, 2**64, size=(T, L), dtype=np.uint64)
    rem = N % 64
    if rem:
        w[:, L - 1] &= np.uint64((0xFFFFFFFFFFFFFFFF << (64 - rem)) & 0xFFFFFFFFFFFFFFFF)
    return w.reshape(-1)


# ---------------------------------------------------------------------------
# numpy restatement of the path (the bench's own independent check; nothing from oracle/)
# ---------------------------------------------------------------------------
def np_key_mask(N, positions):
    """position p -> word p>>6, bit 63-(p&63)   (reference src/SecretKey.cpp:116-121)"""
    m = np.zeros(words_per_block(N), dtype=np.uint64)
    for s_ in positions:
        m[int(s_) >> 6] |= np.uint64(1 << (63 - (int(s_) & 63)))
    return m


def np_count(words, L, mask):
    """blocks whose words cover the key mask: the AND over the D secret positions (src/SecretKey.cpp:131-140)"""
    w = np.asarray(words, dtype=np.uint64).reshape(-1, L)
    return int(((w & mask) == mask).all(axis=1).sum())


def np_mul(a, b, L):
    """out[(i*T2+j)*L+k] = a[i*L+k] & b[j*L+k]   (src/Ciphertext.cpp:153-163)"""
    a2, b2 = np.asarray(a, dtype=np.uint64).reshape(-1, L), np.asarray(b, dtype=np.uint64).reshape(-1, L)
    return (a2[:, None, :] & b2[None, :, :]).reshape(-1)


def np_permute(words, N, perm):
    """out_bit[i] = in_bit[perm[i]], i < N, pad bits zero, every block   (src/Ciphertext.cpp:24-69)"""
    L = words_per_block(N)
    w = np.asarray(words, dtype=np.uint64).reshape(-1, L)
    bits = np.unpackbits(w.astype(">u8").view(np.uint8).reshape(w.shape[0], L * 8), axis=1)   # MSB first = position order
    out = np.zeros_like(bits)
    out[:, :N] = bits[:, np.asarray(perm, dtype=np.int64)]
    return np.packbits(out, axis=1).view(">u8").astype(np.uint64).reshape(-1)


def planted_blocks(rng, T, N, mask, k=None):
    """raw random blocks almost never satisfy a key; set the key bits in a few of them so that the fold has
    something to count"""
    L = words_per_block(N)
    w = seeded_blocks(rng, T, N).reshape(T, L)
    k = int(rng.integers(20, 60)) if k is None else k
    rows = rng.choice(T, size=min(T, k), replace=False)
    w[rows] |= mask
    return w.reshape(-1)


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel, workload, fold=None):
    """dram bytes (read + write) per launch of the dominant kernel, from the committed ncu --set full
    capture of this workload (profiles/<round>_<workload>_ncu_summary.json), or None.  `fold`: the FOLD template
    argument (the third) of mul_outer_kernel<VT, U, FOLD, ALIGN>."""
    import re
    for tag in ("r2", "r1c", "r1b", "r1"):                      # the latest capture first
        try:
            with open(os.path.join(ROOT, "profiles", "%s_%s_ncu_summary.json" % (tag, workload))) as f:
                for name, k in json.load(f)["kernels"].items():
                    m = re.search(kernel + r"<([^>]*)>", name)
                    targs = [x.strip() for x in m.group(1).split(",")] if m else []
                    if kernel in name and (fold is None or (len(targs) >= 3 and targs[2] == str(fold))):
                        return k["dram_traffic_bytes_per_launch"]
        except Exception:
            pass
    return None


class ClockSampler(threading.Thread):
    """SM clock, board power and throttle reasons during the timed region (NVML, ~1 ms period)."""

    def __init__(self, index, period_s=0.0005, with_power=False):
        super().__init__(daemon=True)
        self.index, self.samples, self.max_mhz = index, [], None
        self.period_s, self.with_power = period_s, with_power
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = str(e)

    NAMES = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
             0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
             0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def run(self):
        if not self.ok:
            return
        i = 0
        while not self._stop_evt.is_set():
            try:
                mhz = self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                mw = None
                if self.with_power:              # board power: only the slow samplers (sustained run, side workloads) --
                    try:                         # NVML calls take a driver lock, and the headline's region is 7 ms long
                        mw = self.nv.nvmlDeviceGetPowerUsage(self.h)
                    except Exception:
                        mw = None
                self.samples.append((time.perf_counter(), mhz, r, mw))
            except Exception:
                pass
            i += 1
            time.sleep(self.period_s)

    def stop(self, t_begin=None, t_end=None):
        """Median SM clock and the throttle reasons of the samples taken inside [t_begin, t_end] (perf_counter): the
        thread is started a little before the timed region so that NVML is warm, and only what falls inside counts."""
        self._stop_evt.set()
        self.join(timeout=2)
        inside = [x for x in self.samples if (t_begin is None or x[0] >= t_begin) and (t_end is None or x[0] <= t_end)]
        note = None
        if not inside and self.samples and t_begin is not None:
            # a timed region shorter than one NVML round trip (a few steps only): take the samples closest to it --
            # the GPU ran the same kernels (warm-up, e2e) right before and after
            mid = 0.5 * (t_begin + (t_end if t_end is not None else t_begin))
            inside = sorted(self.samples, key=lambda x: abs(x[0] - mid))[:3]
            note = "timed region shorter than the sampling period: the %d samples nearest to it" % len(inside)
        reasons = set()
        for x in inside:
            for bit, name in self.NAMES.items():
                if x[2] & bit and name != "gpu_idle":
                    reasons.add(name)
        med = float(np.median([x[1] for x in inside])) if inside else None
        out = {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(reasons), "samples": len(inside)}
        if inside:
            out["sm_mhz_min"] = float(min(x[1] for x in inside))
            pw = [x[3] for x in inside if x[3] is not None]
            if pw:
                out["power_w_max"] = max(pw) / 1e3
                out["power_w_median"] = float(np.median(pw)) / 1e3
        if note:
            out["note"] = note
        return out


# ---------------------------------------------------------------------------
# CPU arms (the only place bench.py touches oracle/)
# ---------------------------------------------------------------------------
def cpu_reference_once(N, D, T1, T2, threads, reps, opt="O3"):
    """(kind, mul_s, dec_s) for `threads` replicas of a T1 x T2 multiply + decrypt."""
    from oracle import pyoracle
    if pyoracle.ref_available(opt):
        ref = pyoracle.Ref(opt)
        m, d, _ = ref.bench_mul_decrypt(N, D, T1, T2, threads=threads, reps=reps, seed=1)
        return "reference", m, d
    # the reference build did not travel: time the C restatement (one thread)
    o = pyoracle.Oracle()
    rng = np.random.default_rng(1)
    a, b = seeded_blocks(rng, T1, N), seeded_blocks(rng, T2, N)
    s = rng.permutation(N)[:D].astype(np.uint64)
    best_m = best_d = 1e300
    for _ in range(reps):
        t0 = time.perf_counter()
        prod = o.mul(a, b, words_per_block(N))
        t1 = time.perf_counter()
        o.decrypt(prod, N, s)
        t2 = time.perf_counter()
        best_m, best_d = min(best_m, t1 - t0), min(best_d, t2 - t1)
    return "port", best_m, best_d


def cpu_baseline(N, D, T1, T2):
    kind, m, d = cpu_reference_once(N, D, T1, T2, threads=1, reps=3)
    blocks = T1 * T2
    out = {"value": blocks / (m + d), "unit": UNIT, "cores": 1, "kind": kind,
           "sample": "one %dx%d pair (%d output blocks): public operator* %.3f s + SecretKey::decrypt %.3f s, "
                     "best of 3, single thread (the reference has no threading), built -O3 -DNDEBUG"
                     % (T1, T2, blocks, m, d),
           "mul_blocks_per_s": blocks / m, "decrypt_blocks_per_s": blocks / d,
           "host_cores_available": os.cpu_count()}
    from oracle import pyoracle
    if kind == "reference" and pyoracle.ref_available("O0"):
        # what the shipped CMakeLists (no build type, hence no -O flag) really produces; a quarter-size sample
        _, m0, d0 = cpu_reference_once(N, D, max(1, T1 // 4), T2, threads=1, reps=1, opt="O0")
        out["as_shipped_no_opt_flag_blocks_per_s"] = max(1, T1 // 4) * T2 / (m0 + d0)
    return out


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    N, D, T1, T2, desc = WORKLOADS[args.workload]
    T1, T2 = args.t1 or T1, args.t2 or T2
    threads = max(1, os.cpu_count() or 1)
    # the SAME pair as the GPU arm (T1 x T2) in every replica thread; replicas are capped by host memory: the reference
    # holds v + bitlen of the product twice (operator* copies its result, src/Ciphertext.cpp:241) and one byte per BIT
    # of decrypt scratch (src/SecretKey.cpp:110-124)
    try:
        import psutil
        per_replica = T1 * T2 * (words_per_block(N) * 8 * 4 + N) * 1.2
        threads = max(1, min(threads, int(psutil.virtual_memory().available * 0.6 / per_replica)))
    except Exception:
        pass
    times = []
    kind = "reference"
    for i in range(args.warmup + args.steps):
        kind, m, d = cpu_reference_once(N, D, T1, T2, threads=threads, reps=1)
        if i >= args.warmup:
            times.append(m + d)
    blocks = threads * T1 * T2
    total = float(np.sum(times))
    value = blocks * len(times) / total
    sample = ("%d replica threads x one %dx%d pair per step (%d output blocks/step; the same pair size as the GPU arm), "
              "public operator* + SecretKey::decrypt; harness-level parallelism, the reference itself is single-threaded"
              % (threads, T1, T2, blocks))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": args.workload + ": " + desc, "sample": sample,
                       "left_blocks_per_replica": T1, "right_blocks": T2},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------
# our arm: helpers
# ---------------------------------------------------------------------------
def event_time_us(torch, fn, n_items, reps=3, rounds=3):
    """median over `rounds` of (CUDA-event time of `reps` passes over fn(0..n_items-1)) / calls, in us; one untimed pass first"""
    for i in range(n_items):
        fn(i)
    torch.cuda.synchronize()
    res = []
    for _ in range(rounds):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            for i in range(n_items):
                fn(i)
        e1.record()
        torch.cuda.synchronize()
        res.append(e0.elapsed_time(e1) * 1e3 / (reps * n_items))
    return float(np.median(res))


DUMP_BYTES = 48 << 20      # product words of a whole dump (all ranks), as float64 halves: 16 bytes per word


def sample_outputs(torch, products, L, counts, world):
    """What --dump-outputs writes: the counts and a fixed sample of product blocks.  `products` is a device tensor of
    int64 words holding whole blocks, pair-major.  The sample depends only on the number of blocks and ranks, so two
    runs with the same arguments sample the same blocks; every rank takes 1/world of the budget."""
    total = products.numel() // L
    rng = np.random.default_rng(20240613)
    idx = np.unique(rng.integers(0, total, size=min(total, DUMP_BYTES // (16 * L * world))))
    rows = products.reshape(total, L)[torch.from_numpy(idx).to(products.device)]
    words = rows.cpu().numpy().view(np.uint64)
    return {"counts": counts.cpu().numpy().astype(np.float64),
            "product_blocks": idx.astype(np.float64),
            "product_words": np.stack([words >> np.uint64(32), words & np.uint64(0xFFFFFFFF)], axis=-1).astype(np.float64)}


def write_outputs(path, arrays, rank, world):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ("_rank%d" % rank if world > 1 else "") + ".npy"), a)


def precheck(eng, torch, dev, rank, world, comm):
    """Small cases compared word for word with the numpy restatement above, on every rank, before anything is timed.
    The left operand is sharded exactly as the timed runs shard it; every rank generates the WHOLE operand from the
    same seed, so the expected global count needs no communication.  Raises SystemExit on any difference."""
    done = []
    for N, D, T1g, T2 in ((1247, 16, 53 * world + 3, 37), (16383, 64, 5 * world + 1, 9), (191, 4, 40 * world + 1, 33)):
        L = words_per_block(N)
        ctx = eng.Context(N, D)
        rng = np.random.default_rng([77, N])
        pos = rng.permutation(N)[:D].astype(np.uint64)
        mask = np_key_mask(N, pos)
        key = eng.SecretKey(ctx, pos)
        a_all = planted_blocks(rng, T1g, N, mask, k=max(3, T1g // 7))
        b = planted_blocks(rng, T2, N, mask, k=5)
        first, count = eng.shard_range(T1g, rank, world)
        a = a_all[first * L:(first + count) * L]
        want_words = np_mul(a, b, L)
        want_local = np_count(want_words, L, mask)                 # counted on the PRODUCT words, not via count(a)*count(b)
        want_total = np_count(np_mul(a_all, b, L), L, mask)
        ca, cb = eng.Ciphertext.from_host(a, ctx), eng.Ciphertext.from_host(b, ctx)
        tag = "Context(%d,%d) %dx%d (rank %d of %d: rows %d..%d)" % (N, D, T1g, T2, rank, world, first, first + count)
        prod = ca * cb
        if not np.array_equal(prod.getValues(), want_words):
            raise SystemExit("precheck FAILED: multiply differs from numpy, " + tag)
        if key.count_satisfied(prod) != want_local:
            raise SystemExit("precheck FAILED: decrypt count differs from numpy, " + tag)
        bit, cnt, fprod = key.mul_decrypt(ca, cb, out="alloc")
        if cnt != want_local or bit != (want_local & 1) or not np.array_equal(fprod.getValues(), want_words):
            raise SystemExit("precheck FAILED: fused multiply->decrypt differs from numpy, " + tag)
        bit, cnt = key.mul_decrypt(ca, cb)
        if cnt != want_local:
            raise SystemExit("precheck FAILED: fused count-only differs from numpy, " + tag)
        perm = np.random.default_rng([78, N]).permutation(N).astype(np.uint64)
        if not np.array_equal(prod.applyPermutation(eng.Permutation(ctx, perm)).getValues(), np_permute(want_words, N, perm)):
            raise SystemExit("precheck FAILED: permute differs from numpy, " + tag)
        if comm is not None:
            got = comm.decrypt(key, prod)                           # fold + NVLink exchange in one kernel, blocking
            if got != (want_total & 1, want_total):
                raise SystemExit("precheck FAILED: sharded decrypt %s, numpy says %d, %s" % (got, want_total, tag))
            tot = torch.zeros(2, dtype=torch.int64, device=dev)
            comm.mul_push(key, ca, cb, out=None, collect_n=1, device_totals_ptr=tot.data_ptr(),
                          device_local_ptr=tot.data_ptr() + 8)     # fused multiply -> fold -> exchange, one kernel
            eng.sync()
            if tot.tolist() != [want_total, want_local]:
                raise SystemExit("precheck FAILED: fused sharded multiply->decrypt %s, numpy says %s, %s"
                                 % (tot.tolist(), [want_total, want_local], tag))
        done.append("N=%d %dx%d" % (N, T1g, T2))
    return {"passed": True, "cases": done,
            "checked": "multiply, fused multiply->decrypt (product words and count), count-only, decrypt count, permute"
                       + (", sharded decrypt and fused sharded multiply->decrypt totals over %d GPUs" % world if comm is not None else "")
                       + " -- every word against the numpy restatement in bench.py",
            "ranks": world}


def other_kernels(eng, torch, ctx, vo, N, D, L, peak, with_cpu):
    """Permute and add on products the bench already holds (BASELINE.md 3-4: reported beside the headline, each
    against the HBM roofline at 16*L bytes per block, with the unmodified reference's public calls on a bounded
    sample).  Never part of `value`; any failure here is reported, not raised."""
    out = {}
    try:
        T = vo[0].n_blocks
        nb = len(vo) // 2 * 2
        if nb < 2:
            return {"skipped": "needs two products to ping-pong between (--pairs >= 2)"}
        perm_np = np.random.default_rng(3).permutation(N).astype(np.uint64)
        perm = eng.Permutation(ctx, perm_np)

        def permute_pass(_):                     # every even product into its odd neighbour: nothing stays in L2
            for i in range(0, nb, 2):
                vo[i].permute_into(perm, vo[i + 1])
        t = event_time_us(torch, permute_pass, 1) * 1e-6 / (nb // 2)
        gbs = T * 16 * L / t / 1e9
        out["permute"] = {"blocks_per_s": T / t, "gbs_read_plus_write": gbs, "frac_of_peak": gbs / peak,
                          "avg_launch_us": t * 1e6, "blocks_per_launch": T}

        def add_pass(_):
            for i in range(0, nb, 2):
                s_ = vo[i] + vo[i + 1]           # csgn_concat into a fresh buffer
                del s_
        t = event_time_us(torch, add_pass, 1) * 1e-6 / (nb // 2)
        gbs = 2 * T * 16 * L / t / 1e9
        out["add"] = {"blocks_per_s": 2 * T / t, "gbs_read_plus_write": gbs, "frac_of_peak": gbs / peak,
                      "avg_launch_us": t * 1e6, "blocks_per_launch": 2 * T}
        if with_cpu:
            from oracle import pyoracle
            if pyoracle.ref_available():
                ref = pyoracle.Ref()
                rng = np.random.default_rng(5)
                Tp = 20000 if N < 4096 else 1500          # the reference unpacks 8 bytes per BIT: 43 us per block at N=1247
                v = seeded_blocks(rng, Tp, N)
                h = ref.ct(v, N, D)
                t0 = time.perf_counter()
                hp = ref.lib.ref_ct_permute(h, perm_np.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), N)
                tp = time.perf_counter() - t0
                ref.ct_free(hp)
                Ta = 100000 if N < 4096 else 8000
                h2 = ref.ct(seeded_blocks(rng, Ta, N), N, D)
                t0 = time.perf_counter()
                hs = ref.lib.ref_ct_add(h2, h)
                ta = time.perf_counter() - t0
                for x in (h, h2, hs):
                    ref.ct_free(x)
                out["permute"]["cpu_reference_blocks_per_s"] = Tp / tp
                out["permute"]["cpu_sample"] = ("public applyPermutation on a %d-block ciphertext, %.2f s, one thread; the "
                                                "reference walks every block but RETURNS only block 0 (src/Ciphertext.cpp:33-40)"
                                                % (Tp, tp))
                out["add"]["cpu_reference_blocks_per_s"] = (Ta + Tp) / ta
                out["add"]["cpu_sample"] = "public operator+ of %d + %d blocks, %.3f s, one thread" % (Ta, Tp, ta)
    except Exception as e:  # noqa: BLE001
        out["error"] = "%s: %s" % (type(e).__name__, e)
    return out


def other_workloads(eng, torch, dist, dev, rank, world, comm, peak, chain_d):
    """BASELINE.json configs[3] and [4] next to the headline, every kernel CUDA-event timed against the same roofline
    and every count compared with the host-known truth.  N > 1: the left operand is split over the ranks (cfg5: the
    SAME total work at every N -- strong scaling; cfg4: 1000 rows per rank -- weak scaling, 10^9 blocks at 8 GPUs);
    times are the max over ranks, rates are whole-job."""
    res = {}

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        t = torch.tensor([x], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(t)
        return int(t.item())

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def kernel_entry(us, blocks_rank, bytes_per_block, total_blocks):
        gbs = blocks_rank * bytes_per_block / us / 1e3
        return {"us": us, "gbs_per_gpu": gbs, "frac_of_peak": gbs / peak, "blocks_per_s": total_blocks / us * 1e6}

    # ---- configs[4]: Context(16383,64) ------------------------------------------------------------------------
    N, D = 16383, 64
    L = words_per_block(N)
    ctx = eng.Context(N, D)
    pos = np.random.default_rng(7).permutation(N)[:D].astype(np.uint64)
    mask = np_key_mask(N, pos)
    key = eng.SecretKey(ctx, pos)
    perm = eng.Permutation(ctx, np.random.default_rng(3).permutation(N).astype(np.uint64))
    for name, T in (("cfg5_300x300", 300), ("cfg5_2000x2000", 2000)):
        try:
            first, count = eng.shard_range(T, rank, world)
            if count == 0:
                raise RuntimeError("more ranks than rows")
            rng = np.random.default_rng([5, T])
            a_all, b = planted_blocks(rng, T, N, mask), planted_blocks(rng, T, N, mask)
            a = a_all[first * L:(first + count) * L]
            want = np_count(a_all, L, mask) * np_count(b, L, mask)
            prod_bytes = count * T * L * 8
            P = int(max(2, min(12, 2.4e9 // prod_bytes)))
            da = torch.from_numpy(a.view(np.int64)).to(dev)
            db = torch.from_numpy(b.view(np.int64)).to(dev)
            outs = torch.empty((P, count * T * L), dtype=torch.int64, device=dev)
            va, vb = eng.Ciphertext.from_tensor(da, ctx), eng.Ciphertext.from_tensor(db, ctx)
            vo = [eng.Ciphertext.from_tensor(outs[p], ctx) for p in range(P)]
            cnt = torch.zeros(P, dtype=torch.int64, device=dev)
            reps = 3 if prod_bytes < 1e9 else 1
            sampler = ClockSampler(dev.index, period_s=0.01, with_power=True)
            sampler.start()
            sync_all()
            t0 = time.perf_counter()
            t_mul = allmax(event_time_us(torch, lambda i: va.mul_into(vb, vo[i]), P, reps))
            t_dec = allmax(event_time_us(torch, lambda i: key.count_satisfied_async(vo[i], cnt.data_ptr() + 8 * i), P, reps))
            got_two = allsum(int(cnt[0].item()))
            t_fus = allmax(event_time_us(torch, lambda i: key.mul_count_async(va, vb, cnt.data_ptr() + 8 * i, out=vo[i]), P, reps))
            got_fused = allsum(int(cnt[P - 1].item()))
            t_perm = allmax(event_time_us(torch, lambda i: vo[i].permute_into(perm, vo[(i + 1) % P]), P, reps))
            clocks = sampler.stop(t0, time.perf_counter())
            if got_two != want or got_fused != want:
                raise RuntimeError("count differs from the host-known truth: two-pass %d, fused %d, numpy %d" % (got_two, got_fused, want))
            blocks = T * T
            res[name] = {"context": "Context(16383,64)", "blocks": blocks, "bytes_per_block": 8 * L,
                         "scaling": "strong (left operand split over %d GPUs)" % world if world > 1 else "single GPU",
                         "rotating_products": P, "product_bytes_per_gpu": prod_bytes,
                         "multiply": kernel_entry(t_mul, count * T, 8 * L, blocks),
                         "decrypt": kernel_entry(t_dec, count * T, 8 * L, blocks),
                         "fused_multiply_decrypt": kernel_entry(t_fus, count * T, 8 * L, blocks),
                         "permute": kernel_entry(t_perm, count * T, 16 * L, blocks),
                         "mul_then_decrypt_blocks_per_s": blocks / (t_mul + t_dec) * 1e6,
                         "count_checked_vs_host_truth": want, "clocks": clocks}
            del va, vb, vo, outs, da, db
        except Exception as e:  # noqa: BLE001
            res[name] = {"error": "%s: %s" % (type(e).__name__, e)}
        torch.cuda.empty_cache()

    # ---- configs[3]: the chain (a*b)*d at Context(1247,16), chain_d blocks in d -------------------------------
    try:
        N, D, T1, T2 = 1247, 16, 1000, 1000
        L = words_per_block(N)
        ctx = eng.Context(N, D)
        pos = np.random.default_rng(7).permutation(N)[:D].astype(np.uint64)
        mask = np_key_mask(N, pos)
        key = eng.SecretKey(ctx, pos)
        a = planted_blocks(np.random.default_rng([1, rank]), T1, N, mask, k=31)      # this rank's 1000 rows
        b = planted_blocks(np.random.default_rng([2]), T2, N, mask, k=17)
        d = planted_blocks(np.random.default_rng([3]), chain_d, N, mask, k=5)
        want = allsum(np_count(a, L, mask)) * np_count(b, L, mask) * np_count(d, L, mask)
        da, db, dd = (torch.from_numpy(x.view(np.int64)).to(dev) for x in (a, b, d))
        x = torch.empty(T1 * T2 * L, dtype=torch.int64, device=dev)
        y = torch.empty(T1 * T2 * chain_d * L, dtype=torch.int64, device=dev)
        va, vb, vd = (eng.Ciphertext.from_tensor(t_, ctx) for t_ in (da, db, dd))
        vx, vy = eng.Ciphertext.from_tensor(x, ctx), eng.Ciphertext.from_tensor(y, ctx)
        tot = torch.zeros(2, dtype=torch.int64, device=dev)
        out_blocks = T1 * T2 * chain_d

        def fold_two_pass(_):
            if comm is not None:
                comm.push(key, vy, 1, tot.data_ptr())
            else:
                key.count_satisfied_async(vy, tot.data_ptr())

        def fold_fused(_):
            if comm is not None:
                comm.mul_push(key, vx, vd, out=vy, collect_n=1, device_totals_ptr=tot.data_ptr())
            else:
                key.mul_count_async(vx, vd, tot.data_ptr(), out=vy)

        sampler = ClockSampler(dev.index, period_s=0.01, with_power=True)
        sampler.start()
        sync_all()
        t0 = time.perf_counter()
        t_m1 = allmax(event_time_us(torch, lambda i: va.mul_into(vb, vx), 1, 3))
        t_m2 = allmax(event_time_us(torch, lambda i: vx.mul_into(vd, vy), 1, 2))
        t_dec = allmax(event_time_us(torch, fold_two_pass, 1, 2))
        got_two = int(tot[0].item())
        if world > 1 and comm is None:
            got_two = allsum(got_two)
        t_fus = allmax(event_time_us(torch, fold_fused, 1, 2))
        got_fused = int(tot[0].item())
        if world > 1 and comm is None:
            got_fused = allsum(got_fused)
        clocks = sampler.stop(t0, time.perf_counter())
        if got_two != want or got_fused != want:
            raise RuntimeError("count differs from the host-known truth: two-pass %d, fused %d, numpy %d" % (got_two, got_fused, want))
        total = out_blocks * world
        res["cfg4_chain"] = {"context": "Context(1247,16)", "chain": "(a*b)*d: 1000 x 1000 x %d blocks per GPU" % chain_d,
                             "blocks_per_gpu": out_blocks, "blocks_total": total, "product_bytes_per_gpu": out_blocks * 8 * L,
                             "scaling": "weak (1000 rows of a per GPU)" if world > 1 else "single GPU",
                             "multiply_1M": {"us": t_m1},
                             "multiply_chain": kernel_entry(t_m2, out_blocks, 8 * L, total),
                             "decrypt" + ("_with_exchange" if comm is not None else ""): kernel_entry(t_dec, out_blocks, 8 * L, total),
                             "fused_multiply_decrypt" + ("_with_exchange" if comm is not None else ""): kernel_entry(t_fus, out_blocks, 8 * L, total),
                             "two_pass_blocks_per_s": total / (t_m1 + t_m2 + t_dec) * 1e6,
                             "fused_blocks_per_s": total / (t_m1 + t_fus) * 1e6,
                             "count_checked_vs_host_truth": want, "clocks": clocks}
        del va, vb, vd, vx, vy, x, y
    except Exception as e:  # noqa: BLE001
        res["cfg4_chain"] = {"error": "%s: %s" % (type(e).__name__, e)}
    torch.cuda.empty_cache()
    return res


def cpp_e2e(pairs, steps):
    """tools/cpp_e2e.cpp: the same step through the certFHE C++ drop-in API, in its own process (the GPU is shared)."""
    exe = os.path.join(ROOT, "tools", "bin", "cpp_e2e")
    if not os.path.exists(exe):
        return {"skipped": "tools/bin/cpp_e2e not built"}
    try:
        r = subprocess.run([exe, str(pairs), str(steps)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
        lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
        if r.returncode != 0 or not lines:
            return {"error": "rc %d: %s" % (r.returncode, (r.stderr or r.stdout)[-400:])}
        return json.loads(lines[-1])
    except Exception as e:  # noqa: BLE001
        return {"error": "%s: %s" % (type(e).__name__, e)}


def connect_exchange(args, world, dev):
    """(comm, description).  comm is None at N=1 and for --exchange nccl.  Every rank must take the same
    path, so a rank that cannot map its peers' mailboxes makes all of them fall back to NCCL -- loudly."""
    if world == 1:
        return None, "single GPU: no exchange"
    if args.exchange == "nccl":
        return None, "separate NCCL all-reduce of the counts"
    import torch
    import torch.distributed as dist
    from csgn_b200 import sharding
    comm, err = None, ""
    try:
        comm = sharding.connect_peers()
    except Exception as e:  # noqa: BLE001
        err = str(e)
    ok = torch.tensor([1 if comm is not None else 0], dtype=torch.int64, device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if int(ok.item()) == 1:
        return comm, ("fused into the kernel: its last CTA stores the count into every rank's mailbox over "
                      "NVLink and the launch closing the batch collects the sums (csrc/peer.cuh); no NCCL call in the step")
    sys.stderr.write("bench: peer mailboxes unavailable (%s); using the NCCL all-reduce\n" % err)
    return None, "separate NCCL all-reduce (peer mailboxes unavailable: %s)" % (err or "on another rank")


# ---------------------------------------------------------------------------
# our arm: the headline
# ---------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from csgn_b200 import engine as eng

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    N, D, T1, T2, desc = WORKLOADS[args.workload]
    T1g, T2 = args.t1 or T1, args.t2 or T2          # T1g: the left operand as given on the command line
    if args.t1 or args.t2:
        desc = "Context(%d,%d): %dx%d -> %d output blocks, multiply then decrypt" % (N, D, T1g, T2, T1g * T2)
    L, P = words_per_block(N), args.pairs
    eng.init(local)
    # a real (non-default) stream: handle 0 would mean "the library's own stream" to csgn_set_stream,
    # and torch.cuda.Event only sees the stream it is recorded on
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)
    ctx = eng.Context(N, D)
    comm, exchange = connect_exchange(args, world, dev)
    fused = args.mode == "fused"

    pre = None
    if not args.no_precheck:
        pre = precheck(eng, torch, dev, rank, world, comm)

    # --- synthetic inputs: pinned host copies (e2e) and device copies (value) ---------
    # Global left operand of pair p has T1*world blocks; this rank owns csgn_shard_range.
    strong = args.scaling == "strong" and world > 1
    first, count = eng.shard_range(T1g if strong else T1g * world, rank, world)
    T1 = count                                        # this rank's blocks of the left operand
    if strong and T1g % world:
        raise SystemExit("--scaling strong needs --t1 divisible by the number of GPUs")
    host_a = torch.empty((P, T1 * L), dtype=torch.int64).pin_memory()
    host_b = torch.empty((P, T2 * L), dtype=torch.int64).pin_memory()
    key_pos = np.random.default_rng(7).permutation(N)[:D].astype(np.uint64)
    key = eng.SecretKey(ctx, key_pos)
    key_mask = np_key_mask(N, key_pos)

    # host-known truth: satisfied blocks of every operand, counted in numpy from the host copies
    truth_a, truth_b = np.zeros(P, dtype=np.int64), np.zeros(P, dtype=np.int64)
    for p in range(P):
        rng_a = np.random.default_rng([1000 + p, rank])       # this rank's shard of A_p
        rng_b = np.random.default_rng([2000 + p])             # B_p, identical on every rank
        wa, wb = planted_blocks(rng_a, T1, N, key_mask), planted_blocks(rng_b, T2, N, key_mask)
        host_a[p].numpy().view(np.uint64)[:] = wa
        host_b[p].numpy().view(np.uint64)[:] = wb
        truth_a[p], truth_b[p] = np_count(wa, L, key_mask), np_count(wb, L, key_mask)
    expected = torch.from_numpy(truth_a * truth_b).to(dev)    # count(a_shard * b) on this rank ...
    if world > 1:
        dist.all_reduce(expected)                             # ... summed over the shards
    expected_host = expected.cpu()

    dev_a, dev_b = host_a.to(dev), host_b.to(dev)
    out = torch.empty((P, T1 * T2 * L), dtype=torch.int64, device=dev)
    # two result buffers: the exchange of step k may still be running while step k+1 computes
    counts2 = [torch.zeros(P, dtype=torch.int64, device=dev) for _ in range(2)]
    pending = [None, None]
    va = [eng.Ciphertext.from_tensor(dev_a[p], ctx) for p in range(P)]
    vb = [eng.Ciphertext.from_tensor(dev_b[p], ctx) for p in range(P)]
    vo = [eng.Ciphertext.from_tensor(out[p], ctx) for p in range(P)]
    count_ptrs2 = [c.data_ptr() for c in counts2]
    step_no = [0]

    def drain():
        for i in (0, 1):
            if pending[i] is not None:
                pending[i].wait()
                pending[i] = None

    lagged = comm is not None and args.collect == "lagged"
    arr_a, arr_b, arr_o = eng.handle_array(va), eng.handle_array(vb), eng.handle_array(vo)
    arrays = (arr_a, arr_b, arr_o)

    def step_device(evs=None, final=True, fused_step=True):
        slot = step_no[0] & 1
        step_no[0] += 1
        if pending[slot] is not None:        # the all-reduce issued two steps ago: long finished
            pending[slot].wait()
            pending[slot] = None
        if evs:
            evs[0].record()
        if fused_step:
            if evs:
                evs[1].record()
            if comm is None:
                eng.mul_count_batch_async(key, None, None, count_ptrs2[slot], arrays=arrays)
            elif lagged and step_no[0] > 1:
                comm.mul_push_batch(key, arrays, count_ptrs2[slot ^ 1], lag=P)
                if final:
                    comm.collect(P, count_ptrs2[slot])
            else:
                comm.mul_push_batch(key, arrays, count_ptrs2[slot])
        else:
            eng.mul_into_batch(None, None, None, arrays=arrays)
            if evs:
                evs[1].record()
            if comm is None:
                key.count_satisfied_batch_async(None, count_ptrs2[slot], array=arr_o)
            elif lagged and step_no[0] > 1:
                comm.push_batch(key, None, count_ptrs2[slot ^ 1], lag=P, array=arr_o)
                if final:
                    comm.collect(P, count_ptrs2[slot])
            else:
                comm.push_batch(key, None, count_ptrs2[slot], array=arr_o)
        if evs:
            evs[2].record()
        if world > 1 and comm is None:
            pending[slot] = dist.all_reduce(counts2[slot], async_op=True)
        if evs:
            evs[3].record()

    def barrier():
        drain()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def check_counts(where, steps_done=2):
        for c in counts2[:min(2, max(1, steps_done))]:        # a single step only ever wrote slot 0
            if not torch.equal(expected, c):
                raise SystemExit("bench check failed (%s): device counts %s != host-known truth %s" % (where, c, expected))

    def timed_run(K, fused_step, sample=True):
        """W warm-up steps, a check, then exactly K timed steps between barriers; returns the measurements"""
        W_ = max(3, args.warmup)
        step_no[0] = 0
        for c in counts2:
            c.zero_()
        for i in range(W_):
            step_device(final=(i == W_ - 1), fused_step=fused_step)
        barrier()
        check_counts("after warm-up, %s" % ("fused" if fused_step else "two-pass"))
        for c in counts2:
            c.zero_()
        step_no[0] = 0
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(K)]
        sampler = ClockSampler(local) if sample else None
        if sampler:
            sampler.start()                  # before the barrier: NVML's first calls are slow
        barrier()
        launches0 = eng.launch_count()
        t_begin = time.perf_counter()
        for k in range(K):
            step_device(evs[k], final=(k == K - 1), fused_step=fused_step)
        barrier()
        t_end = time.perf_counter()
        clocks = sampler.stop(t_begin, t_end) if sampler else None
        launches = eng.launch_count() - launches0
        check_counts("after the timed region, %s" % ("fused" if fused_step else "two-pass"), K)
        total_ms = evs[0][0].elapsed_time(evs[K - 1][3])
        p1 = [e[0].elapsed_time(e[1]) for e in evs]        # two-pass: the multiplies
        p2 = [e[1].elapsed_time(e[2]) for e in evs]        # two-pass: the folds; fused: the whole step's kernels
        ar_ms = sum(e[2].elapsed_time(e[3]) for e in evs)
        t = torch.tensor([total_ms, sum(p1), sum(p2), ar_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, p1_ms, p2_ms, ar_ms = (float(x) for x in t.tolist())
        return {"total_ms": total_ms, "p1_ms": p1_ms, "p2_ms": p2_ms, "ar_ms": ar_ms, "p1_steps": p1, "p2_steps": p2,
                "clocks": clocks, "launches": int(launches), "wall_s": t_end - t_begin}

    K = args.steps
    main = timed_run(K, fused)
    dump = sample_outputs(torch, out, L, counts2[(K - 1) & 1], world) if args.dump_outputs else None   # the last step's slot
    blocks_per_step = P * T1 * T2 * world            # whole job (T1 = per-rank share)
    value = blocks_per_step * K / (main["total_ms"] * 1e-3)
    bytes_per_block = 8 * L
    peak, peak_src = measured_peak_gbs()
    per_gpu_bytes = P * T1 * T2 * bytes_per_block * K

    def kstat(ms, steps):
        gbs = per_gpu_bytes / (ms * 1e-3) / 1e9
        return {"blocks_per_s_per_gpu": P * T1 * T2 * K / (ms * 1e-3), "gbs": gbs, "frac_of_peak": gbs / peak,
                "avg_launch_us": ms * 1e3 / (K * P), "min_step_launch_us": min(steps) * 1e3 / P,
                "median_step_launch_us": float(np.median(steps)) * 1e3 / P}

    if fused:
        kernels = {"fused_multiply_decrypt": kstat(main["p2_ms"], main["p2_steps"])}
        dom_ms, dom_name, dom_fold = main["p2_ms"], "mul_outer_kernel<uint4, U, FOLD=1> (product written + decrypt-folded in one pass)", 1
    else:
        kernels = {"multiply": kstat(main["p1_ms"], main["p1_steps"]), "decrypt": kstat(main["p2_ms"], main["p2_steps"])}
        dom_ms, dom_name, dom_fold = main["p1_ms"], "mul_outer_kernel<uint4, U, FOLD=0>", 0
    kernels["allreduce_ms_per_step"] = main["ar_ms"] / K
    dom_gbs = per_gpu_bytes / (dom_ms * 1e-3) / 1e9

    # --- e2e: pinned host operands through the public C ABI ---------------------------
    e2e = None
    if not args.no_e2e:
        uploader = eng.UploadBatch([host_a[p].data_ptr() for p in range(P)] + [host_b[p].data_ptr() for p in range(P)],
                                   [T1] * P + [T2] * P, ctx)
        # results travel back through a ring of pinned host buffers; each D2H gets an event and is checked on the host
        # one step LATER (after the next step has been enqueued), so the GPU never idles while the host reads
        host_ring = [torch.zeros(P, dtype=torch.int64).pin_memory() for _ in range(4)]
        ring_ev = [torch.cuda.Event() for _ in range(4)]
        pending_checks = []                                                # [(event, host buffer)], oldest first
        e2e_no = [0]
        d2h_no = [0]
        e2e_lag = comm is not None and args.collect == "lagged"

        def fetch(src):
            """enqueue the D2H of one step's P counts"""
            i = d2h_no[0] % 4
            d2h_no[0] += 1
            host_ring[i].copy_(src, non_blocking=True)
            ring_ev[i].record(stream)
            pending_checks.append((ring_ev[i], host_ring[i]))

        def check_oldest():
            ev, buf = pending_checks.pop(0)
            ev.synchronize()
            if not torch.equal(buf, expected_host):
                raise SystemExit("e2e result differs from the host-known truth: %s vs %s" % (buf, expected_host))

        def step_e2e(final=False):
            # N > 1 with the lagged collect: the launch closing step k collects step k-1's sums (they arrived long
            # ago, so no rank waits for a slower one); the D2H enqueued after it carries step k-1's result.
            slot = e2e_no[0] & 1
            e2e_no[0] += 1
            ops = uploader.upload()                                        # csgn_buf_upload_batch: 2P operands, H2D on the copy stream
            ha, hb = eng.handle_slice(ops, 0, P), eng.handle_slice(ops, P, P)
            ho = (ctypes.c_void_p * P)()                                   # the library allocates the P products
            lag_now = e2e_lag and e2e_no[0] > 1
            dst = count_ptrs2[slot ^ 1] if lag_now else count_ptrs2[slot]
            if fused:
                if comm is None:
                    eng.mul_count_batch_async(key, None, None, dst, arrays=(ha, hb, ho))
                else:
                    comm.mul_push_batch(key, (ha, hb, ho), dst, lag=P if lag_now else 0)
            else:
                eng.mul_batch_arrays(ha, hb, ho)                           # csgn_mul_batch
                if comm is not None:
                    comm.push_batch(key, None, dst, lag=P if lag_now else 0, array=ho)
                else:
                    key.count_satisfied_batch_async(None, dst, array=ho)
            eng.free_handles(ops)                                          # stream-ordered frees
            eng.free_handles(ho)
            if world > 1 and comm is None:
                dist.all_reduce(counts2[slot])
            if e2e_lag:
                if lag_now:
                    fetch(counts2[slot ^ 1])                               # step k-1's sums, collected by step k's closing launch
                if final:                                                  # nothing follows: fetch this step's sums too
                    comm.collect(P, count_ptrs2[slot])
                    fetch(counts2[slot])
            else:
                fetch(counts2[slot])
            while len(pending_checks) > 1:                                 # everything but the newest: already behind the queue
                check_oldest()

        def run_e2e(n):
            e2e_no[0] = 0
            for i in range(n):
                step_e2e(final=(i == n - 1))
            while pending_checks:
                check_oldest()

        run_e2e(max(3, args.warmup))
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run_e2e(K)                                                         # the last result is on the host ...
        e1.record()                                                        # ... before the clock stops
        barrier()
        e2e_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
        e2e = {"value": blocks_per_step * K / (float(e2e_ms.item()) * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": int(P * (T1 + T2) * L * 8), "d2h_bytes_per_step": int(P * 8),
               "ms_per_step": float(e2e_ms.item()) / K,
               "path": ("csgn_buf_upload_batch (2P operands, pinned host) -> %s; one D2H of the P counts per step, read and checked "
                        "against the host-known truth on the host every step (one step behind the enqueue); per GPU"
                        % (("csgn_mul_decrypt_sharded_batch_async" if comm is not None else "csgn_mul_count_batch_async")
                           if fused else
                           ("csgn_mul_batch -> " + ("csgn_decrypt_sharded_batch_async" if comm is not None
                                                    else "csgn_decrypt_count_batch_async"))))}

    # --- side measurements (never part of `value`) -------------------------------------
    extras = not args.no_extras
    two_pass = sustained = None
    if extras:
        other = timed_run(K, not fused, sample=False)       # the other definition of the step, same buffers
        o_val = blocks_per_step * K / (other["total_ms"] * 1e-3)
        if fused:
            two_pass = {"value": o_val, "unit": UNIT, "ms_per_step": other["total_ms"] / K,
                        "multiply": kstat(other["p1_ms"], other["p1_steps"]), "decrypt": kstat(other["p2_ms"], other["p2_steps"]),
                        "gpu_launches": other["launches"],
                        "note": "round-1 definition of the step: csgn_mul_into_batch then csgn_decrypt_count_batch_async"}
        else:
            two_pass = {"fused_value": o_val, "unit": UNIT, "ms_per_step": other["total_ms"] / K,
                        "fused_multiply_decrypt": kstat(other["p2_ms"], other["p2_steps"])}
    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": max(3, args.warmup),
            "ms_per_step": main["total_ms"] / K, "higher_is_better": True, "scaling": "strong" if strong else "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": args.workload + ": " + desc, "pairs_per_step": P,
                       "mode": ("fused: one kernel per pair writes the product and decrypt-folds it in registers"
                                if fused else "two-pass: multiply kernels, then decrypt kernels"),
                       "streams": "library lanes (CSGN_LANES, default 2)",
                       "left_blocks_per_rank": T1, "right_blocks": T2,
                       "blocks_per_step": blocks_per_step, "bytes_per_block": bytes_per_block,
                       "l2": "no flush needed: a step writes %d x %.0f MB of products (>> 126 MB L2)%s"
                             % (P, T1 * T2 * L * 8 / 1e6, "" if fused else ", each product is read %d kernels after it was written" % P),
                       "sharding": "left operand by block range, right operand replicated; per step one %d-word "
                                   "exchange of the counts" % P if world > 1 else "single GPU",
                       "exchange": exchange + ((" [collect: %s]" % args.collect) if comm is not None else ""),
                       "inputs": "numpy default_rng raw blocks, pad bits zero, key bits set in 20-60 blocks per operand; "
                                 "key = default_rng(7).permutation(N)[:D]",
                       "checked": "every count of the timed loops == host-known truth (numpy count(a_shard)*count(b), "
                                  "summed over ranks)"},
            "roofline": {"bound": "hbm", "kernel": dom_name, "achieved": dom_gbs, "peak": peak,
                         "unit": "GB/s", "frac": dom_gbs / peak, "frac_of_nominal_8000": dom_gbs / 8000.0,
                         "traffic": ncu_traffic("mul_outer_kernel", args.workload, dom_fold),
                         "traffic_note": "ncu --set full, one isolated cold-cache launch: dram read+write bytes; the rest "
                                         "of the 160 MB product is still dirty in the 126 MB L2 when the launch ends and "
                                         "is written back under the next kernel (profiles/README.md)",
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": T1 * T2 * bytes_per_block,
                         "avg_launch_us": dom_ms * 1e3 / (K * P)},
            "kernels": kernels,
            "clocks": main["clocks"], "gpu_launches": main["launches"], "wall_ms_per_step": 1e3 * main["wall_s"] / K,
        }
        if e2e:
            line["e2e"] = e2e
        if pre:
            line["precheck"] = pre
        if two_pass:
            line["two_pass"] = two_pass
        if world == 1 and extras:
            line["other_kernels"] = other_kernels(eng, torch, ctx, vo, N, D, L, peak, not args.no_cpu_baseline)
    if extras and not args.no_other_workloads:
        # next to the headline's buffers (2.6 GB): the chain product is 20 GB per GPU, cfg5 2000x2000 16 GB
        ow = other_workloads(eng, torch, dist, dev, rank, world, comm, peak, args.chain_d)
        if line is not None:
            line["other_workloads"] = ow
    # last, so that its heat and power state do not colour the other measurements
    if extras and args.sustain_s > 0:
        # the same step loop for >= sustain_s seconds: does the figure survive sustained streaming?
        per_chunk = max(50, int(0.25 / max(1e-6, main["total_ms"] * 1e-3 / K)))
        sampler = ClockSampler(local, period_s=0.005, with_power=True)
        sampler.start()
        barrier()
        step_no[0] = 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_begin = time.perf_counter()
        e0.record()
        n_steps = 0
        while True:
            for _ in range(per_chunk):
                step_device(final=False, fused_step=fused)
            n_steps += per_chunk
            stream.synchronize()
            go = torch.tensor([1 if time.perf_counter() - t_begin < args.sustain_s else 0], dtype=torch.int64, device=dev)
            if world > 1:
                dist.all_reduce(go, op=dist.ReduceOp.MAX)      # every rank runs the same number of steps
            if int(go.item()) == 0:
                break
        step_device(final=True, fused_step=fused)
        n_steps += 1
        e1.record()
        barrier()
        t_end = time.perf_counter()
        s_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(s_ms, op=dist.ReduceOp.MAX)
        check_counts("after the sustained run")
        sustained = {"seconds": float(s_ms.item()) * 1e-3, "steps": n_steps,
                     "value": blocks_per_step * n_steps / (float(s_ms.item()) * 1e-3), "unit": UNIT,
                     "ms_per_step": float(s_ms.item()) / n_steps, "clocks": sampler.stop(t_begin, t_end),
                     "bytes_through_hbm_per_gpu": n_steps * P * T1 * T2 * bytes_per_block * (1 if fused else 2),
                     "note": "same loop as `value` (host synchronises every %d steps to read the clock)" % per_chunk}
    if sustained and line is not None:
        line["sustained"] = sustained
    if rank == 0:
        if world == 1 and extras and args.workload == "cfg2" and not (args.t1 or args.t2):
            torch.cuda.synchronize()
            line["e2e_cpp"] = cpp_e2e(P, K)
        if world == 1 and not args.no_cpu_baseline:
            # the reference overflows its int counters above 131,080 blocks at N=16383 (SURVEY hazard 4): the CPU
            # sample always uses the workload's own sizes, whatever --t1/--t2 say
            line["cpu_baseline"] = cpu_baseline(N, D, *WORKLOADS[args.workload][2:4])
        print(json.dumps(line), flush=True)
    if dump:
        write_outputs(args.dump_outputs, dump, rank, world)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def run_chain(args):
    """cfg4: x = a_shard * b (1M blocks), y = x * d (1e6*chain_d blocks), decrypt(y) with the cross-GPU exchange.
    --mode fused: the second product and its decrypt (and the exchange) are ONE kernel."""
    import torch
    import torch.distributed as dist
    from csgn_b200 import engine as eng

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    N, D, T1, T2, desc = WORKLOADS["cfg4"]
    Td, L = args.chain_d, words_per_block(N)
    eng.init(local)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)
    ctx = eng.Context(N, D)
    comm, exchange = connect_exchange(args, world, dev)
    fused = args.mode == "fused"
    pre = None if args.no_precheck else precheck(eng, torch, dev, rank, world, comm)
    key_pos = np.random.default_rng(7).permutation(N)[:D].astype(np.uint64)
    key = eng.SecretKey(ctx, key_pos)
    key_mask = np_key_mask(N, key_pos)

    host = {"a": planted_blocks(np.random.default_rng([1, rank]), T1, N, key_mask, 31),
            "b": planted_blocks(np.random.default_rng([2]), T2, N, key_mask, 17),
            "d": planted_blocks(np.random.default_rng([3]), Td, N, key_mask, 5)}
    # host-known truth (numpy): count((a*b)*d) = sum over ranks of count(a_shard) * count(b) * count(d)
    want = torch.tensor([np_count(host["a"], L, key_mask)], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(want)
    want = want * (np_count(host["b"], L, key_mask) * np_count(host["d"], L, key_mask))
    pinned = {k: torch.from_numpy(v.view(np.int64)).pin_memory() for k, v in host.items()}
    devt = {k: v.to(dev) for k, v in pinned.items()}
    va, vb, vd = (eng.Ciphertext.from_tensor(devt[k], ctx) for k in ("a", "b", "d"))
    x = torch.empty(T1 * T2 * L, dtype=torch.int64, device=dev)
    y = torch.empty(T1 * T2 * Td * L, dtype=torch.int64, device=dev)
    vx, vy = eng.Ciphertext.from_tensor(x, ctx), eng.Ciphertext.from_tensor(y, ctx)
    counts = torch.zeros(1, dtype=torch.int64, device=dev)
    host_counts = torch.zeros(1, dtype=torch.int64).pin_memory()

    def chain_tail(src_x, src_d):
        """y = x*d and its decrypt"""
        if fused:
            if comm is not None:
                comm.mul_push(key, src_x, src_d, out=vy, collect_n=1, device_totals_ptr=counts.data_ptr())
            else:
                key.mul_count_async(src_x, src_d, counts.data_ptr(), out=vy)
            return
        src_x.mul_into(src_d, vy)

    def step(evs=None):
        if evs:
            evs[0].record()
        va.mul_into(vb, vx)
        if evs:
            evs[1].record()
        chain_tail(vx, vd)
        if evs:
            evs[2].record()
        if not fused:
            if comm is not None:
                comm.push(key, vy, 1, counts.data_ptr())     # fold, push and collect in the one kernel
            else:
                key.count_satisfied_async(vy, counts.data_ptr())
        if evs:
            evs[3].record()
        if world > 1 and comm is None:
            dist.all_reduce(counts)
        if evs:
            evs[4].record()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    W = max(3, args.warmup)
    for _ in range(W):
        step()
    barrier()
    if not torch.equal(want, counts):
        raise SystemExit("cfg4 check failed: count((a*b)*d) %s != host-known truth %s" % (counts, want))

    K = args.steps
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(5)] for _ in range(K)]
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    launches0 = eng.launch_count()
    t_begin = time.perf_counter()
    for k in range(K):
        step(evs[k])
    barrier()
    clocks = sampler.stop(t_begin, time.perf_counter())
    launches = eng.launch_count() - launches0
    if not torch.equal(want, counts):
        raise SystemExit("cfg4 check failed after the timed region: %s != %s" % (counts, want))
    dump = sample_outputs(torch, y, L, counts, world) if args.dump_outputs else None
    phases = [sum(e[i].elapsed_time(e[i + 1]) for e in evs) for i in range(4)]
    t = torch.tensor([evs[0][0].elapsed_time(evs[K - 1][4])] + phases, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, mul1_ms, mul2_ms, dec_ms, ar_ms = (float(v) for v in t.tolist())
    out_blocks = T1 * T2 * Td                      # per GPU
    value = out_blocks * world * K / (total_ms * 1e-3)
    peak, peak_src = measured_peak_gbs()
    mul2_gbs = out_blocks * 8 * L * K / (mul2_ms * 1e-3) / 1e9

    # e2e: the three operands come from pinned host memory every step; the bit goes back
    def step_e2e():
        ha = eng.Ciphertext.from_host_ptr(pinned["a"].data_ptr(), T1, ctx)
        hb = eng.Ciphertext.from_host_ptr(pinned["b"].data_ptr(), T2, ctx)
        hd = eng.Ciphertext.from_host_ptr(pinned["d"].data_ptr(), Td, ctx)
        ha.mul_into(hb, vx)
        chain_tail(vx, hd)           # the 20 GB product is written in place: no room for two of them
        if not fused:
            if comm is not None:
                comm.push(key, vy, 1, counts.data_ptr())
            else:
                key.count_satisfied_async(vy, counts.data_ptr())
        if world > 1 and comm is None:
            dist.all_reduce(counts)
        host_counts.copy_(counts, non_blocking=True)
        stream.synchronize()
        if int(host_counts.item()) != int(want.item()):
            raise SystemExit("cfg4 e2e result differs from the host-known truth")

    e2e = None
    if not args.no_e2e:
        for _ in range(W):
            step_e2e()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            step_e2e()
        e1.record()
        barrier()
        ems = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ems, op=dist.ReduceOp.MAX)
        e2e = {"value": out_blocks * world * K / (float(ems.item()) * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": int((T1 + T2 + Td) * L * 8), "d2h_bytes_per_step": 8,
               "ms_per_step": float(ems.item()) / K,
               "path": "csgn_buf_upload x3 (pinned host) -> csgn_mul_into -> %s -> D2H count, checked every step"
                       % ("fused multiply->decrypt" if fused else "csgn_mul_into -> decrypt")}
    if rank == 0:
        kern = {"multiply_1M": {"avg_launch_us": mul1_ms * 1e3 / K},
                ("fused_multiply_decrypt_chain" if fused else "multiply_chain"):
                    {"gbs": mul2_gbs, "frac_of_peak": mul2_gbs / peak, "avg_launch_us": mul2_ms * 1e3 / K},
                "allreduce_ms_per_step": ar_ms / K}
        if not fused:
            dec_gbs = out_blocks * 8 * L * K / (dec_ms * 1e-3) / 1e9
            kern["decrypt"] = {"gbs": dec_gbs, "frac_of_peak": dec_gbs / peak, "avg_launch_us": dec_ms * 1e3 / K}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u64", "data": "synthetic",
                "config": {"workload": "cfg4: " + desc, "chain_d": Td, "blocks_per_gpu": out_blocks, "mode": args.mode,
                           "blocks_total": out_blocks * world, "product_bytes_per_gpu": out_blocks * 8 * L,
                           "l2": "no flush needed: the product (%.1f GB per GPU) is far larger than L2" % (out_blocks * 8 * L / 1e9),
                           "sharding": "left operand by block range, b and d replicated, one-word exchange per decrypt",
                           "exchange": exchange,
                           "checked": "count((a*b)*d) == numpy count(a)*count(b)*count(d) summed over ranks"},
                "roofline": {"bound": "hbm", "kernel": "mul_outer_kernel" + (" FOLD=1" if fused else ""), "achieved": mul2_gbs,
                             "peak": peak, "unit": "GB/s",
                             "frac": mul2_gbs / peak, "traffic": None, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": out_blocks * 8 * L, "avg_launch_us": mul2_ms * 1e3 / K},
                "kernels": kern, "clocks": clocks, "gpu_launches": int(launches)}
        if e2e:
            line["e2e"] = e2e
        if pre:
            line["precheck"] = pre
        if world == 1 and not args.no_cpu_baseline:
            cb = cpu_baseline(N, D, T1, T2)
            cb["sample"] += "; per-block cost of the chain is the same multiply+decrypt work"
            line["cpu_baseline"] = cb
        print(json.dumps(line), flush=True)
    if dump:
        write_outputs(args.dump_outputs, dump, rank, world)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference_arm(args)
    if args.workload == "cfg4":
        return run_chain(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
