"""bench.py prints ONE JSON line with the keys the driver reads.  CPU: the reference arm (the unmodified reference
on the host cores, oracle/_ref).  GPU: our arm at a few steps."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}


def _run(args, timeout):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=timeout, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line():
    from oracle import pyoracle
    if not pyoracle.ref_available():
        pytest.skip("oracle/_ref not built here")
    d = _run(["--impl", "reference", "--steps", "1", "--warmup", "0"], 600)
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"] == "ctxt-mul+decrypt output blocks/s" and d["unit"] == "blocks/s" and d["higher_is_better"] is True
    cb = d["cpu_baseline"]
    assert cb["kind"] == "reference" and cb["cores"] >= 1 and cb["value"] == d["value"] > 1e4 and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "blocks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["config"]["workload"].startswith("cfg2")


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_bench_numpy_restatement_matches_the_oracle():
    """bench.py checks the GPU with its OWN numpy restatement (precheck, host-known truth); that restatement is pinned
    to the oracle here, on CPU, for three contexts incl. odd L."""
    import numpy as np
    from oracle.pyoracle import Oracle, random_blocks, random_key
    bench = _bench_module()
    o = Oracle()
    rng = np.random.default_rng(31)
    for N, D in ((1247, 3), (191, 2), (16383, 4), (128, 2)):
        L = bench.words_per_block(N)
        s = random_key(rng, N, D)
        mask = bench.np_key_mask(N, s)
        a = bench.planted_blocks(rng, 23, N, mask, k=7)
        b = bench.planted_blocks(rng, 9, N, mask, k=4)
        assert not np.any(a.reshape(-1, L)[:, -1] & ~np.uint64(((1 << 64) - 1) << ((64 - N % 64) % 64) & ((1 << 64) - 1)))   # pad bits stay zero
        prod = bench.np_mul(a, b, L)
        assert np.array_equal(prod, o.mul(a, b, L))
        assert bench.np_count(a, L, mask) == o.count_satisfied(a, N, s) >= 7
        assert bench.np_count(prod, L, mask) == o.count_satisfied(prod, N, s) == bench.np_count(a, L, mask) * bench.np_count(b, L, mask)
        perm = rng.permutation(N).astype(np.uint64)
        assert np.array_equal(bench.np_permute(prod, N, perm), o.permute_all(prod, N, perm))


@pytest.mark.gpu
def test_our_arm_line():
    d = _run(["--steps", "3", "--warmup", "3", "--no-cpu-baseline", "--sustain-s", "0.3"], 1200)
    assert BASE_KEYS <= set(d) and "impl" not in d
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] >= 3 and d["scaling"] == "weak" and d["dtype"] == "u64"
    assert d["value"] > 1e10 and d["config"]["workload"].startswith("cfg2") and d["config"]["mode"].startswith("fused")
    roof = d["roofline"]
    assert roof["bound"] == "hbm" and roof["unit"] == "GB/s" and roof["peak"] > 1000
    assert abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-9 and roof["achieved"] > 3000
    assert roof["algorithmic_bytes_per_launch"] == 160000000
    e2e = d["e2e"]
    assert e2e["value"] > 1e10 and e2e["h2d_bytes_per_step"] == 16 * 2000 * 160 and e2e["d2h_bytes_per_step"] == 128
    assert d["gpu_launches"] == 3 * 16                       # one fused multiply->decrypt kernel per pair, nothing else
    assert d["precheck"]["passed"] is True and len(d["precheck"]["cases"]) == 3
    two = d["two_pass"]                                      # the round-1 step (separate kernels) on the same buffers
    assert two["gpu_launches"] == 3 * 32 and 5e9 < two["value"] < d["value"]
    assert d["sustained"]["seconds"] >= 0.3 and d["sustained"]["value"] > 1e10
    extra = d["other_kernels"]                               # permute and add, reported beside the headline
    assert "error" not in extra and extra["permute"]["blocks_per_s"] > 5e9 and extra["add"]["gbs_read_plus_write"] > 3000
    ow = d["other_workloads"]                                # BASELINE.json configs[3] and [4]
    for name in ("cfg5_300x300", "cfg5_2000x2000", "cfg4_chain"):
        assert "error" not in ow[name], ow[name]
    assert ow["cfg4_chain"]["blocks_per_gpu"] == 125000000 and ow["cfg4_chain"]["multiply_chain"]["frac_of_peak"] > 0.8
    assert ow["cfg5_2000x2000"]["multiply"]["frac_of_peak"] > 0.8
    cpp = d["e2e_cpp"]                                       # the same step through libcertFHE.so
    assert cpp.get("checked") is True and cpp["value"] > 1e9, cpp
    assert d["clocks"]["sm_mhz"] and not (set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"})


@pytest.mark.gpu
def test_two_pass_mode_line():
    d = _run(["--steps", "3", "--warmup", "3", "--no-cpu-baseline", "--no-extras", "--mode", "two-pass"], 600)
    assert d["config"]["mode"].startswith("two-pass") and d["gpu_launches"] == 3 * 32
    assert set(d["kernels"]) >= {"multiply", "decrypt"} and d["value"] > 5e9


@pytest.mark.gpu
def test_dump_outputs(tmp_path):
    """--dump-outputs: the counts of the last timed step and a seeded sample of its products, float64, within 64 MB,
    equal to the numpy restatement on the bench's seeded inputs and identical from run to run.  One timed step: only
    the first of the two count slots is written, so the dump must take the last step's slot."""
    import numpy as np
    P = 2
    args = ["--steps", "1", "--warmup", "3", "--pairs", str(P), "--no-extras", "--no-cpu-baseline", "--no-e2e"]
    runs = []
    for i in range(2):
        d = _run(args + ["--dump-outputs", str(tmp_path / str(i))], 600)
        assert d["steps"] == 1 and d["gpu_launches"] == P
        runs.append({p.name: np.load(p) for p in (tmp_path / str(i)).iterdir()})
    out = runs[0]
    assert set(out) == {"counts.npy", "product_blocks.npy", "product_words.npy"}
    assert set(runs[1]) == set(out) and all(np.array_equal(out[k], runs[1][k]) for k in out)
    assert all(a.dtype == np.float64 for a in out.values()) and sum(a.nbytes for a in out.values()) <= 64 << 20
    bench = _bench_module()
    N, D, T1, T2, _ = bench.WORKLOADS["cfg2"]
    L = bench.words_per_block(N)
    mask = bench.np_key_mask(N, np.random.default_rng(7).permutation(N)[:D])
    halves = out["product_words.npy"].astype(np.uint64)
    words = (halves[..., 0] << np.uint64(32)) | halves[..., 1]
    blocks = out["product_blocks.npy"].astype(np.int64)
    assert words.shape == (blocks.size, L) and blocks.size > 1000
    for p in range(P):
        a = bench.planted_blocks(np.random.default_rng([1000 + p, 0]), T1, N, mask).reshape(T1, L)
        b = bench.planted_blocks(np.random.default_rng([2000 + p]), T2, N, mask).reshape(T2, L)
        assert out["counts.npy"][p] == bench.np_count(a, L, mask) * bench.np_count(b, L, mask)
        mine = blocks // (T1 * T2) == p
        ij = blocks[mine] % (T1 * T2)
        assert mine.any() and np.array_equal(words[mine], a[ij // T2] & b[ij % T2])
