"""The certFHE C++ drop-in (csgn_b200/certfhe -> libcertFHE.so).

CPU: the library exists in-tree, exports the reference's public class API and resolves
the C ABI it sits on.  GPU: the acceptance program, the one-process differential run
against the unmodified reference, and the reference's own demo programs compiled
UNMODIFIED against our headers all run on the B200."""
import json
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import sha, unhex
from csgn_b200 import build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "bin")
DEMOS = os.path.join(ROOT, "build", "dropin", "bin")


def _run(path, timeout=600):
    return subprocess.run([path], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=timeout)


def _ref_built():
    return os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libcertfhe_ref.so"))


def _stored_cases():
    """The reference's outputs on the golden cases (tests/golden/make_golden.py)."""
    with open(os.path.join(ROOT, "tests", "golden", "csgn_golden.json")) as f:
        return json.load(f)["cases"]


def _dropin_on_stored_inputs(exe, mode, cases, env=None):
    """tests/cpp/dropin_golden.cpp on the stored cases' inputs: {observable: printed value} per case."""
    lines = [str(len(cases))] + [" ".join(str(x) for x in [c["N"], c["D"], c["seed"], len(c["bits_a"]), len(c["bits_b"])]
                                          + c["bits_a"] + c["bits_b"] + c["key"]) for c in cases]
    r = subprocess.run([exe, mode], input="\n".join(lines) + "\n", stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stdout[-3000:]
    out = []
    for line in r.stdout.splitlines():
        name, _, rest = line.partition(" ")
        if name == "case":
            out.append({})
        elif out:
            out[-1][name] = rest
    assert len(out) == len(cases), r.stdout[-3000:]
    return out, r.stdout


def _check_host_side(c, o):
    nums = lambda s: np.array([int(x) for x in s.split()], dtype=np.uint64)
    assert [int(x) for x in o["context"].split()] == c["context"] and int(o["sk_size"]) == c["sk_size"]
    perm = nums(o["perm"])
    assert sha(perm) == c["perm_sha256"] and [int(x) for x in perm[:16]] == c["perm_head"]
    if "perm" in c:
        assert [int(x) for x in perm] == c["perm"]
    assert sha(nums(o["perm_inverse"])) == c["perm_inverse_sha256"]
    assert np.array_equal(nums(o["perm_compose"]), np.arange(c["N"], dtype=np.uint64)) == c["perm_compose_is_identity"]
    assert [int(x) for x in o["permuted_key"].split()] == c["permuted_key"]


def _check_evaluation(c, o):
    L = c["L"]
    assert o["enc_a"] == c["enc_a"] and o["enc_b"] == c["enc_b"]        # encryption in the reference's rand() order
    prod, summ = unhex(o["mul"]), unhex(o["add"])
    assert prod.size == c["mul_len"] and sha(prod) == c["mul_sha256"] and sha(unhex(o["mul_bitlen"])) == c["mul_bitlen_sha256"]
    assert np.array_equal(prod[:2 * L], unhex(c["mul_head"])) and np.array_equal(prod[-L:], unhex(c["mul_tail"]))
    if "mul" in c:
        assert o["mul"] == c["mul"]
    assert summ.size == c["add_len"] and sha(summ) == c["add_sha256"] and sha(unhex(o["add_bitlen"])) == c["add_bitlen_sha256"]
    assert [int(x) for x in o["dec"].split()] == [c["dec_a"], c["dec_b"], c["dec_mul"], c["dec_add"]]
    strict_bl = [int(x) for x in o["permute_strict_bitlen"].split()]
    assert len(strict_bl) == c["permute_strict_len"] and o["permute_strict"] == c["permute_strict"]
    assert strict_bl == c["permute_strict_bitlen"] if L <= 32 else sha(np.array(strict_bl, dtype=np.uint64)) == c["permute_strict_bitlen"]
    assert sha(unhex(o["permute_each_block"])) == c["permute_each_block_sha256"]
    if "permute_each_block" in c:
        assert o["permute_each_block"] == c["permute_each_block"]
    assert int(o["dec_permuted"]) == c["dec_permuted"] and int(o["ct_size_one_block"]) == c["ct_size_one_block"]


def test_libcertfhe_exports_the_reference_api():
    path = build.libcertfhe_path()
    assert os.path.exists(path), "run `python -m csgn_b200.build`"
    syms = subprocess.run(["nm", "-DC", "--defined-only", path], stdout=subprocess.PIPE, text=True).stdout
    wanted = [
        "certFHE::Library::initializeLibrary()",
        "certFHE::Context::Context(unsigned long, unsigned long)",
        "certFHE::Context::getDefaultN() const",
        "certFHE::Plaintext::Plaintext(int)",
        "certFHE::SecretKey::SecretKey(certFHE::Context const&)",
        "certFHE::SecretKey::encrypt(certFHE::Plaintext&)",
        "certFHE::SecretKey::decrypt(certFHE::Ciphertext&)",
        "certFHE::SecretKey::applyPermutation(certFHE::Permutation const&)",
        "certFHE::SecretKey::setKey(unsigned long*, unsigned long)",
        "certFHE::Ciphertext::Ciphertext(unsigned long const*, unsigned long const*, unsigned long, certFHE::Context const&)",
        "certFHE::Ciphertext::operator+(certFHE::Ciphertext const&) const",
        "certFHE::Ciphertext::operator+=(certFHE::Ciphertext const&)",
        "certFHE::Ciphertext::operator*(certFHE::Ciphertext const&) const",
        "certFHE::Ciphertext::operator*=(certFHE::Ciphertext const&)",
        "certFHE::Ciphertext::operator=(certFHE::Ciphertext const&)",
        "certFHE::Ciphertext::applyPermutation(certFHE::Permutation const&)",
        "certFHE::Ciphertext::applyPermutation_inplace(certFHE::Permutation const&)",
        "certFHE::Ciphertext::getValues() const",
        "certFHE::Ciphertext::getBitlen() const",
        "certFHE::Ciphertext::size()",
        "certFHE::Permutation::Permutation(certFHE::Context const&)",
        "certFHE::Permutation::getInverse()",
        "certFHE::Permutation::operator+(certFHE::Permutation const&) const",
        "certFHE::operator<<(std::ostream&, certFHE::Ciphertext const&)",
        "certFHE::Timer::stopAndPrint()",
        "certFHE::Helper::exists(unsigned long const*, unsigned long, unsigned long)",
    ]
    for w in wanted:
        assert w in syms, w
    # it computes nothing itself: the evaluation entry points are undefined here and come from libcsgn
    undef = subprocess.run(["nm", "-D", "--undefined-only", path], stdout=subprocess.PIPE, text=True).stdout
    for f in ("csgn_mul", "csgn_mul_decrypt_deferred", "csgn_concat", "csgn_concat_lazy", "csgn_append", "csgn_decrypt_deferred",
              "csgn_permute", "csgn_buf_upload_copy"):
        assert re.search(r"\bU %s\b" % f, undef), f
    ldd = subprocess.run(["ldd", path], stdout=subprocess.PIPE, text=True).stdout
    assert "libcsgn.so" in ldd and "not found" not in ldd


def test_cpp_test_programs_are_built():
    assert os.path.exists(os.path.join(BIN, "accept_demos"))


def test_host_side_classes_match_the_reference_without_a_gpu():
    """Context / Plaintext / Permutation / SecretKey host logic, one process with the unmodified reference; where that
    build is absent, the same classes on the stored reference cases against the reference's stored outputs."""
    exe = os.path.join(BIN, "host_vs_reference")
    if not os.path.exists(exe) or not _ref_built():
        cases = _stored_cases()
        for c, o in zip(cases, _dropin_on_stored_inputs(os.path.join(BIN, "dropin_golden"), "host", cases)[0]):
            _check_host_side(c, o)
        return
    r = _run(exe)
    assert r.returncode == 0, r.stdout[-4000:]
    assert "host-side classes identical to the reference" in r.stdout


@pytest.mark.gpu
def test_acceptance_program():
    r = _run(os.path.join(BIN, "accept_demos"))
    assert r.returncode == 0, r.stdout[-4000:]
    out = r.stdout
    assert "Dec ( Enc (1) + Enc (0) ) = 1" in out
    assert "Dec ( Enc (1) * Enc (0) ) = 0" in out
    assert " Dec ( Enc ( 1 ) ) = 1" in out
    assert "Fresh ciphertext size: 352 bytes" in out and "After addition ciphertext size: 672 bytes" in out
    assert "Secret key size: 144 bytes" in out


@pytest.mark.gpu
def test_differential_against_the_unmodified_reference():
    """The drop-in and the unmodified reference in one process; where that build is absent, every observable of the
    drop-in on the stored reference cases against the reference's stored outputs."""
    exe = os.path.join(BIN, "diff_vs_reference")
    if not os.path.exists(exe) or not _ref_built():
        cases = _stored_cases()
        for c, o in zip(cases, _dropin_on_stored_inputs(os.path.join(BIN, "dropin_golden"), "all", cases)[0]):
            _check_host_side(c, o)
            _check_evaluation(c, o)
        return
    r = _run(exe, timeout=1200)
    assert r.returncode == 0, r.stdout[-4000:]
    assert "identical to the reference on every observable" in r.stdout
    assert "config2 N=1247 1000x1000 -> 1000000 blocks" in r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("demo,lines", [
    ("tester_basic_operations", ["Dec ( Enc (1) + Enc (0) ) = 1", "Dec ( Enc (1) * Enc (0) ) = 0"]),
    ("tester_permutations", [" Dec ( Enc ( 1 ) ) = 1"]),
    ("tester_timings", ["N= 1247", "D= 16", "S= 38", "Security(lambda)= 120", "Secret key size: 144 bytes",
                        "Fresh ciphertext size: 352 bytes", "After multiplication ciphertext size: 352 bytes",
                        "After addition ciphertext size: 672 bytes"]),
])
def test_unmodified_reference_demos_run_on_the_dropin(demo, lines):
    exe = os.path.join(DEMOS, demo)
    if not os.path.exists(exe):
        pytest.skip("reference demos are compiled only where /root/reference was present")
    r = _run(exe)
    assert r.returncode == 0, r.stdout[-4000:]
    for line in lines:
        assert line in r.stdout, (line, r.stdout[-2000:])


@pytest.mark.gpu
def test_cpp_api_sharded_over_the_gpus_of_the_box(tmp_path):
    """tests/cpp/sharded_demo.cpp: one process per GPU started by a plain loop (no torch, no MPI); the ranks meet through
    a directory, Ciphertext::shard() + shard-local products + SecretKey::decrypt with the exchange inside the fold
    kernel.  One process on a one-GPU box (same code path, own mailbox only), min(4, n) processes otherwise."""
    import torch
    exe = os.path.join(BIN, "sharded_demo")
    assert os.path.exists(exe)
    world = max(1, min(4, torch.cuda.device_count()))
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), LOCAL_RANK=str(r), WORLD_SIZE=str(world), CSGN_RENDEZVOUS_DIR=str(tmp_path),
                   CSGN_JOB_TAG="pytest%d" % os.getpid(), CSGN_PEER_TIMEOUT_MS="20000")
        procs.append(subprocess.Popen([exe], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = []
    for p in procs:
        try:
            out, _ = p.communicate(timeout=600)
        except subprocess.TimeoutExpired:
            p.kill()
            out, _ = p.communicate()
        outs.append((p.returncode, out))
    for r, (rc, out) in enumerate(outs):
        assert rc == 0, "rank %d:\n%s" % (r, out[-3000:])
        assert "sharded_demo rank %d/%d: all checks passed" % (r, world) in out
    assert not [f for f in os.listdir(tmp_path) if f.endswith(".handle")]      # every rank removed its handle file


def test_host_classes_clean_under_sanitizers(tmp_path):
    """The host-side classes (Context, Plaintext, Permutation, SecretKey key handling, encrypt, Timer, Helper) built with
    -fsanitize=address,undefined and driven by the differential program: no report, same verdict (SURVEY.md 5: the
    reference itself trips ASan/UBSan in several places -- App. B; this port must not).  CPU only.  Where the reference's
    headers and build are absent, the driver of the stored reference cases (host mode) is built instead and its output
    checked against the reference's stored outputs."""
    ref_hdr = os.path.join(build.REFERENCE, "src", "certFHE.h")
    ref_lib = os.path.join(ROOT, "oracle", "_ref", "libcertfhe_ref.so")
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0:protect_shadow_gap=0:halt_on_error=1",
               UBSAN_OPTIONS="halt_on_error=1:print_stacktrace=1")
    if not (os.path.exists(ref_hdr) and os.path.exists(ref_lib)):
        exe = str(tmp_path / "dropin_golden_asan")
        cmd = ["g++", "-O1", "-g", "-std=c++11", "-fsanitize=address,undefined", "-fno-omit-frame-pointer", "-w",
               "-I" + build.CERTFHE, "-I" + build.INCLUDE, "-o", exe, os.path.join(ROOT, "tests", "cpp", "dropin_golden.cpp"),
               os.path.join(build.CERTFHE, "host_types.cpp"), os.path.join(build.CERTFHE, "device_types.cpp"),
               "-L" + build.LIBDIR, "-lcsgn", "-Wl,-rpath," + build.LIBDIR]
        c = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
        assert c.returncode == 0, c.stdout[-3000:]
        cases = _stored_cases()
        outs, text = _dropin_on_stored_inputs(exe, "host", cases, env=env)
        assert "AddressSanitizer" not in text and "runtime error" not in text, text[-3000:]
        for case, o in zip(cases, outs):
            _check_host_side(case, o)
        return
    exe = str(tmp_path / "host_vs_reference_asan")
    cmd = ["g++", "-O1", "-g", "-std=c++11", "-fsanitize=address,undefined", "-fno-omit-frame-pointer", "-w",
           "-I" + build.CERTFHE, "-I" + build.INCLUDE, '-DCSGN_REFERENCE_HEADER="%s"' % ref_hdr, "-o", exe,
           os.path.join(ROOT, "tests", "cpp", "host_vs_reference.cpp"),
           os.path.join(build.CERTFHE, "host_types.cpp"), os.path.join(build.CERTFHE, "device_types.cpp"),
           "-L" + build.LIBDIR, "-lcsgn", "-L" + os.path.dirname(ref_lib), "-lcertfhe_ref", "-pthread",
           "-Wl,-rpath," + build.LIBDIR, "-Wl,-rpath," + os.path.dirname(ref_lib)]
    c = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert c.returncode == 0, c.stdout[-3000:]
    r = subprocess.run([exe], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:]
    assert "identical to the reference" in r.stdout
    assert "AddressSanitizer" not in r.stdout and "runtime error" not in r.stdout, r.stdout[-3000:]
