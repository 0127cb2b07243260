"""The `-m gpu` parity tests, run on the CPU box against the product's own C ABI built for the SIMT emulator
(tests/simt: diskann_b200.cu with its launches rewritten by cu2cpp.py + every kernel source + a fake CUDA runtime ->
tests/simt/_build/libdiskann_b200_emu.so).  Host logic (plans, growth retries, the scan operator's suspend / resume,
argument validation, the plain-layout routing) and kernel logic are exercised TOGETHER by the very tests the B200 box
runs, including the opt-in ones for code that has not been on hardware yet.

It is a logic check, not a substitute for hardware: no memory model, no timing, and the emulated library is a test
artifact that the package never looks for (conftest.lib_built loads it by explicit path under DANN_EMULATE=1).
Runs in a subprocess so that the emulated library never shares a process with the tests of the real one."""
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(files, extra_env=None, workers=4, timeout=1500, asan=False):
    env = dict(os.environ)
    env.update({"DANN_EMULATE": "1", "SIMT_SM_COUNT": "8"})
    env.update(extra_env or {})
    # build once here: the xdist workers would otherwise race on the same output file
    sys.path.insert(0, os.path.join(ROOT, "tests", "simt"))
    import build_emu
    build_emu.build_abi(asan=asan)
    if asan:    # python itself is not instrumented: the runtime has to come first in the link order
        env.update({"DANN_EMULATE_ASAN": "1", "LD_PRELOAD": build_emu.libasan(),
                    "ASAN_OPTIONS": "detect_leaks=0:detect_stack_use_after_return=0:abort_on_error=1"})
    cmd = [sys.executable, "-m", "pytest", "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider", "-n", str(workers)] + files
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=timeout)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, tail
    m = re.search(r"(\d+) passed", r.stdout)
    assert m, tail
    return int(m.group(1)), r.stdout


def test_gpu_parity_suite_passes_under_emulation():
    passed, out = _run(["tests/test_gpu_parity.py", "tests/test_zz_c_harness_gpu.py", "tests/test_zz_d_build_small_gpu.py",
                        "tests/test_zz_e_coalescer_gpu.py", "tests/test_zz_f_fuzz_gpu.py",
                        "tests/test_zz_g_oom_paths_emulated.py", "tests/test_zz_h_two_rank_emulated.py",
                        "tests/test_zz_l_wide_codes_gpu.py"])
    assert passed >= 97 + 45 and "skipped" not in out.splitlines()[-1], out[-500:]


def test_two_replica_group_under_emulation():
    """dann_group with two (fake) devices: slices, worker threads, rows in query order, label keys, error path."""
    passed, out = _run(["tests/test_zz_i_group_gpu.py"], {"SIMT_FAKE_DEVICES": "2"}, workers=1)
    assert passed == 3 and "skipped" not in out.splitlines()[-1], out[-500:]


def test_plain_storage_and_one_sync_gettuple_pass_under_emulation():
    """The plain storage layout and the one-synchronisation amgettuple, through the real host code."""
    passed, out = _run(["tests/test_zz_plain_gpu.py"])
    assert passed >= 38 and "skipped" not in out.splitlines()[-1], out[-500:]


def test_edge_case_fuzz_with_the_lean_kernel_tiny_heaps_and_retries():
    """DANN_SEARCH_KERNEL=3 forces the lean warp-per-query kernel (small batches default to the two-warp one)."""
    passed, _ = _run(["tests/test_zz_f_fuzz_gpu.py"], {"DANN_FUZZ_SEEDS": "120", "DANN_SEARCH_KERNEL": "3", "DANN_SEARCH_HS": "16",
                                                       "DANN_DEBUG_SHRINK": "8", "SIMT_SCHED": "2", "SIMT_SM_COUNT": "2"})
    assert passed == 120 + 12     # the seeds + the four reference-KAT cases and the eight medium cases in the same file
    passed, _ = _run(["tests/test_zz_f_fuzz_gpu.py"], {"DANN_FUZZ_SEEDS": "120", "DANN_SEARCH_KERNEL": "1",
                                                       "DANN_SEARCH_BITMAP": "0", "SIMT_SCHED": "1"})
    assert passed == 120 + 12     # the seeds + the four reference-KAT cases and the eight medium cases in the same file


def test_address_sanitizer_finds_nothing_in_host_code_or_kernels():
    """The emulated ABI built with -fsanitize=address: every "device" buffer is a red-zoned host allocation, so an
    out-of-bounds access by a kernel (or by the host code around it) aborts the run.  Edge-case fuzz with the measured
    kernels and with the lean kernel forced on tiny heap tops, forced growth and the one-synchronisation gettuple."""
    if not os.path.exists(__import__("subprocess").run(["gcc", "-print-file-name=libasan.so"], capture_output=True,
                                                       text=True).stdout.strip()):
        pytest.skip("libasan not installed")
    passed, _ = _run(["tests/test_zz_f_fuzz_gpu.py"], {"DANN_FUZZ_SEEDS": "80"}, asan=True)
    assert passed == 80 + 12
    passed, _ = _run(["tests/test_zz_f_fuzz_gpu.py"],
                     {"DANN_FUZZ_SEEDS": "80", "DANN_SEARCH_KERNEL": "3", "DANN_SEARCH_HS": "16", "DANN_DEBUG_SHRINK": "8",
                      "DANN_SCAN_FUSED": "1", "SIMT_SCHED": "2", "SIMT_SM_COUNT": "2"}, asan=True)
    assert passed == 80 + 12


def test_one_synchronisation_gettuple_passes_under_emulation():
    """amgettuple with a single host synchronisation per row is the default (DANN_SCAN_FUSED=1); the step-by-step path
    (DANN_SCAN_FUSED=0) stays covered here."""
    passed, _ = _run(["tests/test_gpu_parity.py", "-k", "scan or gettuple or counters or null or empty"],
                     {"DANN_SCAN_FUSED": "0"})
    assert passed >= 2
    passed, _ = _run(["tests/test_zz_f_fuzz_gpu.py"], {"DANN_SCAN_FUSED": "0", "DANN_DEBUG_SHRINK": "8", "DANN_FUZZ_SEEDS": "120"})
    assert passed == 120 + 12     # the seeds + the four reference-KAT cases and the eight medium cases in the same file


@pytest.mark.parametrize("sched", ["2"])
def test_parity_under_other_lane_schedules(sched):
    """Descending and shuffled fiber order (exposes missing __syncwarp()s) on a slice of the parity suite."""
    passed, _ = _run(["tests/test_gpu_parity.py", "-k", "batch_768d or scan_operator or labeled or counters"],
                     {"SIMT_SCHED": sched})
    assert passed >= 5
