"""The CUDA sources of the engine, compiled by g++ against tests/emu/cuda_emu.h and executed thread-for-thread
on the CPU, run a subset of the `gpu` parity tests (the same test functions, the same oracle, the same
tolerances) -- once plain and once under AddressSanitizer.

This is a check of the kernel and host SOURCE (index arithmetic, staging windows, list layout, launch
sequences, graph capture), not of the sm_100a binary: the B200 runs of the `gpu` marker remain the parity
gate.  The product library is never involved; the emulated build lives in tests/emu/_build/."""
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))

FAST = ("neighbor_build_bit_exact or per_kernel_parity_mixed_scene or wall_clamp or overflow_path or "
        "stale_grid or out_of_grid or rigid_solve_recovers or random_scatter or (prefix_sum and not 200000) or "
        "dfsph_per_kernel_parity or dfsph_kernels_on_overfull or "
        "(reproduces_the_reference_source and (blocks or walls or bodies) and not dfsph) or "
        "(fp64 and (base or close_pairs or cell_zero or win_cap or count_cut)) or loop_controls[max_iterations_1]")
ASAN = ("neighbor_build_bit_exact or per_kernel_parity_mixed_scene or wall_clamp or overflow_path or "
        "rigid_solve_recovers or random_scatter or (prefix_sum and not 200000) or dfsph_per_kernel_parity or "
        "(reproduces_the_reference_source and (walls or bodies)) or (fp64 and (base or close_pairs))")


def _run(lib, extra_env=None, select=FAST, at_least=25):
    env = dict(os.environ, SPH_EMU_LIB=lib, PYTHONPATH=ROOT)
    env.pop("SPH_B200_LIB", None)
    env.update(extra_env or {})
    cmd = [sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider", "-k", select,
           os.path.join(ROOT, "tests", "test_gpu_parity.py"), os.path.join(ROOT, "tests", "test_gpu_dfsph.py"),
           os.path.join(ROOT, "tests", "test_gpu_reference_golden.py"),
           os.path.join(ROOT, "tests", "test_gpu_kernel_edges.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    tail = res.stdout[-3000:] + res.stderr[-3000:]
    assert res.returncode == 0, tail
    m = re.search(r"(\d+) passed", res.stdout)
    assert m and int(m.group(1)) >= at_least, tail
    assert "skipped" not in res.stdout.splitlines()[-1], tail  # the emulation must actually run them
    return int(m.group(1))


def test_gpu_parity_subset_on_the_emulated_build():
    import build_emu
    lib = build_emu.build()
    _run(lib)


def test_gpu_parity_subset_under_address_sanitizer():
    import build_emu
    asan_rt = subprocess.run(["/usr/bin/gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan_rt) or not os.path.exists(asan_rt):
        pytest.skip("libasan not available")
    lib = build_emu.build(asan=True)
    _run(lib, {"LD_PRELOAD": asan_rt, "ASAN_OPTIONS": "detect_leaks=0"}, select=ASAN, at_least=17)
