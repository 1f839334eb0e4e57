"""CPU-only: the `-m gpu` test files themselves, against the host-emulated library.

The layer tests themselves (tests/test_gpu_zlayers.py) and with them the Python mirror of the
layer entry points (laser_b200/layers.py, tensor.py) run against the host-emulated build of the whole
library (tests/emu_build.py: build_capi_host_emu -- capi.cu compiled by g++ over stand-ins for the CUDA
runtime, kernels on host threads).  Sizes that would take too long on host threads are skipped there.
The emulated build is loaded only in the subprocess below (LASER_B200_LIB); the product never sees it."""
import os
import re
import subprocess
import sys

import pytest

from emu_build import build_capi_host_emu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_layer_tests_pass_against_the_host_emulated_library():
    so = build_capi_host_emu()
    env = dict(os.environ, LASER_B200_LIB=so, LASER_B200_EMU="1", PYTHONPATH=ROOT)
    out = subprocess.run([sys.executable, "-m", "pytest", os.path.join(ROOT, "tests", "test_gpu_zlayers.py"), "-m", "gpu", "-q",
                          "-p", "no:cacheprovider"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    tail = out.stdout[-3000:] + out.stderr[-2000:]
    assert out.returncode == 0, tail
    m = re.search(r"(\d+) passed", out.stdout)
    assert m and int(m.group(1)) >= 50, tail
    assert "failed" not in out.stdout, tail


FAST = "golden or simt_bit_exact or degenerate or auto_path or tensor_contract or env_selects or bf16 or host_pointer_entry_strided or tf32x1"


def _run_gpu_files(files, extra, timeout):
    so = build_capi_host_emu()
    env = dict(os.environ, LASER_B200_LIB=so, LASER_B200_EMU="1", PYTHONPATH=ROOT)
    out = subprocess.run([sys.executable, "-m", "pytest"] + [os.path.join(ROOT, "tests", f) for f in files] +
                         ["-m", "gpu", "-q", "-p", "no:cacheprovider"] + extra, cwd=ROOT, env=env, capture_output=True, text=True,
                         timeout=timeout)
    tail = out.stdout[-3000:] + out.stderr[-2000:]
    assert out.returncode == 0 and "failed" not in out.stdout, tail
    return int(re.search(r"(\d+) passed", out.stdout).group(1))


def test_parity_file_subset_against_the_host_emulated_library():
    """tests/test_gpu_parity.py is backend-neutral (tests/backend.py): the same assertions the B200 has to
    meet -- known-answer vectors on every path and dtype, bit-exactness of the exact kernel, bf16, the
    host-pointer entry, dispatch, the Tensor contract -- are checked here on the CPU build.  A fast
    subset by default; LASER_B200_EMU_FULL=1 runs the whole parity, fuzz, pre-packed, fused-epilogue,
    epilogue-path and few-rows / GEMV files (about 12 minutes on 8 cores, sizes too large for the CPU build skipped)."""
    assert _run_gpu_files(["test_gpu_parity.py"], ["-k", FAST], 1500) >= 50


# fast subsets of the epilogue-path and few-rows / GEMV files: the fused epilogue on the exact and few-rows kernels and on the
# split-K reduce (100 x 520 x 1024 splits in two under the emulation's default 8 SMs), the few-rows kernels, GEMV below
# 20000 rows
EPILOGUE_FAST = "exact_kernel_epilogue or split_single_k1024-col-relu or split_single_k1024-row-tanh or planner"
FEW_ROWS_FAST = "kernel_selection or random or batched or host_pointer or (gemv and M1031)"


def test_epilogue_and_few_rows_files_subset_against_the_host_emulated_library():
    """tests/test_gpu_epilogue_paths.py and tests/test_gpu_few_rows_gemv.py: a fast subset by default (the whole files with
    LASER_B200_EMU_FULL=1 below)"""
    assert _run_gpu_files(["test_gpu_epilogue_paths.py"], ["-k", EPILOGUE_FAST], 1500) >= 60
    assert _run_gpu_files(["test_gpu_few_rows_gemv.py"], ["-k", FEW_ROWS_FAST], 1500) >= 60


def test_f16x3_mode_file_against_the_host_emulated_library():
    """tests/test_gpu_zy_f16x3_mode.py (the default fp32 mode) in full, minus the sizes skipped for the CPU build"""
    assert _run_gpu_files(["test_gpu_zy_f16x3_mode.py"], [], 1500) >= 40


@pytest.mark.skipif(os.environ.get("LASER_B200_EMU_FULL", "0") != "1", reason="about 12 minutes; set LASER_B200_EMU_FULL=1")
def test_whole_parity_and_fuzz_files_against_the_host_emulated_library():
    assert _run_gpu_files(["test_gpu_parity.py", "test_gpu_fuzz.py", "test_gpu_prepacked.py", "test_gpu_fused_epilogue.py",
                           "test_gpu_epilogue_paths.py", "test_gpu_few_rows_gemv.py"], [], 9000) >= 850
