"""CPU-only: the direct convolution without a GPU.

- tests/test_gpu_conv2d_direct.py itself runs (-m gpu) against the host-emulated build of the whole library
  (tests/emu_build.py: build_capi_host_emu -- capi.cu compiled by g++ over stand-ins for the CUDA runtime, kernels on host
  threads), once as it is and once under AddressSanitizer: the entry points' checks, the Python mirror and every
  expectation of that file at the sizes a CPU can run.
- The kernel alone (layers.cuh: conv2d_direct_kernel, tests/emu/conv2d_direct_emu.cpp) with the library's launch plan, in both of
  its variants (input staged in shared memory, or read from global memory), against the oracle's im2col convolution bit
  for bit, on one block and on a grid-stride loop over several."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import oracle as O

from emu_build import asan_env, build_capi_host_emu, build_emu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GPU_FILE = os.path.join(ROOT, "tests", "test_gpu_conv2d_direct.py")


def _run_gpu_file(so, extra_env):
    env = dict(os.environ, LASER_B200_LIB=so, LASER_B200_EMU="1", PYTHONPATH=ROOT, **extra_env)
    out = subprocess.run([sys.executable, "-m", "pytest", GPU_FILE, "-m", "gpu", "-q", "-p", "no:cacheprovider"], cwd=ROOT, env=env,
                         capture_output=True, text=True, timeout=1800)
    tail = out.stdout[-3000:] + out.stderr[-2000:]
    assert out.returncode == 0 and "failed" not in out.stdout, tail
    m = re.search(r"(\d+) passed", out.stdout)
    assert m and int(m.group(1)) >= 50, tail


def test_gpu_file_against_the_host_emulated_library():
    _run_gpu_file(build_capi_host_emu(), {})


def test_gpu_file_against_the_host_emulated_library_under_asan():
    env = asan_env()
    _run_gpu_file(build_capi_host_emu(asan=True), env)


# ---- the kernel alone ---------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emu():
    so = build_emu("conv2d_direct_emu", ["layers.cuh", "simt_epilogue.cuh"])
    L = ctypes.CDLL(so)
    i64, vp, ci = ctypes.c_int64, ctypes.c_void_p, ctypes.c_int
    L.emu_conv2d_direct.restype = ci
    L.emu_conv2d_direct.argtypes = [vp, vp, vp, i64, i64 * 12, vp, ci, ci, ci]
    return L


def ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


def run(emu, inp, ker, ishape, kshape, padding, strides, grid, unstaged):
    o = O.conv2d_out_shape(ishape, kshape, padding, strides)
    geom = (ctypes.c_int64 * 12)(ishape[1], ishape[2], ishape[3], kshape[0], kshape[2], kshape[3], padding[0], padding[1],
                                 strides[0], strides[1], o[2], o[3])
    out = np.full(int(np.prod(o)) + 64, np.nan, np.float32)
    staged = emu.emu_conv2d_direct(ptr(out), ptr(inp), ptr(ker), ishape[0], geom, None, 0, grid, int(not unstaged))
    assert staged == (0 if unstaged else 1)
    assert np.isnan(out[-64:]).all()    # nothing written past the output
    return out[:-64].reshape(o)


CASES = [
    ((2, 3, 17, 19), (4, 3, 3, 3), (1, 1), (1, 1)),
    ((2, 2, 15, 18), (3, 2, 3, 3), (0, 1), (2, 1)),
    ((1, 2, 40, 50), (11, 2, 3, 3), (1, 2), (1, 1)),      # two pixel tiles, two channel groups
    ((1, 64, 7, 9), (9, 64, 3, 3), (1, 1), (1, 1)),       # K = 576: a block boundary inside a channel
    ((1, 128, 5, 6), (17, 128, 3, 3), (1, 1), (2, 1)),    # K = 1152, three channel groups
    ((2, 3, 12, 12), (5, 3, 5, 5), (2, 2), (2, 2)),
]


@pytest.mark.parametrize("unstaged", [False, True], ids=["staged", "global"])
@pytest.mark.parametrize("grid", [1, 3, 0], ids=["grid1", "grid3", "one_block_per_tile"])
@pytest.mark.parametrize("ishape,kshape,padding,strides", CASES)
def test_kernel_bit_identical_to_oracle_im2col(emu, ishape, kshape, padding, strides, grid, unstaged):
    inp = O.fill_uniform_f32(int(np.prod(ishape)), 3, -1, 1).reshape(ishape)
    ker = O.fill_uniform_f32(int(np.prod(kshape)), 4, -1, 1).reshape(kshape)
    got = run(emu, inp, ker, ishape, kshape, padding, strides, grid, unstaged)
    want = O.conv2d_im2col(inp, ishape, ker, kshape, padding, strides)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
