"""ctypes binding of include/laser_b200.h (the C ABI is the product boundary)."""
import ctypes
import os

from . import _build

PATH_AUTO, PATH_SIMT, PATH_TF32X1, PATH_TF32X3, PATH_BF16, PATH_F16X3 = 0, 1, 2, 3, 4, 7
PATH_NAMES = {0: "auto", 1: "simt", 2: "tf32x1", 3: "tf32x3", 4: "bf16", 7: "f16x3"}
E_OK, E_INVAL, E_NODEVICE, E_CUDA, E_NOMEM, E_UNSUPPORTED = 0, 1, 2, 3, 4, 5
MAXRANK = 6

i64, f32, f64, vp = ctypes.c_int64, ctypes.c_float, ctypes.c_double, ctypes.c_void_p
i32, u64, sz = ctypes.c_int32, ctypes.c_uint64, ctypes.c_size_t


class LaserB200Error(RuntimeError):
    """Non-zero status from liblaser_b200.so (the reference's analogue: LibraryError,
    laser/cpuinfo.nim:358-359)."""

    def __init__(self, code, msg):
        super().__init__("laser_b200 error %d: %s" % (code, msg))
        self.code = code


class Epilogue(ctypes.Structure):
    _fields_ = [("bias", vp), ("bias_per_row", i32), ("activation", i32)]


ACT_NONE, ACT_RELU, ACT_TANH, ACT_SIGMOID = 0, 1, 2, 3


class TensorView(ctypes.Structure):
    _fields_ = [("rank", i32), ("dtype", i32), ("shape", i64 * MAXRANK), ("strides", i64 * MAXRANK),
                ("offset", i64), ("storage", vp)]


def _gemm_sig(scalar):
    return [i64, i64, i64, scalar, vp, i64, i64, vp, i64, i64, scalar, vp, i64, i64]


# every symbol include/laser_b200.h declares, with its ctypes signature
SIGNATURES = {
    "laser_b200_init": (ctypes.c_int, []),
    "laser_b200_shutdown": (None, []),
    "laser_b200_last_error": (ctypes.c_char_p, []),
    "laser_b200_version": (ctypes.c_int, []),
    "laser_b200_launch_count": (i64, []),
    "laser_b200_last_path": (ctypes.c_int, []),
    "laser_b200_profile_begin": (ctypes.c_int, []),
    "laser_b200_profile_end": (ctypes.c_int, [ctypes.POINTER(f64), ctypes.POINTER(i64),
                                              ctypes.POINTER(f64), ctypes.POINTER(i64)]),
    "laser_b200_set_f32_mode": (ctypes.c_int, [ctypes.c_int]),
    "laser_b200_get_f32_mode": (ctypes.c_int, []),
    "laser_b200_gemm_strided_f32": (ctypes.c_int, _gemm_sig(f32)),
    "laser_b200_gemm_strided_f64": (ctypes.c_int, _gemm_sig(f64)),
    "laser_b200_gemm_strided_i32": (ctypes.c_int, _gemm_sig(i32)),
    "laser_b200_gemm_strided_i64": (ctypes.c_int, _gemm_sig(i64)),
    "laser_b200_gemm_strided_bf16": (ctypes.c_int, _gemm_sig(f32)),
    "laser_b200_gemm_strided_f32_dev": (ctypes.c_int, _gemm_sig(f32) + [ctypes.c_int, vp]),
    "laser_b200_gemm_strided_f32_epi_dev": (ctypes.c_int, _gemm_sig(f32) + [ctypes.POINTER(Epilogue), ctypes.c_int, vp]),
    "laser_b200_gemm_strided_f64_dev": (ctypes.c_int, _gemm_sig(f64) + [vp]),
    "laser_b200_gemm_strided_i32_dev": (ctypes.c_int, _gemm_sig(i32) + [vp]),
    "laser_b200_gemm_strided_i64_dev": (ctypes.c_int, _gemm_sig(i64) + [vp]),
    "laser_b200_gemm_strided_bf16_dev": (ctypes.c_int, _gemm_sig(f32) + [vp]),
    "laser_b200_gemm_prepackA_mem_required_f32": (sz, [i64, i64, i64]),
    "laser_b200_gemm_prepackB_mem_required_f32": (sz, [i64, i64, i64]),
    "laser_b200_gemm_prepackA_f32_dev": (ctypes.c_int, [vp, i64, i64, i64, vp, i64, i64, vp]),
    "laser_b200_gemm_prepackB_f32_dev": (ctypes.c_int, [vp, i64, i64, i64, vp, i64, i64, vp]),
    "laser_b200_gemm_packed_f32_dev": (ctypes.c_int, [i64, i64, i64, f32, vp, vp, f32, vp, i64, i64, vp]),
    "laser_b200_gemm_packedB_f32_dev": (ctypes.c_int, [i64, i64, i64, f32, vp, i64, i64, vp, f32, vp, i64, i64, vp]),
    "laser_b200_comm_get_unique_id": (ctypes.c_int, [vp]),
    "laser_b200_comm_init_rank": (ctypes.c_int, [ctypes.POINTER(vp), ctypes.c_int, ctypes.c_int, vp]),
    "laser_b200_comm_init_all": (ctypes.c_int, [ctypes.POINTER(vp), ctypes.c_int]),
    "laser_b200_comm_destroy": (ctypes.c_int, [vp]),
    "laser_b200_comm_rank": (ctypes.c_int, [vp]),
    "laser_b200_comm_size": (ctypes.c_int, [vp]),
    "laser_b200_rowshard_partition": (None, [i64, ctypes.c_int, ctypes.c_int, ctypes.POINTER(i64), ctypes.POINTER(i64)]),
    "laser_b200_gemm_rowsharded_f32_dev": (ctypes.c_int, [vp, i64, i64, i64, f32, vp, i64, i64, vp, i64, i64, ctypes.c_int, f32, vp,
                                                          i64, i64, vp]),
    "laser_b200_gemm_rowsharded_f32": (ctypes.c_int, [ctypes.c_int, i64, i64, i64, f32, vp, i64, i64, vp, i64, i64, f32, vp, i64, i64]),
    "laser_b200_malloc": (ctypes.c_int, [ctypes.POINTER(vp), sz]),
    "laser_b200_free": (ctypes.c_int, [vp]),
    "laser_b200_memcpy_h2d": (ctypes.c_int, [vp, vp, sz]),
    "laser_b200_memcpy_d2h": (ctypes.c_int, [vp, vp, sz]),
    "laser_b200_memset_zero": (ctypes.c_int, [vp, sz]),
    "laser_b200_synchronize": (ctypes.c_int, []),
    "laser_b200_matmul_views": (ctypes.c_int, [ctypes.POINTER(TensorView), ctypes.POINTER(TensorView),
                                               ctypes.POINTER(TensorView), f64, f64, ctypes.c_int, vp]),
    "laser_b200_gemm_strided_batched_f32_dev": (ctypes.c_int, [i64, i64, i64, i64, f32, vp, i64, i64, i64, vp, i64, i64, i64,
                                                               f32, vp, i64, i64, i64, ctypes.c_int, vp]),
    "laser_b200_gemm_strided_batched_f64_dev": (ctypes.c_int, [i64, i64, i64, i64, f64, vp, i64, i64, i64, vp, i64, i64, i64,
                                                               f64, vp, i64, i64, i64, vp]),
    "laser_b200_gemm_strided_batched_i32_dev": (ctypes.c_int, [i64, i64, i64, i64, i32, vp, i64, i64, i64, vp, i64, i64, i64,
                                                               i32, vp, i64, i64, i64, vp]),
    "laser_b200_gemm_strided_batched_i64_dev": (ctypes.c_int, [i64, i64, i64, i64, i64, vp, i64, i64, i64, vp, i64, i64, i64,
                                                               i64, vp, i64, i64, i64, vp]),
    "laser_b200_transpose2D_copy": (ctypes.c_int, [vp, vp, i64, i64, ctypes.c_int]),
    "laser_b200_transpose2D_batched": (ctypes.c_int, [vp, vp, i64, i64, i64, ctypes.c_int]),
    "laser_b200_nchw2nhwc": (ctypes.c_int, [vp, vp, i64, i64, i64, i64, ctypes.c_int]),
    "laser_b200_nhwc2nchw": (ctypes.c_int, [vp, vp, i64, i64, i64, i64, ctypes.c_int]),
    "laser_b200_transpose2D_copy_dev": (ctypes.c_int, [vp, vp, i64, i64, ctypes.c_int, vp]),
    "laser_b200_transpose2D_batched_dev": (ctypes.c_int, [vp, vp, i64, i64, i64, ctypes.c_int, vp]),
    "laser_b200_nchw2nhwc_dev": (ctypes.c_int, [vp, vp, i64, i64, i64, i64, ctypes.c_int, vp]),
    "laser_b200_nhwc2nchw_dev": (ctypes.c_int, [vp, vp, i64, i64, i64, i64, ctypes.c_int, vp]),
    "laser_b200_conv2d_out_shape": (ctypes.c_int, [i64 * 4, i64 * 4, i64 * 2, i64 * 2, i64 * 4]),
    "laser_b200_im2col_workspace_size": (i64, [i64 * 4, i64 * 4, i64 * 2, i64 * 2]),
    "laser_b200_im2col_f32_dev": (ctypes.c_int, [vp, vp, i64, i64 * 4, i64 * 4, i64 * 2, i64 * 2, vp]),
    "laser_b200_conv2d_im2col_f32_dev": (ctypes.c_int, [vp, vp, i64 * 4, vp, i64 * 4, i64 * 2, i64 * 2, vp, i64,
                                                        ctypes.c_int, vp]),
    "laser_b200_conv2d_im2col_f32": (ctypes.c_int, [vp, vp, i64 * 4, vp, i64 * 4, i64 * 2, i64 * 2]),
    "laser_b200_conv2d_direct_f32_dev": (ctypes.c_int, [vp, vp, i64 * 4, vp, i64 * 4, i64 * 2, i64 * 2, ctypes.POINTER(Epilogue),
                                                        vp]),
    "laser_b200_conv2d_direct_f32": (ctypes.c_int, [vp, vp, i64 * 4, vp, i64 * 4, i64 * 2, i64 * 2]),
    "laser_b200_copy_views": (ctypes.c_int, [ctypes.POINTER(TensorView), ctypes.POINTER(TensorView), vp]),
    "laser_b200_foreach_views": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(TensorView), ctypes.POINTER(TensorView),
                                                ctypes.POINTER(TensorView), ctypes.POINTER(TensorView), f64, vp]),
    "laser_b200_debug_classify": (ctypes.c_int, [ctypes.c_int, vp, i64, i64]),
    "laser_b200_debug_f64_dmma_launches": (i64, []),
    "laser_b200_debug_span": (ctypes.c_int, [i64, i64, i64, i64, ctypes.POINTER(i64), ctypes.POINTER(i64),
                                             ctypes.POINTER(ctypes.c_int)]),
    "laser_b200_fill_uniform_f32_dev": (ctypes.c_int, [vp, i64, u64, f32, f32, vp]),
}

_lib = None


def lib():
    """Load (building first if needed) the in-tree shared library.  Raises if it
    cannot be built or loaded: there is no Python/CPU fallback for any compute entry."""
    global _lib
    if _lib is None:
        path = os.environ.get("LASER_B200_LIB") or _build.build()   # override: A/B builds in tools/
        L = ctypes.CDLL(path)
        # tests/emu can build the library for the CPU (kernels on host threads) to test host logic without
        # a GPU; such a build marks itself and is only ever accepted inside those tests' own subprocesses
        if hasattr(L, "laser_b200_is_host_emulation") and os.environ.get("LASER_B200_EMU") != "1":
            raise RuntimeError("%s is a host-emulation TEST build of liblaser_b200 (tests/emu); refusing to use it as "
                               "the product library" % path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the header and the library disagree
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def lib_path():
    return _build.LIB_PATH


def check(code):
    if code != 0:
        msg = lib().laser_b200_last_error()
        raise LaserB200Error(code, msg.decode() if msg else "")
