"""laser_b200 -- B200-native (sm_100a) drop-in for mratsim/laser's strided GEMM hot path.

The product is the C-ABI shared library laser_b200/lib/liblaser_b200.so (hand-written CUDA:
tcgen05/TMEM/TMA tensor-core kernels + an exact SIMT kernel); this package is the thin
host-side mirror of the reference interface on top of it.  See DESIGN.md / INTEGRATION.md.
"""
from ._capi import (PATH_AUTO, PATH_BF16, PATH_F16X3, PATH_NAMES, PATH_SIMT, PATH_TF32X1, PATH_TF32X3, LaserB200Error, lib,
                    lib_path)
from .gemm import (DevPtr, fill_uniform_f32, gemm_strided, gemm_strided_fused, get_f32_mode, init, last_path,
                   launch_count, profile_begin, profile_end, set_f32_mode, shutdown,
                   synchronize)
from .layers import (FOREACH_OPS, conv2d_direct, conv2d_im2col, conv2d_out_shape, copyFrom, forEach, gemm_strided_batched, im2col,
                     im2col_workspace_size, nchw2nhwc, nhwc2nchw, transpose2D_batched, transpose2D_copy)
from .prepacked import (alloc_packed, gemm_packed, gemm_packedB, gemm_prepackA, gemm_prepackA_mem_required,
                        gemm_prepackB, gemm_prepackB_mem_required)
from .tensor import LASER_MAXRANK, Storage, Tensor, matmul, newTensor, toTensor

__version__ = "0.1.0"
