"""Host mirror of the steps either side of the GEMM in the reference's intended use
(SURVEY.md section 8f, rank 4), on top of the C ABI:

    transpose2D_copy(dst, src, NR, NC)            laser/primitives/swapaxes.nim:16-54
    transpose2D_batched(dst, src, N, NR, NC)      swapaxes.nim:56-81
    nchw2nhwc / nhwc2nchw(dst, src, N, C, H, W)   swapaxes.nim:83-112
    conv2d_out_shape, im2col_workspace_size       benchmarks/convolution/conv2d_common.nim:15-45,
                                                  conv2d_im2col.nim:8-18
    im2col, conv2d_im2col                         conv2d_im2col.nim:44-166
    conv2d_direct                                 conv2d_direct_convolution.nim:8-76
    gemm_strided_batched                          (roadmap item of the reference, README.md:253-263)
    copyFrom(dst, src)                            laser/tensor/initialization.nim:80-112

Same argument order and meaning as the reference; numpy arrays go through the host-pointer
entries (synchronous), torch CUDA tensors / laser_b200.Tensor / DevPtr through the `_dev`
entries on the current stream.  Shapes are (n, c, h, w) / (c_out, c_in, kH, kW) tuples."""
import ctypes

import numpy as np

from ._capi import PATH_AUTO, Epilogue, check, lib
from .gemm import _current_stream, _resolve, _scalar
from .tensor import _ITEMSIZE, Tensor

FOREACH_OPS = {"copy": 0, "fill": 1, "scale": 2, "add": 3, "sub": 4, "mul": 5, "fma": 6, "axpy": 7, "bench": 8}

__all__ = ["forEach", "FOREACH_OPS", "transpose2D_copy", "transpose2D_batched", "nchw2nhwc", "nhwc2nchw", "conv2d_out_shape",
           "im2col_workspace_size", "im2col", "conv2d_im2col", "conv2d_direct", "gemm_strided_batched", "copyFrom"]

_i64 = ctypes.c_int64


def _i4(t):
    if len(t) != 4:
        raise ValueError("expected a 4-tuple, got %r" % (t,))
    return (_i64 * 4)(*[int(v) for v in t])


def _i2(t):
    if len(t) != 2:
        raise ValueError("expected a 2-tuple, got %r" % (t,))
    return (_i64 * 2)(*[int(v) for v in t])


def _pair(dst, src):
    pd, td, dd = _resolve(dst)
    ps, ts, ds = _resolve(src)
    if td != ts:
        raise TypeError("dst and src element types differ: %s, %s" % (td, ts))
    if dd != ds:
        raise TypeError("dst and src must both be host pointers or both be device pointers")
    return pd, ps, _ITEMSIZE[td], dd


def _transpose(name, dst, src, dims, stream):
    pd, ps, esz, dev = _pair(dst, src)
    if dev:
        stream = _current_stream() if stream is None else stream
        check(getattr(lib(), "laser_b200_%s_dev" % name)(pd, ps, *dims, esz, stream))
    else:
        check(getattr(lib(), "laser_b200_" + name)(pd, ps, *dims, esz))


def transpose2D_copy(dst, src, NR, NC, stream=None):
    """dst[NC, NR] <- transpose of the contiguous src[NR, NC]."""
    _transpose("transpose2D_copy", dst, src, (NR, NC), stream)


def transpose2D_batched(dst, src, N, NR, NC, stream=None):
    _transpose("transpose2D_batched", dst, src, (N, NR, NC), stream)


def nchw2nhwc(dst_nhwc, src_nchw, N, C, H, W, stream=None):
    _transpose("nchw2nhwc", dst_nhwc, src_nchw, (N, C, H, W), stream)


def nhwc2nchw(dst_nchw, src_nhwc, N, C, H, W, stream=None):
    _transpose("nhwc2nchw", dst_nchw, src_nhwc, (N, C, H, W), stream)


def conv2d_out_shape(ishape, kshape, padding, strides):
    out = (_i64 * 4)()
    check(lib().laser_b200_conv2d_out_shape(_i4(ishape), _i4(kshape), _i2(padding), _i2(strides), out))
    return tuple(out)


def im2col_workspace_size(ishape, kshape, padding, strides):
    """ELEMENTS of workspace for one image: c * kH * kW * outH * outW (conv2d_im2col.nim:8-18)."""
    n = int(lib().laser_b200_im2col_workspace_size(_i4(ishape), _i4(kshape), _i2(padding), _i2(strides)))
    if n < 0:
        check(lib().laser_b200_conv2d_out_shape(_i4(ishape), _i4(kshape), _i2(padding), _i2(strides), (_i64 * 4)()))
    return n


def _dev_f32(x):
    p, t, d = _resolve(x)
    if not d or t != "f32":
        raise TypeError("expected a float32 device pointer")
    return p


def im2col(workspace, input, ishape, kshape, padding, strides, images=1, stream=None):
    """`images` images [c, h, w] starting at `input` -> `images` matrices [c*kH*kW, outH*outW]."""
    stream = _current_stream() if stream is None else stream
    check(lib().laser_b200_im2col_f32_dev(_dev_f32(workspace), _dev_f32(input), images, _i4(ishape), _i4(kshape),
                                          _i2(padding), _i2(strides), stream))


def conv2d_im2col(output, input, ishape, kernel, kshape, padding, strides, workspace=None, workspace_images=1,
                  path=PATH_AUTO, stream=None):
    """NCHW convolution through im2col + GEMM.  numpy arrays: host entry (library-owned
    workspace); device pointers: `workspace` must hold workspace_images * im2col_workspace_size
    float32 elements (may be None for 1x1 / stride 1 / no padding)."""
    po, to, do = _resolve(output)
    pi, ti, di = _resolve(input)
    pk, tk, dk = _resolve(kernel)
    if not (to == ti == tk == "f32"):
        raise TypeError("conv2d_im2col is float32 only")
    if not (do == di == dk):
        raise TypeError("output, input, kernel must all be host pointers or all be device pointers")
    if not do:
        if workspace is not None or path != PATH_AUTO:
            raise ValueError("the host-pointer entry owns its workspace and has no path argument")
        check(lib().laser_b200_conv2d_im2col_f32(po, pi, _i4(ishape), pk, _i4(kshape), _i2(padding), _i2(strides)))
        return
    stream = _current_stream() if stream is None else stream
    pw = _dev_f32(workspace) if workspace is not None else 0
    check(lib().laser_b200_conv2d_im2col_f32_dev(po, pi, _i4(ishape), pk, _i4(kshape), _i2(padding), _i2(strides), pw,
                                                 int(workspace_images), int(path), stream))


ACTIVATIONS = {"none": 0, "relu": 1, "tanh": 2, "sigmoid": 3}


def conv2d_direct(output, input, ishape, kernel, kshape, padding, strides, bias=None, activation=None, stream=None):
    """NCHW convolution without a workspace, one kernel launch per call; bit for bit what conv2d_im2col returns on
    path=PATH_SIMT.  numpy arrays: host entry (synchronous, no epilogue: `bias` / `activation` are a TypeError);
    device pointers: `bias` (NULL or a float32 device vector of c_out values) and `activation` (none | relu | tanh |
    sigmoid, or its code) are applied once to the final sum, act(x + bias[c_out])."""
    po, to, do = _resolve(output)
    pi, ti, di = _resolve(input)
    pk, tk, dk = _resolve(kernel)
    if not (to == ti == tk == "f32"):
        raise TypeError("conv2d_direct is float32 only")
    if not (do == di == dk):
        raise TypeError("output, input, kernel must all be host pointers or all be device pointers")
    if not do:
        if bias is not None or activation is not None:
            raise TypeError("the host-pointer entry has no epilogue: bias and activation need device buffers")
        check(lib().laser_b200_conv2d_direct_f32(po, pi, _i4(ishape), pk, _i4(kshape), _i2(padding), _i2(strides)))
        return
    epi = None
    if bias is not None or activation is not None:
        epi = Epilogue()
        if bias is not None:
            epi.bias = _dev_f32(bias)
        epi.bias_per_row = 1
        epi.activation = ACTIVATIONS[activation] if isinstance(activation, str) else int(activation or 0)
    stream = _current_stream() if stream is None else stream
    check(lib().laser_b200_conv2d_direct_f32_dev(po, pi, _i4(ishape), pk, _i4(kshape), _i2(padding), _i2(strides),
                                                 ctypes.byref(epi) if epi is not None else None, stream))


def gemm_strided_batched(batch, M, N, K, alpha, A, rowStrideA, colStrideA, batchStrideA, B, rowStrideB, colStrideB,
                         batchStrideB, beta, C, rowStrideC, colStrideC, batchStrideC, path=PATH_AUTO, stream=None):
    """`batch` problems C_b <- alpha * A_b * B_b + beta * C_b on device pointers (f32, f64, i32,
    i64); a batch stride of 0 shares that operand; outputs must not overlap."""
    pa, ta, da = _resolve(A)
    pb, tb, db = _resolve(B)
    pc, tc, dc = _resolve(C)
    if not (ta == tb == tc) or ta == "bf16":
        raise TypeError("batched GEMM needs A, B, C of one type among f32, f64, i32, i64 (got %s, %s, %s)" % (ta, tb, tc))
    if not (da and db and dc):
        raise TypeError("batched GEMM takes device pointers")
    stream = _current_stream() if stream is None else stream
    args = [batch, M, N, K, _scalar(ta, alpha), pa, rowStrideA, colStrideA, batchStrideA, pb, rowStrideB, colStrideB,
            batchStrideB, _scalar(ta, beta), pc, rowStrideC, colStrideC, batchStrideC]
    if ta == "f32":
        check(lib().laser_b200_gemm_strided_batched_f32_dev(*args, int(path), stream))
    else:
        if path not in (PATH_AUTO, 1):
            raise ValueError("path %d is not available for %s" % (path, ta))
        check(getattr(lib(), "laser_b200_gemm_strided_batched_%s_dev" % ta)(*args, stream))


def copyFrom(dst, src, stream=None):
    """dst <- src for two device Tensors of the same shape and dtype, any strides; only the
    elements the dst view exposes are written (initialization.nim:80-112)."""
    if not isinstance(dst, Tensor) or not isinstance(src, Tensor):
        raise TypeError("copyFrom takes laser_b200.Tensor views (use Tensor.from_torch for torch tensors)")
    vd, vs = dst.view_struct(), src.view_struct()
    stream = _current_stream() if stream is None else stream
    check(lib().laser_b200_copy_views(ctypes.byref(vd), ctypes.byref(vs), stream))
    return dst


def forEach(op, out, x=None, y=None, z=None, alpha=0.0, stream=None):
    """forEach o in out, x in a, y in b, z in c: <body> on device Tensors of one shape, any strides
    (laser/strided_iteration/foreach.nim:229-251).  `op` names the body:
      copy o = x | fill o = alpha | scale o = alpha*x | add o = x+y | sub o = x-y | mul o = x*y |
      fma o = x + y*z | axpy o = alpha*x + y | bench o = x + y - sin(z) (the reference's iteration benchmark)"""
    code = FOREACH_OPS[op] if isinstance(op, str) else int(op)
    views = [t.view_struct() if t is not None else None for t in (out, x, y, z)]
    refs = [ctypes.byref(v) if v is not None else None for v in views]
    stream = _current_stream() if stream is None else stream
    check(lib().laser_b200_foreach_views(code, refs[0], refs[1], refs[2], refs[3], float(alpha), stream))
    return out
