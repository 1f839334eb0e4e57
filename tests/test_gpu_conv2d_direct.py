"""GPU: the direct convolution entry (laser_b200_conv2d_direct_f32{,_dev}, conv2d_direct_convolution.nim:8-76) through the
C ABI.  Its contract is bit identity with the exact im2col path (conv2d_im2col on PATH_SIMT), so almost every check here
compares uint32 bit patterns (NaN matched by position) against that path run on the same device buffers; the small
shapes are also checked against the CPU oracle, and the fused bias + activation against im2col followed by the fused
GEMM on PATH_SIMT, image by image.

Backend-neutral like test_gpu_zlayers.py: with LASER_B200_EMU=1 numpy buffers stand in for device memory and the file
runs against the host-emulated library (tests/test_emulated_conv2d_direct.py); sizes too large for the CPU are skipped."""
import ctypes
import json
import os

import numpy as np
import pytest

import oracle as O

EMU = os.environ.get("LASER_B200_EMU", "0") == "1"
pytestmark = pytest.mark.gpu
if not EMU:
    torch = pytest.importorskip("torch")
import laser_b200 as L  # noqa: E402
from laser_b200 import _capi  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


class HostDev(L.DevPtr):
    """EMU backend: a numpy array posing as device memory."""

    def __init__(self, arr):
        self.arr = np.ascontiguousarray(arr)
        super().__init__(self.arr.ctypes.data, "f32")


def dev(a):
    a = np.ascontiguousarray(a, np.float32)
    return HostDev(a.copy()) if EMU else torch.from_numpy(a).cuda()


def full(shape, value):
    return dev(np.full(shape, value, np.float32))


def to_np(t):
    if EMU:
        return t.arr
    torch.cuda.synchronize()
    return t.cpu().numpy()


def addr(t):
    return t.ptr if EMU else t.data_ptr()


def at(t, offset):
    """f32 device pointer `offset` elements into t"""
    return L.DevPtr(addr(t) + 4 * offset, "f32")


def cpu_budget(outputs, taps):
    if EMU and outputs * max(taps, 64) > 6_000_000:
        pytest.skip("too large for the CPU stand-in")


def assert_same_bits(got, want):
    got = np.ascontiguousarray(got, np.float32).reshape(-1)
    want = np.ascontiguousarray(want, np.float32).reshape(-1)
    assert got.shape == want.shape
    gn, wn = np.isnan(got), np.isnan(want)
    assert np.array_equal(gn, wn), "NaN positions differ"
    g, w = got.view(np.uint32)[~gn], want.view(np.uint32)[~wn]
    bad = np.flatnonzero(g != w)
    assert bad.size == 0, "%d of %d values differ, first at %d: %r vs %r" % (bad.size, g.size, bad[0], got[~gn][bad[0]],
                                                                               want[~wn][bad[0]])


def data(ishape, kshape, seed=1, lo=-1.0, hi=1.0):
    inp = O.fill_uniform_f32(int(np.prod(ishape)), seed, lo, hi).reshape(ishape)
    ker = O.fill_uniform_f32(int(np.prod(kshape)), seed + 1, lo, hi).reshape(kshape)
    return inp, ker


def im2col_simt(tin, ishape, tker, kshape, padding, strides):
    """conv2d_im2col on PATH_SIMT over device buffers: the values conv2d_direct must reproduce"""
    oshape = L.conv2d_out_shape(ishape, kshape, padding, strides)
    per = L.im2col_workspace_size(ishape, kshape, padding, strides)
    out = full(oshape, -3.0)
    ws = full((max(1, ishape[0] * per),), 0)
    L.conv2d_im2col(out, tin, ishape, tker, kshape, padding, strides, workspace=ws, workspace_images=max(1, ishape[0]),
                    path=L.PATH_SIMT)
    return to_np(out)


def direct(tin, ishape, tker, kshape, padding, strides, **kw):
    out = full(L.conv2d_out_shape(ishape, kshape, padding, strides), np.nan)
    L.conv2d_direct(out, tin, ishape, tker, kshape, padding, strides, **kw)
    return to_np(out)


def conv_ref(inp, ishape, ker, kshape, padding, strides):
    """Oracle convolution, the expectation of test_gpu_zlayers.py: strided or padded 1x1 kernels go through im2col + the GEMM
    oracle (the reference's 1x1 shortcut reads the image in place there)."""
    if kshape[2] * kshape[3] != 1 or (tuple(strides) == (1, 1) and tuple(padding) == (0, 0)):
        return O.conv2d_im2col(inp, ishape, ker, kshape, padding, strides)
    o = O.conv2d_out_shape(ishape, kshape, padding, strides)
    M, K, N = kshape[0], ishape[1], o[2] * o[3]
    out = np.zeros((ishape[0], M, N), np.float32)
    kmat = np.ascontiguousarray(ker, np.float32).reshape(M, K)
    for n in range(ishape[0]):
        ws = np.ascontiguousarray(O.im2col(np.ascontiguousarray(inp[n]), ishape, kshape, padding, strides))
        O.gemm_strided(M, N, K, 1.0, kmat, K, 1, ws, N, 1, 0.0, out[n], N, 1)
    return out.reshape(o)


# ---- 1. known answers ------------------------------------------------------------------------------
def conv_cases():
    with open(os.path.join(HERE, "golden", "conv2d_known_answer.json")) as f:
        return json.load(f)["cases"]


@pytest.mark.parametrize("case", conv_cases(), ids=lambda c: c["src"])
def test_known_answer(case):
    inp = np.array(case["input"], np.float32); ker = np.array(case["kernel"], np.float32)
    tgt = np.array(case["target"], np.float32)
    ish, ksh, pad, st = case["ishape"], case["kshape"], case["padding"], case["strides"]
    out = np.full(tgt.shape, 99.0, np.float32)
    L.conv2d_direct(out, inp, ish, ker, ksh, pad, st)             # host entry
    assert np.array_equal(out, tgt)
    assert np.array_equal(direct(dev(inp), ish, dev(ker), ksh, pad, st), tgt)


# ---- 2./3. bit identity with the exact im2col path, and with the CPU oracle ----------------------------
SHAPES = [
    ((16, 3, 224, 224), (20, 3, 3, 3), (0, 0), (1, 1)),      # the reference bench shape (conv2d_bench.nim), all 16 images
    ((16, 3, 224, 224), (64, 3, 7, 7), (3, 3), (2, 2)),      # ResNet stem
    ((2, 3, 17, 19), (4, 3, 3, 3), (1, 1), (1, 1)),          # padding (1, 1)
    ((2, 2, 13, 16), (5, 2, 3, 3), (2, 1), (1, 1)),          # padding (2, 1)
    ((2, 3, 20, 21), (6, 3, 3, 3), (1, 1), (2, 2)),          # stride (2, 2)
    ((2, 2, 15, 18), (3, 2, 3, 3), (0, 1), (2, 1)),          # stride (2, 1): the width uses sW
    ((2, 4, 9, 9), (3, 4, 1, 1), (1, 1), (2, 2)),            # 1x1, stride 2, padding
    ((3, 4, 7, 10), (3, 4, 1, 1), (0, 0), (1, 1)),           # 1x1, unit stride: im2col reads the image in place
    ((2, 3, 20, 20), (8, 3, 5, 5), (2, 2), (1, 1)),          # 5x5
    ((1, 3, 30, 30), (9, 3, 7, 7), (3, 3), (2, 2)),          # 7x7
    ((1, 64, 12, 12), (10, 64, 3, 3), (1, 1), (1, 1)),       # K = 576: one 512-tap block boundary
    ((1, 128, 10, 10), (12, 128, 3, 3), (1, 1), (1, 1)),     # K = 1152: two
    ((2, 3, 16, 16), (1, 3, 3, 3), (0, 0), (1, 1)),          # c_out = 1
    ((1, 16, 12, 12), (64, 16, 3, 3), (1, 1), (1, 1)),       # c_out = 64
    ((1, 8, 10, 10), (129, 8, 3, 3), (1, 1), (1, 1)),        # c_out = 129: a last group of one channel
    ((1, 2, 9, 10), (3, 2, 3, 3), (0, 0), (1, 1)),           # outW = 8  (= 0 mod 4)
    ((1, 2, 9, 11), (3, 2, 3, 3), (0, 0), (1, 1)),           # outW = 9  (= 1 mod 4)
    ((1, 2, 9, 12), (3, 2, 3, 3), (0, 0), (1, 1)),           # outW = 10 (= 2 mod 4)
    ((1, 2, 9, 13), (3, 2, 3, 3), (0, 0), (1, 1)),           # outW = 11 (= 3 mod 4)
    ((3, 2, 12, 7), (4, 2, 3, 3), (1, 0), (1, 1)),           # W < 16
    ((1, 2, 40, 50), (5, 2, 3, 3), (1, 1), (1, 1)),          # two pixel tiles per image
    ((2, 2, 5, 20000), (3, 2, 3, 3), (1, 1), (1, 1)),        # one staged channel would not fit: input read from global
    ((2, 64, 3, 4000), (9, 64, 3, 3), (1, 1), (1, 1)),       # the same with K > 512
    ((32, 64, 56, 56), (64, 64, 3, 3), (1, 1), (1, 1)),      # large K and c_out
]
SMALL = [s for s in SHAPES if s[0][0] * s[0][2] * s[0][3] <= 20000]   # the oracle runs on one CPU thread


def _ids(s):
    return "%s-%s-p%s-s%s" % ("x".join(map(str, s[0])), "x".join(map(str, s[1])), "".join(map(str, s[2])), "".join(map(str, s[3])))


@pytest.mark.parametrize("ishape,kshape,padding,strides", SHAPES, ids=[_ids(s) for s in SHAPES])
def test_bit_identical_to_im2col_simt(ishape, kshape, padding, strides):
    oshape = L.conv2d_out_shape(ishape, kshape, padding, strides)
    cpu_budget(int(np.prod(oshape)), ishape[1] * kshape[2] * kshape[3])
    inp, ker = data(ishape, kshape, 11)
    tin, tker = dev(inp), dev(ker)
    assert_same_bits(direct(tin, ishape, tker, kshape, padding, strides), im2col_simt(tin, ishape, tker, kshape, padding, strides))


@pytest.mark.parametrize("ishape,kshape,padding,strides", SMALL, ids=[_ids(s) for s in SMALL])
def test_bit_identical_to_oracle(ishape, kshape, padding, strides):
    oshape = L.conv2d_out_shape(ishape, kshape, padding, strides)
    cpu_budget(int(np.prod(oshape)), ishape[1] * kshape[2] * kshape[3])
    inp, ker = data(ishape, kshape, 21)
    assert_same_bits(direct(dev(inp), ishape, dev(ker), kshape, padding, strides),
                     conv_ref(inp, ishape, ker, kshape, padding, strides))
    out = np.full(oshape, np.nan, np.float32)
    L.conv2d_direct(out, inp, ishape, ker, kshape, padding, strides)   # host entry
    assert_same_bits(out, conv_ref(inp, ishape, ker, kshape, padding, strides))


def test_offset_pointers():
    ishape, kshape, padding, strides = (2, 3, 14, 17), (5, 3, 3, 3), (1, 1), (1, 1)
    oshape = L.conv2d_out_shape(ishape, kshape, padding, strides)
    inp, ker = data(ishape, kshape, 31)
    tin = dev(np.concatenate([[7.0], inp.reshape(-1)]).astype(np.float32))
    tker = dev(np.concatenate([[5.0], ker.reshape(-1)]).astype(np.float32))
    tout = full((int(np.prod(oshape)) + 1,), np.nan)
    L.conv2d_direct(at(tout, 1), at(tin, 1), ishape, at(tker, 1), kshape, padding, strides)
    got = to_np(tout)
    assert np.isnan(got[0])
    assert_same_bits(got[1:], im2col_simt(dev(inp), ishape, dev(ker), kshape, padding, strides))


# ---- 4. fused bias + activation ----------------------------------------------------------------------
def im2col_then_fused_gemm(inp, ishape, ker, kshape, padding, strides, bias, activation):
    B, Cout = ishape[0], kshape[0]
    o = L.conv2d_out_shape(ishape, kshape, padding, strides)
    K, N = ishape[1] * kshape[2] * kshape[3], o[2] * o[3]
    ws = full((K * N,), 0)
    tker = dev(ker)
    out = full(o, np.nan)
    img = ishape[1] * ishape[2] * ishape[3]
    tin = dev(inp)
    for n in range(B):
        L.im2col(ws, at(tin, n * img), ishape, kshape, padding, strides, images=1)
        L.gemm_strided_fused(Cout, N, K, 1.0, tker, K, 1, ws, N, 1, 0.0, at(out, n * Cout * N), N, 1, bias=bias,
                             bias_per_row=True, activation=activation, path=L.PATH_SIMT)
    return to_np(out)


@pytest.mark.parametrize("with_bias", [False, True], ids=["nobias", "bias"])
@pytest.mark.parametrize("activation", ["none", "relu", "tanh", "sigmoid"])
@pytest.mark.parametrize("ishape,kshape", [((2, 3, 11, 13), (5, 3, 3, 3)), ((1, 64, 8, 9), (10, 64, 3, 3))],
                         ids=["K27", "K576"])
def test_epilogue_matches_im2col_and_fused_gemm(ishape, kshape, activation, with_bias):
    padding, strides = (1, 1), (1, 1)
    inp, ker = data(ishape, kshape, 41)
    bias = dev(O.fill_uniform_f32(kshape[0], 43, -2, 2)) if with_bias else None
    want = im2col_then_fused_gemm(inp, ishape, ker, kshape, padding, strides, bias, activation)
    got = direct(dev(inp), ishape, dev(ker), kshape, padding, strides, bias=bias, activation=activation)
    assert_same_bits(got, want)
    if activation == "relu":
        assert (got >= 0).all() and (got == 0).any()


# ---- 5. non-finite values --------------------------------------------------------------------------
def test_nan_in_image_and_inf_weight_with_padding():
    ishape, kshape, padding, strides = (2, 2, 12, 13), (4, 2, 3, 3), (1, 2), (1, 1)
    inp, ker = data(ishape, kshape, 51)
    inp[1, 0, 5, 6] = np.nan
    ker[2, 1, 0, 0] = np.inf      # times the zeros outside the image: NaN on the border of channel 2
    tin, tker = dev(inp), dev(ker)
    got = direct(tin, ishape, tker, kshape, padding, strides)
    assert_same_bits(got, im2col_simt(tin, ishape, tker, kshape, padding, strides))
    assert np.isnan(got[:, 2, 0, :]).all() and np.isnan(got[1, :, 5, 6]).all()
    assert not np.isnan(got[0, 0]).any()


# ---- 6. overwrite, bounds -------------------------------------------------------------------------
@pytest.mark.parametrize("ishape,kshape", [((2, 3, 9, 10), (5, 3, 3, 3)), ((1, 64, 6, 7), (9, 64, 3, 3))])
def test_output_overwritten_and_nothing_outside_written(ishape, kshape):
    padding, strides = (1, 1), (1, 1)
    n_out = int(np.prod(L.conv2d_out_shape(ishape, kshape, padding, strides)))
    inp, ker = data(ishape, kshape, 61)
    tin, tker = dev(inp), dev(ker)
    G, SENT = 1031, -12345.5
    results = []
    for prefill in (np.nan, 0.0):
        buf = np.full(n_out + 2 * G, SENT, np.float32)
        buf[G:G + n_out] = prefill
        tb = dev(buf)
        L.conv2d_direct(at(tb, G), tin, ishape, tker, kshape, padding, strides)
        got = to_np(tb)
        assert (got[:G] == SENT).all() and (got[G + n_out:] == SENT).all()
        results.append(got[G:G + n_out].copy())
    assert_same_bits(results[0], results[1])
    assert not np.isnan(results[0]).any()


# ---- 7. one launch per call -------------------------------------------------------------------------
@pytest.mark.parametrize("B", [0, 1, 16, 70000])
def test_one_launch_per_call(B):
    ishape, kshape, padding, strides = (B, 1, 5, 5), (2, 1, 3, 3), (0, 0), (1, 1)
    cpu_budget(B * 18, 9 * 30)
    inp, ker = data(ishape, kshape, 71)
    tin, tker = dev(inp), dev(ker)
    out = full(L.conv2d_out_shape(ishape, kshape, padding, strides), np.nan)
    n0 = L.launch_count()
    L.conv2d_direct(out, tin, ishape, tker, kshape, padding, strides)
    assert L.launch_count() - n0 == (1 if B else 0)
    got = to_np(out)
    if B == 0:
        return
    assert_same_bits(got, im2col_simt(tin, ishape, tker, kshape, padding, strides))


# ---- 8. more than 2^31 outputs -----------------------------------------------------------------------
@pytest.mark.skipif(EMU, reason="9.7 GB of output")
def test_beyond_2_31_outputs():
    ishape, kshape, padding, strides = (9, 3, 1024, 1024), (256, 3, 3, 3), (1, 1), (1, 1)
    oshape = L.conv2d_out_shape(ishape, kshape, padding, strides)
    assert np.prod(oshape, dtype=np.int64) > 2 ** 31
    g = torch.Generator(device="cuda").manual_seed(5)
    tin = torch.rand(ishape, device="cuda", generator=g) * 2 - 1
    tker = torch.rand(kshape, device="cuda", generator=g) * 2 - 1
    out = torch.full(oshape, float("nan"), device="cuda")
    L.conv2d_direct(out, tin, ishape, tker, kshape, padding, strides)
    one = (1,) + tuple(ishape[1:])
    last = torch.full((1,) + tuple(oshape[1:]), -1.0, device="cuda")
    ws = torch.zeros(L.im2col_workspace_size(one, kshape, padding, strides), device="cuda")
    L.conv2d_im2col(last, tin[-1:], one, tker, kshape, padding, strides, workspace=ws, path=L.PATH_SIMT)
    torch.cuda.synchronize()
    assert torch.equal(out[-1:].view(torch.int32), last.view(torch.int32))
    del out


# ---- 9. errors -------------------------------------------------------------------------------------
BAD = [
    ((1, 1, 4, 4), (1, 2, 3, 3), (1, 1), (1, 1)),    # c_in mismatch
    ((1, 1, 4, 4), (1, 1, 3, 3), (1, 1), (0, 1)),    # stride 0
    ((1, 1, 4, 4), (1, 1, 3, 3), (1, 1), (1, 4)),    # stride >= extent
    ((1, 1, 4, 4), (1, 1, 7, 3), (1, 1), (1, 1)),    # filter larger than the padded image
]


def _code(fn):
    try:
        fn()
    except L.LaserB200Error as e:
        return e.code
    return 0


@pytest.mark.parametrize("ishape,kshape,padding,strides", BAD)
def test_argument_errors_match_im2col(ishape, kshape, padding, strides):
    x = full((64,), 0)
    want = _code(lambda: L.conv2d_im2col(x, x, ishape, x, kshape, padding, strides, workspace=x))
    assert want == _capi.E_INVAL
    assert _code(lambda: L.conv2d_direct(x, x, ishape, x, kshape, padding, strides)) == want
    h = np.zeros(64, np.float32)
    assert _code(lambda: L.conv2d_direct(h, h, ishape, h, kshape, padding, strides)) == want


def test_null_pointers_and_epilogue_values():
    lib = L.lib()
    x = full((256,), 0)
    i4, i2 = ctypes.c_int64 * 4, ctypes.c_int64 * 2
    ish, ksh, pad, st = i4(1, 1, 6, 6), i4(2, 1, 3, 3), i2(1, 1), i2(1, 1)
    p = addr(x)
    for args in ((None, p, p), (p, None, p), (p, p, None)):
        rc_direct = lib.laser_b200_conv2d_direct_f32_dev(args[0], args[1], ish, args[2], ksh, pad, st, None, None)
        rc_im2col = lib.laser_b200_conv2d_im2col_f32_dev(args[0], args[1], ish, args[2], ksh, pad, st, p, 1, L.PATH_SIMT, None)
        assert rc_direct == rc_im2col == _capi.E_INVAL
        assert lib.laser_b200_conv2d_direct_f32(args[0], args[1], ish, args[2], ksh, pad, st) == _capi.E_INVAL
    bias = full((2,), 1.0)
    for bias_ptr, per_row, act in ((addr(bias), 0, 0), (addr(bias), 2, 1), (None, 0, 4), (addr(bias), 1, -1)):
        epi = _capi.Epilogue(bias_ptr, per_row, act)
        assert lib.laser_b200_conv2d_direct_f32_dev(p, p, ish, p, ksh, pad, st, ctypes.byref(epi), None) == _capi.E_INVAL
    ok = _capi.Epilogue(None, 0, 1)      # no bias: bias_per_row is not looked at
    xo, xk = full((72,), 0), full((18,), 0)
    assert lib.laser_b200_conv2d_direct_f32_dev(addr(xo), p, ish, addr(xk), ksh, pad, st, ctypes.byref(ok), None) == 0
    assert (to_np(xo) == 0).all()
    with pytest.raises(TypeError):
        h = np.zeros(64, np.float32)
        L.conv2d_direct(h, h, (1, 1, 6, 6), h, (2, 1, 3, 3), (1, 1), (1, 1), activation="relu")
    with pytest.raises(L.LaserB200Error):
        L.conv2d_direct(x, x, (1, 1, 6, 6), x, (2, 1, 3, 3), (1, 1), (1, 1), activation=4)
