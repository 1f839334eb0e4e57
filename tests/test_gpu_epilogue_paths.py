"""GPU: the fused epilogue C <- act(alpha*A*B + beta*C + bias) on every branch that applies it -- the tensor-core kernel's
TMA-staged, plain vector and scalar stores, the split-K reduce (every tile split, and the partial last wave, where direct
and split tiles of one launch finish in two different kernels), TF32X1, the general exact kernel and both few-rows
kernels across a kc = 512 block boundary.  Every case is checked three ways:

  1. against the same path without an epilogue (`plain`): fused == act(plain + bias) within one rounding of a contracted
     multiply-add and the error of the activation; bit for bit when nothing is fused; exactly (bias and relu are one IEEE
     addition and a max) on the exact kernels, whose `plain` is pinned bit for bit to the CPU oracle;
  2. against act(alpha*A*B + beta*C + bias) in float64, with the tolerance of the product's path;
  3. nothing outside the C view changes.

Each case also asserts the branch it was written for: last_path(), and for tensor-core cases the number of GEMM-kernel
launches of a profiled call (2: split-K product + reduce, 1: direct), predicted by a restatement of the planner
(tc_params.h: tc_plan) for the device's SM count -- if the planner changes, these tests fail instead of silently testing
another branch."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as O
from backend import EMU, dev, emu_budget, sync
from util import embed, extract

pytestmark = pytest.mark.gpu

if not EMU:
    import torch
import laser_b200 as L  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
TINY = 2.0 ** -126
ACT64 = {"none": lambda x: x, "relu": lambda x: np.maximum(x, 0.0), "tanh": np.tanh,
         "sigmoid": lambda x: 1.0 / (1.0 + np.exp(-x))}
TOL = {L.PATH_F16X3: 1e-4, L.PATH_TF32X3: 1e-4, L.PATH_TF32X1: 5e-3}   # scaled bound of the product (test_gpu_fuzz.py)
SENTINEL = -7777.0


def sm_count():
    if EMU:
        return int(os.environ.get("LASER_B200_EMU_SMS", "8"))
    return torch.cuda.get_device_properties(0).multi_processor_count


def cdiv(a, b):
    return -(-a // b)


def tc_split(M, N, K, path, sms, kc=128):
    """(tiles, units, k_splits, n_direct) of an fp32 tensor-core call: tc_params.h tc_plan with the library's defaults
    (CTA pairs when M > 128, kc = 128 for the three-pass modes, split-K on, tail_min_k = 2048)"""
    pair = M > 128
    block_k = 64 if path == L.PATH_F16X3 else 32          # k-tile: 128 bytes of fp16 / fp32 pieces
    num_kb = cdiv(K, block_k)
    kb_per_block = num_kb if path == L.PATH_TF32X1 else min(max(cdiv(kc, block_k), 1), num_kb)
    tiles = cdiv(M, 256 if pair else 128) * cdiv(N, 256)
    units = sms // 2 if pair else sms
    blocks = cdiv(num_kb, kb_per_block)
    max_s = min(blocks // cdiv(512 // block_k, kb_per_block), 16)   # every split keeps >= 512 K-elements
    rem = tiles if tiles < units else tiles % units
    S = min(units // rem if rem else 1, max_s)
    if S >= 2 and (tiles < units or K >= 2048):
        per = cdiv(blocks, S)
        if cdiv(blocks, per) >= 2:
            return tiles, units, cdiv(blocks, per), tiles - rem
    return tiles, units, 1, tiles


def ulp(x):
    return np.spacing(np.abs(x).astype(np.float32)).astype(np.float64)


def act_bound(act, y):
    """error of tanhf / 1/(1+expf) on the device and in glibc: 4 ulp of the result, at least 2^-126"""
    return np.maximum(4.0 * ulp(y), TINY) if act in ("tanh", "sigmoid") else 0.0


@functools.lru_cache(maxsize=2)
def operands(M, N, K, seed):
    """A, B in U(-0.1,0.1) -- products of order 1, next to biases in U(-1,1), so that every activation works in its
    non-linear range and a bias of +-100 saturates it -- and their float64 products A@B, |A|@|B|"""
    A = O.fill_uniform_f32(M * K, seed + 1, -0.1, 0.1).reshape(M, K)
    B = O.fill_uniform_f32(K * N, seed + 2, -0.1, 0.1).reshape(K, N)
    A64, B64 = A.astype(np.float64), B.astype(np.float64)
    return A, B, A64 @ B64, np.abs(A64) @ np.abs(B64)


def embed_b(B, lb):
    """util.embed, plus 'pitch:P': row-major with row pitch P >= N (sentinel in the gap)"""
    if lb.startswith("pitch:"):
        K, N = B.shape
        P = int(lb[6:])
        big = np.full((K, P), SENTINEL, np.float32); big[:, :N] = B
        return big.reshape(-1), 0, P, 1
    return embed(B, lb)


def bias_vector(kind, M, N, seed):
    """-> (values, per_row, device pointer) for a bias kind:
    'row' / 'col': U(-1,1) per row / column; 'col+4': per column, 4 bytes past a 16-byte boundary;
    'row!' / 'col!': as 'row' / 'col' with +-100 on every 37th entry (saturates tanh and sigmoid)."""
    if kind is None:
        return None, False, None
    per_row = kind.startswith("row")
    n = M if per_row else N
    v = O.fill_uniform_f32(n, seed + 4, -1, 1).copy()
    if kind.endswith("!"):
        idx = np.arange(5, n, 37)
        v[idx] = np.where(np.arange(idx.size) % 2 == 0, 100.0, -100.0)
    if kind == "col+4":
        t = dev(np.concatenate([np.full(1, SENTINEL, np.float32), v]))
        return v, per_row, (t, L.DevPtr(t.data_ptr() + 4, "f32"))
    t = dev(v)
    return v, per_row, (t, L.DevPtr(t.data_ptr(), "f32"))


def outside_unchanged(after, before, oc, rsc, csc, M, N):
    mask = np.ones(after.size, bool)
    mask[(oc + np.arange(M)[:, None] * rsc + np.arange(N)[None, :] * csc).ravel()] = False
    return np.array_equal(after[mask], before[mask], equal_nan=True)


def check_case(M, N, K, path, variant, lc="row", lb="row", seed=0, plain_path=None, want_path=None):
    """Run one product with and without the epilogue variant (bias kind, activation, alpha, beta) and apply the three
    gates and the branch probe.  Returns the GEMM-kernel launches of the profiled call (tensor-core paths) or None."""
    bias_kind, act, alpha, beta = variant
    emu_budget(float(M) * N * K)
    A, B, prod, absprod = operands(M, N, K, seed)
    C0 = O.fill_uniform_f32(M * N, seed + 3, -1, 1).reshape(M, N) if beta != 0.0 else np.full((M, N), np.nan, np.float32)
    bias, per_row, bias_dev = bias_vector(bias_kind, M, N, seed)
    bb, ob, rsb, csb = embed_b(B, lb)
    bc, oc, rsc, csc = embed(C0, lc)
    ta, tb = dev(A), dev(bb)
    pa, pb = L.DevPtr(ta.data_ptr(), "f32"), L.DevPtr(tb.data_ptr() + 4 * ob, "f32")
    plain_path = path if plain_path is None else plain_path
    want_path = path if want_path is None else want_path

    bias_ptr = None if bias_dev is None else bias_dev[1]

    def run(fused, profile=False):
        tc = dev(bc)
        pc = L.DevPtr(tc.data_ptr() + 4 * oc, "f32")
        if profile:
            L.profile_begin()
        if fused:
            L.gemm_strided_fused(M, N, K, alpha, pa, K, 1, pb, rsb, csb, beta, pc, rsc, csc, bias=bias_ptr,
                                 bias_per_row=per_row, activation=act, path=path)
        else:
            L.gemm_strided(M, N, K, alpha, pa, K, 1, pb, rsb, csb, beta, pc, rsc, csc, path=plain_path)
        prof = L.profile_end() if profile else None
        sync()
        after = tc.cpu().numpy().copy()
        assert outside_unchanged(after, bc, oc, rsc, csc, M, N), "a write outside the C view"
        return extract(after, oc, rsc, csc, M, N), prof

    got, _ = run(True)
    assert L.last_path() == want_path, (L.last_path(), want_path)
    plain, _ = run(False)
    assert np.isfinite(got).all() and np.isfinite(plain).all()
    b64 = np.zeros((1, 1)) if bias is None else (bias[:, None] if per_row else bias[None, :]).astype(np.float64)
    pl = plain.astype(np.float64)
    out = got.astype(np.float64)

    if want_path == L.PATH_SIMT:
        # exact kernels: plain is the reference's order of operations; the epilogue is one IEEE addition then act
        want_plain = C0.copy()
        O.gemm_strided(M, N, K, alpha, A, K, 1, B, N, 1, beta, want_plain, N, 1)
        assert np.array_equal(plain.view(np.uint32), want_plain.view(np.uint32)), "exact path differs from the oracle"
        pre32 = plain + (np.zeros((1, 1), np.float32) if bias is None else b64.astype(np.float32))
        if act in ("none", "relu"):
            assert np.array_equal(got, ACT64[act](pre32).astype(np.float32))
        else:
            want = ACT64[act](pre32.astype(np.float64))
            assert np.all(np.abs(out - want) <= act_bound(act, want)), np.abs(out - want).max()
        launches = None
    else:
        # 1. consistency with the plain product of the same path
        pre = pl + b64
        if bias is None and act == "none":
            assert np.array_equal(got.view(np.uint32), plain.view(np.uint32)), "an empty epilogue changed the result"
        else:
            want = ACT64[act](pre)
            err = np.abs(out - want) - (ulp(pl) + ulp(pre) + act_bound(act, want))
            assert np.all(err <= 0), ("fused vs plain", np.unravel_index(np.argmax(err), err.shape), err.max())
        # 2. accuracy against float64
        c64 = np.nan_to_num(C0.astype(np.float64)) if beta != 0.0 else 0.0
        ref = ACT64[act](alpha * prod + beta * c64 + b64)
        scale = abs(alpha) * absprod + abs(beta) * np.abs(c64)
        err = np.abs(out - ref) - (TOL[want_path] * scale + ulp(pl) + ulp(pre) + act_bound(act, ref))
        assert np.all(err <= 0), ("fused vs float64", np.unravel_index(np.argmax(err), err.shape), err.max())
        # branch probe: a profiled call of the same product (separate: profiling turns programmatic dependent launch off)
        _, prof = run(True, profile=True)
        launches = prof["gemm_launches"]
        _, _, ks, _ = tc_split(M, N, K, want_path, sm_count())
        assert launches == (2 if ks > 1 else 1), (launches, ks, sm_count())
    if bias_kind is not None and bias_kind.endswith("!") and act in ("tanh", "sigmoid"):
        sat = np.zeros((M, N), bool)
        idx = np.arange(5, M if per_row else N, 37)
        if per_row:
            sat[idx, :] = True
        else:
            sat[:, idx] = True
        s = got[sat]
        if act == "tanh":
            assert np.all(np.abs(s) == 1.0)
        else:
            assert np.all((s == 1.0) | (s <= TINY))
    return launches


# (bias kind, activation, alpha, beta); beta = 0 runs over a C full of NaN.  The (alpha, beta) pairs are the ones the
# parity file treats as exact for the SIMT kernels.
VARIANTS = [
    ("col", "relu", 1.0, 0.0),
    ("row", "tanh", 0.5, -1.25),
    ("col+4", "sigmoid", 0.5, -1.25),
    (None, "sigmoid", -2.0, 0.0),
    ("row", "none", 1.0, 1.0),
    ("col+4", "tanh", -2.0, 0.0),
    (None, "none", 0.5, -1.25),
    ("row!", "tanh", 1.0, 0.0),
    ("col!", "sigmoid", 0.5, -1.25),
]
LARGE_VARIANTS = [VARIANTS[i] for i in (0, 1, 2, 8)]   # 2304^2 outputs: one variant per activation, both bias orientations


def vid(v):
    return "%s-%s-a%g-b%g" % (v[0] or "nobias", v[1], v[2], v[3])


F16, T3, T1 = L.PATH_F16X3, L.PATH_TF32X3, L.PATH_TF32X1
# (name, M, N, K, path, C layout, k_splits on 148 SMs, n_direct on 148 SMs)
TC_CASES = [
    ("pair_tma_ragged", 300, 520, 700, F16, "row", 1, 6),          # TMA-staged store; columns 512-519: scalar store, same row
    ("pair_tma_ragged_tf32x3", 300, 520, 700, T3, "row", 1, 6),
    ("single_cta", 100, 520, 700, F16, "row", 1, 3),
    ("tiles_per_cta", 2304, 2304, 1024, F16, "row", 1, 81),        # 81 pair tiles on 74 pairs
    ("split_pair", 300, 520, 4096, F16, "row", 8, 0),
    ("split_pair_tf32x3", 300, 520, 4096, T3, "row", 8, 0),
    ("split_single", 100, 520, 4096, F16, "row", 8, 0),
    ("split_single_k1024", 100, 520, 1024, F16, "row", 2, 0),
    ("split_single_k1024_tf32x3", 100, 520, 1024, T3, "row", 2, 0),
    ("tail_wave", 2304, 2304, 2048, F16, "row", 4, 74),            # 74 direct tiles + 7 tiles x 4 splits
    ("tail_wave_tf32x3", 2304, 2304, 2048, T3, "row", 4, 74),
    ("tf32x1", 300, 520, 700, T1, "row", 1, 6),
    ("tf32x1_tiles_per_cta", 2304, 2304, 1024, T1, "row", 1, 81),
    ("scalar_odd_ldc", 300, 520, 700, F16, "padded", 1, 6),
    ("scalar_col", 300, 520, 700, F16, "col", 1, 6),
    ("scalar_negcol", 300, 520, 700, T3, "negcol", 1, 6),
    ("split_odd_ldc", 300, 520, 4096, F16, "padded", 8, 0),
    ("split_col", 300, 520, 4096, F16, "col", 8, 0),
    ("split_negcol", 300, 520, 4096, T3, "negcol", 8, 0),
]
TC_PARAMS = [pytest.param(c, v, id="%s-%s" % (c[0], vid(v)))
             for c in TC_CASES for v in (LARGE_VARIANTS if c[1] * c[2] > 2e6 else VARIANTS)]


def test_planner_restatement_on_148_sms():
    """the split column of the case table, from the restated planner for a B200's 148 SMs (what each case is for)"""
    for name, M, N, K, path, _, ks, nd in TC_CASES:
        tiles, units, got_ks, got_nd = tc_split(M, N, K, path, 148)
        assert (got_ks, got_nd) == (ks, nd), name
        if name.startswith("single") or "split_single" in name:
            assert M <= 128 and units == 148
        if "tiles_per_cta" in name or "tail_wave" in name:
            assert tiles > units
        if "tail_wave" in name:
            assert 0 < nd < tiles


@pytest.mark.parametrize("case,variant", TC_PARAMS)
def test_tensor_core_epilogue(case, variant, record_property):
    name, M, N, K, path, lc, _, _ = case
    record_property("gemm_launches", check_case(M, N, K, path, variant, lc=lc))


@pytest.mark.parametrize("variant", [v for v in VARIANTS if v[0] or v[1] != "none"], ids=vid)
def test_auto_tall_n3_with_epilogue_takes_f16x3(variant, record_property):
    """N <= 4 and tall: AUTO sends a plain product to the GEMV kernels, which have no epilogue -- with one it must take
    the default tensor-core mode (plain reference: the same product on F16X3; an empty epilogue is a plain product)"""
    record_property("gemm_launches", check_case(1500, 3, 700, L.PATH_AUTO, variant, plain_path=L.PATH_F16X3,
                                                want_path=L.PATH_F16X3))


def test_plain_vector_store_without_tma():
    """LASER_B200_C_TMA=0: direct tiles leave through plain 16-byte stores (read once per process, hence a subprocess)"""
    code = ("import sys; sys.path[:0] = [%r, %r]\n"
            "import test_gpu_epilogue_paths as T\n"
            "for v in T.VARIANTS[:3] + T.VARIANTS[6:]:\n"
            "    assert T.check_case(300, 520, 700, T.L.PATH_F16X3, v) == 1\n"
            "print('ok')\n") % (HERE, os.path.dirname(HERE))
    env = dict(os.environ, LASER_B200_C_TMA="0")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stdout[-3000:] + out.stderr[-3000:]


# exact kernels: the general SIMT kernel (odd ldc) and the few-rows kernels across the kc = 512 boundary, B with a row
# pitch that is a multiple of 4 (cp.async kernel) or column-major (register kernel)
SIMT_CASES = [("general_odd_ldc", 150, 270, 1100, "row", "padded")] + \
             [("few_rows_%s_M%d" % (kern, M), M, 1031, 1100, lb, "row")
              for M in (8, 20, 32) for kern, lb in (("async", "pitch:1032"), ("register", "col"))]


@pytest.mark.parametrize("variant", VARIANTS, ids=vid)
@pytest.mark.parametrize("case", SIMT_CASES, ids=lambda c: c[0])
def test_exact_kernel_epilogue(case, variant):
    name, M, N, K, lb, lc = case
    check_case(M, N, K, L.PATH_SIMT, variant, lc=lc, lb=lb)
