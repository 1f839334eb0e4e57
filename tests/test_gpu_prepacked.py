"""GPU: the pre-packed API (gemm_prepackA/B + gemm_packed), mirroring the reference's own
pre-packed self-tests (gemm_prepacked.nim:300-523: the known-answer vectors pushed through
prepack + gemm_packed) plus strided/random checks against the oracle and the unpacked path."""
import numpy as np
import pytest

import oracle as O
from backend import dev, emu_budget, sync
from util import embed, extract, golden_cases

pytestmark = pytest.mark.gpu
import laser_b200 as L  # noqa: E402


def pack_both(M, N, K, tA, oa, rsa, csa, tB, ob, rsb, csb):
    pa = L.alloc_packed(L.gemm_prepackA_mem_required(M, N, K)); pb = L.alloc_packed(L.gemm_prepackB_mem_required(M, N, K))
    L.gemm_prepackA(pa, M, N, K, L.DevPtr(tA.data_ptr() + 4 * oa, "f32"), rsa, csa)
    L.gemm_prepackB(pb, M, N, K, L.DevPtr(tB.data_ptr() + 4 * ob, "f32"), rsb, csb)
    return pa, pb


@pytest.mark.parametrize("case", golden_cases(), ids=lambda c: c["src"])
def test_golden_through_prepack(case):
    M, N, K = case["M"], case["N"], case["K"]
    a = np.array(case["a"], np.float32); b = np.array(case["b"], np.float32)
    tA, tB = dev(a), dev(b); tC = dev(np.full((M, N), 99.0, np.float32))
    pa, pb = pack_both(M, N, K, tA, 0, K, 1, tB, 0, N, 1)
    L.gemm_packed(M, N, K, 1.0, pa, pb, 0.0, tC, N, 1)
    sync()
    assert np.array_equal(tC.cpu().numpy(), np.array(case["c"], np.float32))


@pytest.mark.parametrize("la,lb", [("row", "row"), ("col", "col"), ("colslice", "negrow"), ("padded", "both2")])
def test_packed_matches_oracle_and_unpacked(la, lb):
    M, N, K = 300, 520, 777
    A = O.fill_uniform_f32(M * K, 91, 0, 1).reshape(M, K); B = O.fill_uniform_f32(K * N, 92, 0, 1).reshape(K, N)
    C0 = O.fill_uniform_f32(M * N, 93, 0, 1).reshape(M, N)
    want = C0.copy(); O.gemm_strided(M, N, K, 0.5, A, K, 1, B, N, 1, -1.25, want, N, 1)
    ba, oa, rsa, csa = embed(A, la); bb, ob, rsb, csb = embed(B, lb)
    tA, tB = dev(ba), dev(bb)
    pa, pb = pack_both(M, N, K, tA, oa, rsa, csa, tB, ob, rsb, csb)
    tC = dev(C0); L.gemm_packed(M, N, K, 0.5, pa, pb, -1.25, tC, N, 1)
    tC2 = dev(C0); L.gemm_packedB(M, N, K, 0.5, L.DevPtr(tA.data_ptr() + 4 * oa, "f32"), rsa, csa, pb, -1.25, tC2, N, 1)
    tC3 = dev(C0)
    L.gemm_strided(M, N, K, 0.5, L.DevPtr(tA.data_ptr() + 4 * oa, "f32"), rsa, csa, L.DevPtr(tB.data_ptr() + 4 * ob, "f32"), rsb, csb,
                   -1.25, tC3, N, 1, path=L.PATH_F16X3)
    sync()
    got = tC.cpu().numpy()
    assert O.max_relative_error(got, want) < 1e-4
    # same tiles, same order of accumulation: packing changes nothing numerically
    assert np.array_equal(got, tC2.cpu().numpy()) and np.array_equal(got, tC3.cpu().numpy())


@pytest.mark.parametrize("lc", ["row", "col"])
@pytest.mark.parametrize("shape", [(100, 520, 777), (300, 520, 4096)], ids=["single_cta", "split_k"])
def test_packed_single_cta_split_k_and_col_major_c(shape, lc):
    """a single-CTA tile (M <= 128) and a split-K product (partial planes reduced by a second kernel), C row- or
    column-major: packed A and B, packed B only and the unpacked F16X3 call agree bit for bit"""
    M, N, K = shape
    emu_budget(float(M) * N * K)
    A = O.fill_uniform_f32(M * K, 94, -1, 1).reshape(M, K); B = O.fill_uniform_f32(K * N, 95, -1, 1).reshape(K, N)
    C0 = O.fill_uniform_f32(M * N, 96, -1, 1).reshape(M, N)
    bc, oc, rsc, csc = embed(C0, lc)
    tA, tB = dev(A), dev(B)
    pa, pb = pack_both(M, N, K, tA, 0, K, 1, tB, 0, N, 1)
    outs = [dev(bc) for _ in range(3)]
    L.gemm_packed(M, N, K, 0.5, pa, pb, -1.25, outs[0], rsc, csc)
    L.gemm_packedB(M, N, K, 0.5, tA, K, 1, pb, -1.25, outs[1], rsc, csc)
    L.gemm_strided(M, N, K, 0.5, tA, K, 1, tB, N, 1, -1.25, outs[2], rsc, csc, path=L.PATH_F16X3)
    sync()
    got = [extract(t.cpu().numpy(), oc, rsc, csc, M, N) for t in outs]
    scale = 0.5 * (np.abs(A.astype(np.float64)) @ np.abs(B.astype(np.float64))) + 1.25 * np.abs(C0)
    ref = 0.5 * (A.astype(np.float64) @ B.astype(np.float64)) - 1.25 * C0
    assert np.max(np.abs(got[0] - ref) / scale) < 1e-4
    assert np.array_equal(got[0].view(np.uint32), got[1].view(np.uint32))
    assert np.array_equal(got[0].view(np.uint32), got[2].view(np.uint32))


def test_mem_required_and_reuse():
    M, N, K = 1000, 640, 512
    assert L.gemm_prepackB_mem_required(M, N, K) >= N * K * 4 + N * 4 and L.gemm_prepackA_mem_required(M, N, K) >= M * K * 4 + M * 4
    assert L.gemm_prepackB_mem_required(0, 0, 0) == 0
    B = O.fill_uniform_f32(K * N, 5, 0, 1).reshape(K, N); tB = dev(B)
    pb = L.alloc_packed(L.gemm_prepackB_mem_required(M, N, K)); L.gemm_prepackB(pb, M, N, K, tB, N, 1)
    n0 = L.launch_count()
    for seed in (1, 2, 3):       # fixed B, fresh A: one split (A only) + one GEMM launch per product
        A = O.fill_uniform_f32(M * K, seed, 0, 1).reshape(M, K)
        want = np.zeros((M, N), np.float32); O.gemm_strided(M, N, K, 1.0, A, K, 1, B, N, 1, 0.0, want, N, 1)
        tC = dev(np.empty((M, N), np.float32)); L.gemm_packedB(M, N, K, 1.0, dev(A), K, 1, pb, 0.0, tC, N, 1)
        sync()
        assert O.max_relative_error(tC.cpu().numpy(), want) < 1e-4
    assert L.launch_count() - n0 == 6
