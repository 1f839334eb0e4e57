"""GPU: the exact few-rows kernels and the GEMV kernels, each on the branches it dispatches to on its own.

Few rows (M <= 32, N >= 1024: the im2col convolution's product; PATH_SIMT, and AUTO whatever the fp32 mode): the
cp.async kernel (B with unit column stride, row pitch a multiple of 4 and a 16-byte aligned base) and the register
kernel (every other B), MT = 8 / 16 / 24 / 32, ragged N, kc = 512 block boundaries, strided A and C, alpha / beta, several
tiles per CTA, batched and through the host-pointer entry -- all BIT FOR BIT against the CPU oracle.

GEMV (AUTO, N <= 4, M >= 1024, no epilogue): the shared-memory, vectorised and scalar variants, strided B and C,
beta = 0 over NaN, and the grid-stride loop -- against float64 with the order-independent bound
|got - ref| <= K * 2^-23 * (|alpha| |A||B| + |beta| |C|) (the warp reduction sums in another order than the oracle).

Every case also checks that nothing outside the C view changes."""
import os

import numpy as np
import pytest

import oracle as O
from backend import EMU, dev, emu_budget, sync
from util import embed, extract

pytestmark = pytest.mark.gpu

if not EMU:
    import torch
import laser_b200 as L  # noqa: E402

SENTINEL = -7777.0
AB = [(1.0, 0.0), (0.5, -1.25), (1.0, 1.0), (-2.0, 0.0)]   # the (alpha, beta) pairs the exact kernels reproduce bit for bit


def sm_count():
    if EMU:
        return int(os.environ.get("LASER_B200_EMU_SMS", "8"))
    return torch.cuda.get_device_properties(0).multi_processor_count


def cdiv(a, b):
    return -(-a // b)


def embed_b(B, lb):
    """util.embed, plus row-major B with a row pitch rounded up to a multiple of 4 ('pitch4') or one that is not a
    multiple of 4 ('pitch_odd'); the gap holds a sentinel"""
    if lb in ("pitch4", "pitch_odd"):
        K, N = B.shape
        P = cdiv(N, 4) * 4 + (1 if lb == "pitch_odd" else 0)
        big = np.full((K, P), SENTINEL, np.float32); big[:, :N] = B
        return big.reshape(-1), 0, P, 1
    return embed(B, lb)


def few_rows_kernel(b_addr, rsB, csB, batch=1, bsB=0):
    """which few-rows kernel a B operand selects (capi.cu, gemm_simt: async_ok)"""
    ok = csB == 1 and rsB % 4 == 0 and (batch == 1 or bsB % 4 == 0) and b_addr % 16 == 0
    return "async" if ok else "register"


def outside_unchanged(after, before, oc, rsc, csc, M, N):
    mask = np.ones(after.size, bool)
    mask[(oc + np.arange(M)[:, None] * rsc + np.arange(N)[None, :] * csc).ravel()] = False
    return np.array_equal(after[mask], before[mask], equal_nan=True)


def run_product(M, N, K, la, lb, lc, alpha, beta, path, seed):
    """one product through the device entry on embedded operands -> (A, B, C0, C, launches, B address, rsB, csB)"""
    emu_budget(float(M) * N * K)
    A = O.fill_uniform_f32(M * K, seed + 1, -1, 1).reshape(M, K)
    B = O.fill_uniform_f32(K * N, seed + 2, -1, 1).reshape(K, N)
    C0 = O.fill_uniform_f32(M * N, seed + 3, -1, 1).reshape(M, N) if beta != 0.0 else np.full((M, N), np.nan, np.float32)
    ba, oa, rsa, csa = embed(A, la); bb, ob, rsb, csb = embed_b(B, lb); bc, oc, rsc, csc = embed(C0, lc)
    ta, tb, tc = dev(ba), dev(bb), dev(bc)
    b_addr = tb.data_ptr() + 4 * ob
    n0 = L.launch_count()
    L.gemm_strided(M, N, K, alpha, L.DevPtr(ta.data_ptr() + 4 * oa, "f32"), rsa, csa, L.DevPtr(b_addr, "f32"), rsb, csb, beta,
                   L.DevPtr(tc.data_ptr() + 4 * oc, "f32"), rsc, csc, path=path)
    launches = L.launch_count() - n0
    sync()
    after = tc.cpu().numpy()
    assert outside_unchanged(after, bc, oc, rsc, csc, M, N), "a write outside the C view"
    return A, B, C0, extract(after, oc, rsc, csc, M, N), launches, b_addr, rsb, csb


def check_few_rows(M, N, K, la, lb, lc, ab, path, seed=0):
    """exact few-rows product, bit for bit against the oracle; returns the kernel the B operand selected"""
    assert M <= 32 and N >= 1024
    alpha, beta = ab
    A, B, C0, got, launches, b_addr, rsb, csb = run_product(M, N, K, la, lb, lc, alpha, beta, path, seed)
    assert L.last_path() == L.PATH_SIMT and launches == 1
    want = C0.copy(); O.gemm_strided(M, N, K, alpha, A, K, 1, B, N, 1, beta, want, N, 1)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (M, N, K, la, lb, lc, ab, path)
    return few_rows_kernel(b_addr, rsb, csb)


# --------------------------------------------------------------------------------- few rows: every kernel, ragged N
# (M, N, K, A layout, B layout, C layout, (alpha, beta), path, kernel the B layout selects)
KERNEL_CASES = [
    (24, 1031, 1100, "row", "pitch4", "row", (1.0, 0.0), L.PATH_AUTO, "async"),       # zero-filled partial cp.async
    (1, 1025, 513, "col", "pitch4", "padded", (0.5, -1.25), L.PATH_SIMT, "async"),
    (32, 4093, 65, "negrow", "pitch4", "col", (1.0, 1.0), L.PATH_SIMT, "async"),
    (16, 1024, 1100, "row", "row", "row", (1.0, 0.0), L.PATH_AUTO, "async"),           # the plain store
    (8, 1031, 512, "row", "row", "misaligned", (-2.0, 0.0), L.PATH_AUTO, "register"),  # ragged contiguous: rsB % 4 != 0
    (20, 1031, 1100, "row", "col", "padded", (0.5, -1.25), L.PATH_SIMT, "register"),
    (9, 1025, 27, "col", "misaligned", "row", (1.0, 1.0), L.PATH_AUTO, "register"),
    (31, 4093, 511, "row", "pitch_odd", "col", (1.0, 0.0), L.PATH_SIMT, "register"),
    (4, 1031, 64, "negrow", "negrow", "row", (0.5, -1.25), L.PATH_AUTO, "register"),    # rsB = -1031
    (17, 1024, 9, "row", "negrow", "padded", (-2.0, 0.0), L.PATH_SIMT, "async"),        # rsB = -1024, base 16-byte aligned
    (25, 1024, 1, "row", "col", "misaligned", (0.5, -1.25), L.PATH_SIMT, "register"),
    (3, 1024, 7, "col", "pitch4", "col", (1.0, 1.0), L.PATH_AUTO, "async"),
]


@pytest.mark.parametrize("case", KERNEL_CASES, ids=lambda c: "M%d-N%d-K%d-%s-%s-%s-%s" % (c[0], c[1], c[2], c[3], c[4], c[5], c[8]))
def test_few_rows_kernel_selection(case):
    *args, kernel = case
    assert check_few_rows(*args) == kernel


FEW_M = [1, 3, 4, 8, 9, 16, 17, 24, 25, 31, 32]
FEW_N = [1024, 1025, 1031, 4093]
FEW_K = [1, 7, 9, 27, 64, 65, 511, 512, 513, 1100]


@pytest.mark.parametrize("seed", range(48))
def test_few_rows_random(seed):
    """a seeded sample of M x N x K x layouts x (alpha, beta) x path"""
    rng = np.random.default_rng(5000 + seed)
    M, N, K = int(rng.choice(FEW_M)), int(rng.choice(FEW_N)), int(rng.choice(FEW_K))
    la = str(rng.choice(["row", "col", "negrow"]))
    lb = str(rng.choice(["pitch4", "row", "col", "misaligned", "pitch_odd", "negrow"]))
    lc = str(rng.choice(["row", "padded", "col", "misaligned"]))
    ab = AB[int(rng.integers(len(AB)))]
    path = int(rng.choice([L.PATH_SIMT, L.PATH_AUTO]))
    check_few_rows(M, N, K, la, lb, lc, ab, path, seed=seed)


@pytest.mark.parametrize("path", [L.PATH_SIMT, L.PATH_AUTO])
def test_m33_leaves_the_few_rows_kernels(path):
    """M = 33: PATH_SIMT takes the general exact kernel (still bit for bit), AUTO the tensor cores"""
    M, N, K = 33, 1024, 1100
    A, B, C0, got, _, _, _, _ = run_product(M, N, K, "row", "pitch4", "row", 0.5, -1.25, path, 7)
    want = C0.copy(); O.gemm_strided(M, N, K, 0.5, A, K, 1, B, N, 1, -1.25, want, N, 1)
    if path == L.PATH_SIMT:
        assert L.last_path() == L.PATH_SIMT
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    else:
        assert L.last_path() == L.PATH_F16X3
        scale = 0.5 * (np.abs(A.astype(np.float64)) @ np.abs(B.astype(np.float64))) + 1.25 * np.abs(C0)
        assert np.max(np.abs(got - want) / scale) < 1e-4


@pytest.mark.parametrize("kernel", ["async", "register"])
def test_few_rows_several_tiles_per_cta(kernel):
    """more column tiles than the grid has CTAs: the cp.async kernel keeps ONE FIFO across its tiles (the copies of the
    next tile are in flight while this one is multiplied); the register kernel loops over its tiles"""
    N, K = 163841, 27
    if kernel == "async":
        M, lb = 8, "pitch4"
        tiles, grid = cdiv(N, 1024), sm_count()               # 1024 columns per tile, one CTA per SM
    else:
        M, lb = 20, "col"
        tiles, grid = cdiv(N, 256 * 2), 2 * sm_count()        # NC = 2 columns per thread for M > 16, two CTAs per SM
    assert tiles > grid, (tiles, grid)
    assert check_few_rows(M, N, K, "row", lb, "row", (0.5, -1.25), L.PATH_AUTO) == kernel


@pytest.mark.parametrize("bsB_pad,kernel", [(0, "async"), (1, "register")])
def test_few_rows_batched(bsB_pad, kernel):
    """gemm_strided_batched with a shared A (batch stride 0): one launch of the few-rows kernel over every problem;
    a batch stride of B that is not a multiple of 4 sends it to the register kernel"""
    batch, M, N, K = 3, 20, 1024, 100
    emu_budget(float(batch) * M * N * K)
    A = O.fill_uniform_f32(M * K, 31, -1, 1)
    bsB = K * N + bsB_pad
    B = np.full((batch - 1) * bsB + K * N, SENTINEL, np.float32)
    for b in range(batch):
        B[b * bsB:b * bsB + K * N] = O.fill_uniform_f32(K * N, 32 + b, -1, 1)
    C0 = O.fill_uniform_f32(batch * M * N, 35, -1, 1)
    want = C0.copy()
    O.gemm_strided_batched(batch, M, N, K, 0.5, A, K, 1, 0, B, N, 1, bsB, -1.25, want, N, 1, M * N)
    tA, tB, tC = dev(A), dev(B), dev(C0)
    assert few_rows_kernel(tB.data_ptr(), N, 1, batch, bsB) == kernel
    n0 = L.launch_count()
    L.gemm_strided_batched(batch, M, N, K, 0.5, tA, K, 1, 0, tB, N, 1, bsB, -1.25, tC, N, 1, M * N)
    assert L.launch_count() - n0 == 1 and L.last_path() == L.PATH_SIMT
    sync()
    assert np.array_equal(tC.cpu().numpy().view(np.uint32), want.view(np.uint32))


def test_few_rows_host_pointer_entry():
    M, N, K = 24, 1031, 513
    A = O.fill_uniform_f32(M * K, 41, -1, 1).reshape(M, K); B = O.fill_uniform_f32(K * N, 42, -1, 1).reshape(K, N)
    C0 = O.fill_uniform_f32(M * N, 43, -1, 1).reshape(M, N)
    want = C0.copy(); O.gemm_strided(M, N, K, 0.5, A, K, 1, B, N, 1, -1.25, want, N, 1)
    C = C0.copy()
    L.gemm_strided(M, N, K, 0.5, A, K, 1, B, N, 1, -1.25, C, N, 1)
    assert L.last_path() == L.PATH_SIMT
    assert np.array_equal(C.view(np.uint32), want.view(np.uint32))


# ------------------------------------------------------------------------------------------------------------- GEMV
def gemv_variant(a_addr, rsA, csA, N, K):
    """capi.cu, f32_dev case -1: shared memory / vectorised / scalar"""
    vec = csA == 1 and rsA % 4 == 0 and K % 4 == 0 and a_addr % 16 == 0
    return "smem" if vec and N * K * 4 <= 96 * 1024 else "vec" if vec else "scalar"


# (N, M, K, A layout, B layout, C layout, (alpha, beta), variant); M * N * K > 128^3, so AUTO does not take the exact kernel
GEMV_CASES = [
    (1, 1024, 2052, "row", "row", "row", (1.0, 0.0), "smem"),
    (2, 1031, 2052, "row", "colslice", "padded", (0.5, -1.25), "smem"),
    (3, 20000, 776, "row", "negrow", "col", (1.0, 0.0), "smem"),
    (2, 20000, 776, "row", "row", "negcol", (0.5, -1.25), "smem"),
    (4, 1031, 6148, "row", "row", "negcol", (0.5, -1.25), "vec"),       # 4 x 6148 x 4 B > 96 KB of shared memory
    (4, 20000, 6148, "row", "col", "row", (1.0, 0.0), "vec"),
    (1, 1031, 2053, "row", "row", "col", (0.5, -1.25), "scalar"),       # K odd
    (2, 1024, 1100, "col", "row", "row", (1.0, 0.0), "scalar"),
    (3, 20000, 777, "misaligned", "colslice", "padded", (0.5, -1.25), "scalar"),
    (4, 1024, 776, "misaligned", "negrow", "negcol", (1.0, 0.0), "scalar"),
    (3, 1031, 776, "row", "col", "col", (0.5, -1.25), "smem"),
    (4, 20000, 1025, "col", "row", "padded", (0.5, -1.25), "scalar"),
]


@pytest.mark.parametrize("case", GEMV_CASES, ids=lambda c: "N%d-M%d-K%d-%s-%s-%s-b%g-%s" % (c[0], c[1], c[2], c[3], c[4], c[5], c[6][1], c[7]))
def test_gemv(case):
    N, M, K, la, lb, lc, (alpha, beta), variant = case
    assert N <= 4 and M >= 1024 and M * N * K > 128 ** 3 and L.get_f32_mode() != L.PATH_SIMT   # AUTO -> GEMV
    if M == 20000:
        assert M > 8 * 8 * sm_count()      # more rows than one sweep of the grid's warps: the grid-stride loop iterates
    emu_budget(float(M) * N * K)
    A = O.fill_uniform_f32(M * K, 51, -1, 1).reshape(M, K); B = O.fill_uniform_f32(K * N, 52, -1, 1).reshape(K, N)
    C0 = O.fill_uniform_f32(M * N, 53, -1, 1).reshape(M, N) if beta != 0.0 else np.full((M, N), np.nan, np.float32)
    ba, oa, rsa, csa = embed(A, la); bb, ob, rsb, csb = embed(B, lb); bc, oc, rsc, csc = embed(C0, lc)
    ta, tb, tc = dev(ba), dev(bb), dev(bc)
    a_addr = ta.data_ptr() + 4 * oa
    assert gemv_variant(a_addr, rsa, csa, N, K) == variant
    n0 = L.launch_count()
    L.gemm_strided(M, N, K, alpha, L.DevPtr(a_addr, "f32"), rsa, csa, L.DevPtr(tb.data_ptr() + 4 * ob, "f32"), rsb, csb, beta,
                   L.DevPtr(tc.data_ptr() + 4 * oc, "f32"), rsc, csc)
    assert L.launch_count() - n0 == 1 and L.last_path() == L.PATH_SIMT
    sync()
    after = tc.cpu().numpy()
    assert outside_unchanged(after, bc, oc, rsc, csc, M, N), "a write outside the C view"
    got = extract(after, oc, rsc, csc, M, N).astype(np.float64)
    A64, B64 = A.astype(np.float64), B.astype(np.float64)
    c64 = C0.astype(np.float64) if beta != 0.0 else 0.0
    ref = alpha * (A64 @ B64) + beta * c64
    bound = K * 2.0 ** -23 * (abs(alpha) * (np.abs(A64) @ np.abs(B64)) + abs(beta) * np.abs(c64))
    assert np.isfinite(got).all()
    assert np.all(np.abs(got - ref) <= bound), np.max(np.abs(got - ref) / bound)
