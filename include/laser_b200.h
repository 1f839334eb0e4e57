/*
 * laser_b200.h -- C ABI of the B200-native strided GEMM that drops in for
 * mratsim/laser's `gemm_strided` hot path.
 *
 * Every entry point below states the reference interface it replaces
 * (paths relative to the reference checkout, mratsim/laser @ d310294).
 * Plain pointers and sizes only: no torch / C++ types cross this boundary.
 * The Nim binding a maintainer would add is in INTEGRATION.md and nim/laser_b200.nim.
 *
 * Conventions (identical to the reference):
 *   - A is M x K, B is K x N, C is M x N;  C <- alpha * A*B + beta * C
 *   - element (i, j) of a matrix X lives at X[i*rowStrideX + j*colStrideX]
 *     (laser/primitives/matrix_multiplication/gemm_utils.nim:36-60); strides are
 *     in ELEMENTS, may be any int64 (transposed, sliced, non-unit, negative)
 *   - beta == 0 overwrites C without reading it (NaN/garbage in C never
 *     propagates)                      gemm_ukernel_generic.nim:53-76,97-126
 *   - beta is applied once             gemm.nim:158
 *   - the callee never retains A, B, C past return (host variants) or past
 *     completion of the work queued on `stream` (`_dev` variants); A, B must
 *     not alias C
 *
 * Return value: 0 on success, non-zero LASER_B200_E* otherwise;
 * laser_b200_last_error() gives a thread-local message.  The reference
 * returns void and validates nothing (gemm.nim:184-247); the Nim wrapper turns
 * non-zero into an exception.  There is NO CPU fallback: if no sm_100 device
 * is usable every compute entry point fails with LASER_B200_ENODEVICE.
 */
#ifndef LASER_B200_H
#define LASER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LASER_B200_OK 0
#define LASER_B200_EINVAL 1     /* bad argument (negative size, null pointer) */
#define LASER_B200_ENODEVICE 2  /* no usable sm_100 GPU / driver */
#define LASER_B200_ECUDA 3      /* CUDA runtime or driver error */
#define LASER_B200_ENOMEM 4     /* device allocation failed */
#define LASER_B200_EUNSUPPORTED 5

/* Which kernel family executes a float32 gemm_strided call.
 * AUTO: tensor cores in the fp32-faithful mode in force (default F16X3) when the problem is large
 *       enough, exact SIMT otherwise (M*N*K <= 128^3, the reference's own switch, gemm.nim:140-141).
 *       The reference's analogue of this choice is its run-time ISA dispatch, gemm.nim:228-247. */
#define LASER_B200_PATH_AUTO 0
#define LASER_B200_PATH_SIMT 1    /* exact fp32 FFMA chain, bit-equal to the CPU reference order */
#define LASER_B200_PATH_TF32X1 2  /* tcgen05 kind::tf32, one pass over the caller's memory (fast, ~1e-3 relative) */
#define LASER_B200_PATH_TF32X3 3  /* tcgen05 kind::tf32, hi/lo split, three passes (fp32-faithful, any dynamic range) */
#define LASER_B200_PATH_BF16 4    /* tcgen05 kind::f16 (bf16 inputs, fp32 accumulate)         */
/* 5 and 6 were round-1 modes (tf32 + bf16 correction terms; two bf16 pieces): superseded by F16X3, removed */
#define LASER_B200_PATH_F16X3 7   /* DEFAULT fp32 mode.  Every row of A and column of B is scaled by its own power of two
                                   * (device-side abs-max along K, no host synchronisation) and split into two FP16 pieces
                                   * (11 + 11 bits); three kind::f16 passes hi*lo', lo*hi', hi*hi' over tiles loaded once; the
                                   * epilogue undoes the scales.  1.5 tf32-equivalents per MAC; <= 3*2^-22 per product for
                                   * entries within 2^-17 of their row's / column's maximum, smaller entries keep an absolute
                                   * precision of 2^-39 of that maximum (the row/column-norm error model of a blocked GEMM) */

/* ---- life cycle -------------------------------------------------------
 * The reference has one piece of import-time state, cpuinfo_initialize()
 * (laser/cpuinfo.nim:358-360).  Here a per-device context (stream, TMA
 * descriptor cache, split workspace) is created lazily; init/shutdown are
 * optional. */
int laser_b200_init(void);
void laser_b200_shutdown(void);
const char *laser_b200_last_error(void);
int laser_b200_version(void);
/* number of kernels this library has launched on the calling thread's device
 * context since init (used by bench.py's "gpu_launches"). */
int64_t laser_b200_launch_count(void);
/* LASER_B200_PATH_* actually taken by the calling thread's last gemm call. */
int laser_b200_last_path(void);
/* Device-side timing of the library's own kernels (bench.py's roofline numbers):
 * between profile_begin() and profile_end() every tensor-core GEMM launch and every
 * operand-preparation (hi/lo split, pack) launch sequence is bracketed by CUDA events on
 * the stream it is launched on.  profile_end() synchronises and returns the summed
 * durations in milliseconds and the number of bracketed launches. */
int laser_b200_profile_begin(void);
int laser_b200_profile_end(double *gemm_ms, int64_t *gemm_launches, double *prep_ms,
                           int64_t *prep_launches);
/* default path for PATH_AUTO float32 calls: LASER_B200_PATH_F16X3 (default), _TF32X3, _TF32X1 or _SIMT.
 * Also settable with env LASER_B200_F32_MODE=f16x3|tf32x3|tf32x1|simt. */
int laser_b200_set_f32_mode(int path);
int laser_b200_get_f32_mode(void);

/* ---- THE drop-in entry: host pointers ----------------------------------
 * Replaces  proc gemm_strided*[T: SomeNumber](M, N, K: int, alpha: T, A: ptr T,
 *   rowStrideA, colStrideA: int, B: ptr T, rowStrideB, colStrideB: int, beta: T,
 *   C: ptr T, rowStrideC, colStrideC: int)
 *   laser/primitives/matrix_multiplication/gemm.nim:184-193
 * Same argument order and meaning.  A, B, C are HOST pointers: the call stages
 * the touched spans to the GPU, runs, copies C back and returns when C is valid
 * on the host (synchronous, like the reference). */
int laser_b200_gemm_strided_f32(int64_t M, int64_t N, int64_t K, float alpha,
                                const float *A, int64_t rowStrideA, int64_t colStrideA,
                                const float *B, int64_t rowStrideB, int64_t colStrideB,
                                float beta, float *C, int64_t rowStrideC, int64_t colStrideC);
int laser_b200_gemm_strided_f64(int64_t M, int64_t N, int64_t K, double alpha,
                                const double *A, int64_t rowStrideA, int64_t colStrideA,
                                const double *B, int64_t rowStrideB, int64_t colStrideB,
                                double beta, double *C, int64_t rowStrideC, int64_t colStrideC);
int laser_b200_gemm_strided_i32(int64_t M, int64_t N, int64_t K, int32_t alpha,
                                const int32_t *A, int64_t rowStrideA, int64_t colStrideA,
                                const int32_t *B, int64_t rowStrideB, int64_t colStrideB,
                                int32_t beta, int32_t *C, int64_t rowStrideC, int64_t colStrideC);
int laser_b200_gemm_strided_i64(int64_t M, int64_t N, int64_t K, int64_t alpha,
                                const int64_t *A, int64_t rowStrideA, int64_t colStrideA,
                                const int64_t *B, int64_t rowStrideB, int64_t colStrideB,
                                int64_t beta, int64_t *C, int64_t rowStrideC, int64_t colStrideC);
/* bf16 (new dtype, BASELINE.json config 4): buffers hold bf16 bit patterns,
 * alpha/beta and accumulation are fp32, C is rounded RNE to bf16. */
int laser_b200_gemm_strided_bf16(int64_t M, int64_t N, int64_t K, float alpha,
                                 const uint16_t *A, int64_t rowStrideA, int64_t colStrideA,
                                 const uint16_t *B, int64_t rowStrideB, int64_t colStrideB,
                                 float beta, uint16_t *C, int64_t rowStrideC, int64_t colStrideC);

/* ---- device-resident variants (what the metric is measured on) ---------
 * Same contract as above (gemm.nim:184-193) with DEVICE pointers on the
 * current device, asynchronous on `stream` (a cudaStream_t passed as void*;
 * NULL = the library's own stream, synchronised before return; to run on the legacy default
 * stream pass cudaStreamLegacy, i.e. (void*)0x1).
 * `path` is a LASER_B200_PATH_* value. */
int laser_b200_gemm_strided_f32_dev(int64_t M, int64_t N, int64_t K, float alpha,
                                    const float *A, int64_t rowStrideA, int64_t colStrideA,
                                    const float *B, int64_t rowStrideB, int64_t colStrideB,
                                    float beta, float *C, int64_t rowStrideC, int64_t colStrideC,
                                    int path, void *stream);
int laser_b200_gemm_strided_f64_dev(int64_t M, int64_t N, int64_t K, double alpha,
                                    const double *A, int64_t rowStrideA, int64_t colStrideA,
                                    const double *B, int64_t rowStrideB, int64_t colStrideB,
                                    double beta, double *C, int64_t rowStrideC, int64_t colStrideC,
                                    void *stream);
int laser_b200_gemm_strided_i32_dev(int64_t M, int64_t N, int64_t K, int32_t alpha,
                                    const int32_t *A, int64_t rowStrideA, int64_t colStrideA,
                                    const int32_t *B, int64_t rowStrideB, int64_t colStrideB,
                                    int32_t beta, int32_t *C, int64_t rowStrideC, int64_t colStrideC,
                                    void *stream);
int laser_b200_gemm_strided_i64_dev(int64_t M, int64_t N, int64_t K, int64_t alpha,
                                    const int64_t *A, int64_t rowStrideA, int64_t colStrideA,
                                    const int64_t *B, int64_t rowStrideB, int64_t colStrideB,
                                    int64_t beta, int64_t *C, int64_t rowStrideC, int64_t colStrideC,
                                    void *stream);
int laser_b200_gemm_strided_bf16_dev(int64_t M, int64_t N, int64_t K, float alpha,
                                     const uint16_t *A, int64_t rowStrideA, int64_t colStrideA,
                                     const uint16_t *B, int64_t rowStrideB, int64_t colStrideB,
                                     float beta, uint16_t *C, int64_t rowStrideC, int64_t colStrideC,
                                     void *stream);

/* ---- fused epilogue ------------------------------------------------------
 * C <- act(alpha * A*B + beta * C + bias).  The reference lists this as the intended next step
 * of exactly the epilogue replaced here ("TODO: elementwise epilogue fusion like
 * relu/tanh/sigmoid", gemm.nim:196; gemm_ukernel_generic.nim:50-51,78-79,128-129).
 * bias: NULL, or a device vector added per column (length N, bias_per_row = 0) or per row
 * (length M, bias_per_row = 1).  epi == NULL behaves like laser_b200_gemm_strided_f32_dev. */
#define LASER_B200_ACT_NONE 0
#define LASER_B200_ACT_RELU 1
#define LASER_B200_ACT_TANH 2
#define LASER_B200_ACT_SIGMOID 3
typedef struct {
  const float *bias;
  int32_t bias_per_row;
  int32_t activation;
} laser_b200_epilogue;
int laser_b200_gemm_strided_f32_epi_dev(int64_t M, int64_t N, int64_t K, float alpha,
                                        const float *A, int64_t rowStrideA, int64_t colStrideA,
                                        const float *B, int64_t rowStrideB, int64_t colStrideB,
                                        float beta, float *C, int64_t rowStrideC, int64_t colStrideC,
                                        const laser_b200_epilogue *epi, int path, void *stream);

/* ---- pre-packed operands (device) -----------------------------------------
 * Replaces  gemm_prepackA_mem_required / gemm_prepackB_mem_required, gemm_prepackA / gemm_prepackB
 * and gemm_packed   (laser/primitives/matrix_multiplication/gemm_prepacked.nim:63-292).
 * The reference packs an operand once into micro-panels so that repeated products with the same
 * matrix skip the packing pass; here "packing" is the operand preparation of the default
 * fp32-faithful mode (two fp16 pieces of the scaled operand, K-major compact, plus the per-row
 * scale words), so repeated products skip the preparation pass and read TMA-friendly K-major
 * tiles whatever the source strides were.  Packed buffers are opaque DEVICE memory owned by the caller, sized by
 * *_mem_required (bytes), 256-byte aligned; like the reference's they are only meaningful to the
 * library build that wrote them ("unsafe to store or serialize", gemm_prepacked.nim:120-123).
 * M, N, K are the extents of the product the operand will take part in (A is M x K, B is K x N). */
size_t laser_b200_gemm_prepackA_mem_required_f32(int64_t M, int64_t N, int64_t K);
size_t laser_b200_gemm_prepackB_mem_required_f32(int64_t M, int64_t N, int64_t K);
int laser_b200_gemm_prepackA_f32_dev(void *dst_packedA, int64_t M, int64_t N, int64_t K,
                                     const float *A, int64_t rowStrideA, int64_t colStrideA,
                                     void *stream);
int laser_b200_gemm_prepackB_f32_dev(void *dst_packedB, int64_t M, int64_t N, int64_t K,
                                     const float *B, int64_t rowStrideB, int64_t colStrideB,
                                     void *stream);
/* C <- alpha * A*B + beta * C with both operands pre-packed (gemm_packed, gemm_prepacked.nim:275-292) */
int laser_b200_gemm_packed_f32_dev(int64_t M, int64_t N, int64_t K, float alpha,
                                   const void *packedA, const void *packedB, float beta, float *C,
                                   int64_t rowStrideC, int64_t colStrideC, void *stream);
/* the common case: a fixed (pre-packed) B, a fresh A with any strides */
int laser_b200_gemm_packedB_f32_dev(int64_t M, int64_t N, int64_t K, float alpha, const float *A,
                                    int64_t rowStrideA, int64_t colStrideA, const void *packedB,
                                    float beta, float *C, int64_t rowStrideC, int64_t colStrideC,
                                    void *stream);

/* ---- row panels of C across the GPUs of one box (SURVEY.md 8e) ---------------------------------
 * The reference parallelises this split inside gemm_strided itself: its `ic` loop hands every worker a row block of A
 * and C while all workers share one packed panel of B (gemm.nim:160-176).  Here a worker is a GPU: rank r owns rows of
 * A and C (never moved); B lives on `root` and travels ONCE per product over NCCL (NVLink 5 / NVSwitch) on a
 * communication stream, while the rank's rows of A are already being prepared; no collective inside the MMA loop, no
 * reduction.  In the default fp32 mode a row- or column-major B travels PREPARED -- the fp16 pieces and scale words the
 * tensor-core kernel reads, the same 4 bytes per element -- in LASER_B200_ROWSHARD_PANELS column panels (default 1; with more, the
 * root prepares panel p + 1 while panel p is on the wire and every rank multiplies its rows by panel p as soon as it is
 * there); only the root ever prepares B, and while the other ranks still multiply it is already preparing the next product's.  Otherwise (other modes, general strides, LASER_B200_ROWSHARD_PANELS=0) B itself
 * is broadcast and every rank prepares it.  NCCL is bound at run time (dlopen of libnccl.so.2); without it these entries return LASER_B200_EUNSUPPORTED.
 *
 *   comm_get_unique_id / comm_init_rank   one process (or thread) per GPU: rank 0 obtains the 128-byte id, hands it to
 *                                         the others by any means, every rank calls init_rank with ITS device current
 *   comm_init_all                         one process driving devices 0 .. ngpus-1 (ncclCommInitAll)
 *   rowshard_partition                    the row range of a rank: ceil(M / nranks) rounded up to the 256-row tile
 *   gemm_rowsharded_f32_dev               per-rank entry, DEVICE pointers on the communicator's device, asynchronous on
 *                                         `stream`: C_local <- alpha * A_local * B + beta * C_local with B (K x N, dense in
 *                                         memory) an input on `root`; on every other rank the buffer is scratch (filled
 *                                         with B by the raw broadcast, left alone when B travels prepared)
 *   gemm_rowsharded_f32                   the reference signature with HOST pointers on `ngpus` devices of this process:
 *                                         row panels of A (and of C when beta != 0) go to their device, B to device 0,
 *                                         one broadcast, every device its rows, C comes back; synchronous */
typedef struct laser_b200_comm laser_b200_comm;
#define LASER_B200_UNIQUE_ID_BYTES 128
int laser_b200_comm_get_unique_id(void *id128);
int laser_b200_comm_init_rank(laser_b200_comm **comm, int nranks, int rank, const void *id128);
int laser_b200_comm_init_all(laser_b200_comm **comms, int ngpus);
int laser_b200_comm_destroy(laser_b200_comm *comm);
int laser_b200_comm_rank(const laser_b200_comm *comm);
int laser_b200_comm_size(const laser_b200_comm *comm);
void laser_b200_rowshard_partition(int64_t M, int nranks, int rank, int64_t *first_row, int64_t *rows);
int laser_b200_gemm_rowsharded_f32_dev(laser_b200_comm *comm, int64_t M_local, int64_t N, int64_t K, float alpha,
                                       const float *A_local, int64_t rowStrideA, int64_t colStrideA,
                                       float *B, int64_t rowStrideB, int64_t colStrideB, int root,
                                       float beta, float *C_local, int64_t rowStrideC, int64_t colStrideC,
                                       void *stream);
int laser_b200_gemm_rowsharded_f32(int ngpus, int64_t M, int64_t N, int64_t K, float alpha,
                                   const float *A, int64_t rowStrideA, int64_t colStrideA,
                                   const float *B, int64_t rowStrideB, int64_t colStrideB,
                                   float beta, float *C, int64_t rowStrideC, int64_t colStrideC);

/* ---- device storage for the Tensor contract ----------------------------
 * Device analogue of allocCpuStorage (laser/tensor/allocator.nim:17-29: 64-byte
 * aligned, owned by the storage object) and of copyFromRaw / setZero
 * (laser/tensor/initialization.nim:80-154).  Pointers returned are >= 256-byte
 * aligned device addresses. */
int laser_b200_malloc(void **dev_ptr, size_t bytes);
int laser_b200_free(void *dev_ptr);
int laser_b200_memcpy_h2d(void *dst_dev, const void *src_host, size_t bytes);
int laser_b200_memcpy_d2h(void *dst_host, const void *src_dev, size_t bytes);
int laser_b200_memset_zero(void *dst_dev, size_t bytes);
int laser_b200_synchronize(void);

/* POD view of a Tensor: what laser/tensor/datatypes.nim:18-22 exposes through
 * rank / shape / strides / offset / unsafe_raw_data (strides and offset in
 * elements, LASER_MAXRANK = 6, laser/dynamic_stack_arrays.nim:6). */
#define LASER_B200_MAXRANK 6
typedef struct {
  int32_t rank;
  int32_t dtype; /* 0 f32, 1 f64, 2 i32, 3 i64, 4 bf16 */
  int64_t shape[LASER_B200_MAXRANK];
  int64_t strides[LASER_B200_MAXRANK];
  int64_t offset;
  void *storage; /* device base pointer; unsafe_raw_data = storage + offset */
} laser_b200_tensor_view;

/* C <- alpha * A x B + beta * C on rank-2 device tensor views (any strides):
 * the tensor-level caller of gemm_strided, as gemm_prepacked.nim:306-307 does
 * with `cast[ptr T](t.unsafe_raw_data)`. */
int laser_b200_matmul_views(const laser_b200_tensor_view *A, const laser_b200_tensor_view *B,
                            laser_b200_tensor_view *C, double alpha, double beta, int path,
                            void *stream);

/* ---- the steps either side of the GEMM (SURVEY.md 8f rank 4) -------------------------------
 * Batched GEMM: problem b reads A + b*batchStrideA, B + b*batchStrideB and writes
 * C + b*batchStrideC (strides in elements; a batch stride of 0 shares that operand, e.g. one
 * filter matrix against many images; the outputs of different problems must not overlap).
 * Problems the dispatch sends to the exact kernel (path SIMT, or AUTO with M*N*K <= 128^3) run as
 * ONE launch; tensor-core problems take one launch sequence each.  The reference has no batched entry -- its README lists it
 * as roadmap (README.md:253-263); each problem follows gemm_strided (gemm.nim:184-193). */
int laser_b200_gemm_strided_batched_f32_dev(int64_t batch, int64_t M, int64_t N, int64_t K, float alpha,
                                            const float *A, int64_t rowStrideA, int64_t colStrideA,
                                            int64_t batchStrideA, const float *B, int64_t rowStrideB,
                                            int64_t colStrideB, int64_t batchStrideB, float beta, float *C,
                                            int64_t rowStrideC, int64_t colStrideC, int64_t batchStrideC,
                                            int path, void *stream);

/* f64 / i32 / i64 batches: the exact kernel, always one launch */
int laser_b200_gemm_strided_batched_f64_dev(int64_t batch, int64_t M, int64_t N, int64_t K, double alpha,
                                            const double *A, int64_t rowStrideA, int64_t colStrideA,
                                            int64_t batchStrideA, const double *B, int64_t rowStrideB,
                                            int64_t colStrideB, int64_t batchStrideB, double beta, double *C,
                                            int64_t rowStrideC, int64_t colStrideC, int64_t batchStrideC,
                                            void *stream);
int laser_b200_gemm_strided_batched_i32_dev(int64_t batch, int64_t M, int64_t N, int64_t K, int32_t alpha,
                                            const int32_t *A, int64_t rowStrideA, int64_t colStrideA,
                                            int64_t batchStrideA, const int32_t *B, int64_t rowStrideB,
                                            int64_t colStrideB, int64_t batchStrideB, int32_t beta, int32_t *C,
                                            int64_t rowStrideC, int64_t colStrideC, int64_t batchStrideC,
                                            void *stream);
int laser_b200_gemm_strided_batched_i64_dev(int64_t batch, int64_t M, int64_t N, int64_t K, int64_t alpha,
                                            const int64_t *A, int64_t rowStrideA, int64_t colStrideA,
                                            int64_t batchStrideA, const int64_t *B, int64_t rowStrideB,
                                            int64_t colStrideB, int64_t batchStrideB, int64_t beta, int64_t *C,
                                            int64_t rowStrideC, int64_t colStrideC, int64_t batchStrideC,
                                            void *stream);

/* Physical transposition of contiguous matrices, elem_size in {1, 2, 4, 8} bytes
 * (generic T in the reference):
 *   transpose2D_copy(dst, src, NR, NC)         laser/primitives/swapaxes.nim:16-54
 *   transpose2D_batched(dst, src, N, NR, NC)   swapaxes.nim:56-81
 *   nchw2nhwc / nhwc2nchw(dst, src, N,C,H,W)   swapaxes.nim:83-112
 * dst is overwritten and must not alias src.  Plain names take host pointers and are
 * synchronous (the reference's contract); _dev names take device pointers + stream. */
int laser_b200_transpose2D_copy(void *dst, const void *src, int64_t NR, int64_t NC, int elem_size);
int laser_b200_transpose2D_batched(void *dst, const void *src, int64_t N, int64_t NR, int64_t NC,
                                   int elem_size);
int laser_b200_nchw2nhwc(void *dst_nhwc, const void *src_nchw, int64_t N, int64_t C, int64_t H, int64_t W,
                         int elem_size);
int laser_b200_nhwc2nchw(void *dst_nchw, const void *src_nhwc, int64_t N, int64_t C, int64_t H, int64_t W,
                         int elem_size);
int laser_b200_transpose2D_copy_dev(void *dst, const void *src, int64_t NR, int64_t NC, int elem_size,
                                    void *stream);
int laser_b200_transpose2D_batched_dev(void *dst, const void *src, int64_t N, int64_t NR, int64_t NC,
                                       int elem_size, void *stream);
int laser_b200_nchw2nhwc_dev(void *dst_nhwc, const void *src_nchw, int64_t N, int64_t C, int64_t H,
                             int64_t W, int elem_size, void *stream);
int laser_b200_nhwc2nchw_dev(void *dst_nchw, const void *src_nhwc, int64_t N, int64_t C, int64_t H,
                             int64_t W, int elem_size, void *stream);

/* im2col convolution (benchmarks/convolution/conv2d_im2col.nim, shapes as in conv2d_common.nim:6-10):
 *   ishape = (n, c, h, w)  kshape = (c_out, c_in, kH, kW)  padding = (h, w)  strides = (h, w)
 *   conv2d_out_shape        conv2d_common.nim:15-45 (EINVAL unless 0 < stride < extent, :35-36)
 *   im2col_workspace_size   conv2d_im2col.nim:8-18: ELEMENTS for one image, c*kH*kW*outH*outW
 *   im2col                  conv2d_im2col.nim:44-93: `images` images [c][h][w] (image stride
 *                           c*h*w) -> `images` matrices [c*kH*kW][outH*outW], zero padding
 *   conv2d_im2col           conv2d_im2col.nim:95-166: NCHW in, NCHW out (fully overwritten,
 *                           alpha 1 / beta 0), per image O[c_out x outHW] = F[c_out x K] * W[K x outHW]
 *                           through gemm_strided; `workspace` holds workspace_images >= 1 images
 *                           (the reference's buffer holds one and is reused between images; a
 *                           larger one lets several images share one im2col launch and one batched
 *                           GEMM).  1x1 kernels with unit stride and no padding skip im2col (:121).
 *                           Divergence: the reference takes that shortcut for every 1x1 kernel, which
 *                           is wrong for strided/padded ones; those go through im2col here. */
int laser_b200_conv2d_out_shape(const int64_t ishape[4], const int64_t kshape[4], const int64_t padding[2],
                                const int64_t strides[2], int64_t oshape[4]);
int64_t laser_b200_im2col_workspace_size(const int64_t ishape[4], const int64_t kshape[4],
                                         const int64_t padding[2], const int64_t strides[2]);
int laser_b200_im2col_f32_dev(float *workspace, const float *input, int64_t images, const int64_t ishape[4],
                              const int64_t kshape[4], const int64_t padding[2], const int64_t strides[2],
                              void *stream);
int laser_b200_conv2d_im2col_f32_dev(float *output, const float *input, const int64_t ishape[4],
                                     const float *kernel, const int64_t kshape[4], const int64_t padding[2],
                                     const int64_t strides[2], float *workspace, int64_t workspace_images,
                                     int path, void *stream);
/* host pointers, synchronous, library-owned workspace */
int laser_b200_conv2d_im2col_f32(float *output, const float *input, const int64_t ishape[4],
                                 const float *kernel, const int64_t kshape[4], const int64_t padding[2],
                                 const int64_t strides[2]);

/* direct convolution (benchmarks/convolution/conv2d_direct_convolution.nim:8-76): the same shapes as
 * conv2d_im2col (validated by the same checks), no workspace, ONE kernel launch per call whatever the batch
 * (none for a batch of 0, which leaves `output` untouched).  Every output element is bit for bit what
 * laser_b200_conv2d_im2col_f32_dev(..., path = LASER_B200_PATH_SIMT) returns: one FMA chain from +0 over
 * ascending tap kk = (ci*kH + kr)*kW + kc inside blocks of 512 taps, the blocks added in order.
 * epi: NULL, or bias = NULL / a device vector of c_out values (requires bias_per_row = 1) and an activation
 * 0..3, applied once to the final sum as act(x + bias[co]) -- the values im2col followed by
 * laser_b200_gemm_strided_f32_epi_dev(path SIMT, bias_per_row = 1) gives.  Anything else: EINVAL.
 * Deliberate departures from the reference:
 *   - `output` is overwritten and never read (the reference adds into a zero-initialised `oim`);
 *   - the output column steps the input by the WIDTH stride (the reference multiplies it by the height
 *     stride, conv2d_direct_convolution.nim:61, which differs for non-square strides);
 *   - taps outside the image contribute fma(0, w) like the zeros of the im2col workspace (the reference
 *     skips them), so an infinite weight makes the border outputs NaN exactly as conv2d_im2col does. */
int laser_b200_conv2d_direct_f32_dev(float *output, const float *input, const int64_t ishape[4],
                                     const float *kernel, const int64_t kshape[4], const int64_t padding[2],
                                     const int64_t strides[2], const laser_b200_epilogue *epi, void *stream);
/* host pointers, synchronous, no epilogue: the reference's conv2d_direct signature */
int laser_b200_conv2d_direct_f32(float *output, const float *input, const int64_t ishape[4],
                                 const float *kernel, const int64_t kshape[4], const int64_t padding[2],
                                 const int64_t strides[2]);

/* dst <- src over a common shape, any strides (device tensor views of the same dtype and shape):
 * copyFrom of laser/tensor/initialization.nim:80-112 (contiguous pairs take a plain device copy,
 * the rest the strided kernel -- the reference's forEachStrided d in dst, s in src: d = s). */
int laser_b200_copy_views(laser_b200_tensor_view *dst, const laser_b200_tensor_view *src, void *stream);

/* forEach over up to four equal-shape device tensor views of any strides (float32 / float64):
 *   forEach o in out, x in a, y in b, z in c: <body>     laser/strided_iteration/foreach.nim:229-251
 * An arbitrary body cannot cross a C ABI; the bodies the reference's own code, documentation and
 * iteration benchmark use are opcodes.  Operands an opcode does not read may be NULL; `out` may
 * alias an input element for element (in-place updates). */
#define LASER_B200_FOREACH_COPY 0   /* o = x                 (initialization.nim:68,104) */
#define LASER_B200_FOREACH_FILL 1   /* o = alpha */
#define LASER_B200_FOREACH_SCALE 2  /* o = alpha * x */
#define LASER_B200_FOREACH_ADD 3    /* o = x + y */
#define LASER_B200_FOREACH_SUB 4    /* o = x - y */
#define LASER_B200_FOREACH_MUL 5    /* o = x * y */
#define LASER_B200_FOREACH_FMA 6    /* o = x + y * z         (`x += y * z`, foreach.nim:231-232) */
#define LASER_B200_FOREACH_AXPY 7   /* o = alpha * x + y */
#define LASER_B200_FOREACH_BENCH 8  /* o = x + y - sin(z)    (benchmarks/loop_iteration/iter_bench_prod.nim:88-90) */
int laser_b200_foreach_views(int op, laser_b200_tensor_view *out, const laser_b200_tensor_view *x,
                             const laser_b200_tensor_view *y, const laser_b200_tensor_view *z, double alpha,
                             void *stream);

/* ---- host-logic introspection (pure functions, no GPU needed; used by the CPU tests) --------
 * classify: how the tensor-core path would feed an operand seen as [mn][k] with element strides
 * (s_mn, s_k): 0 = K-major TMA, 1 = MN-major TMA, 2 = general (gathered by pack_general_kernel).
 * span: lowest/highest element offset touched by a rows x cols view and whether the view is dense
 * in that span (decides what the host-pointer entry has to copy). */
int laser_b200_debug_classify(int elem_size, const void *base, int64_t s_mn, int64_t s_k);
int laser_b200_debug_span(int64_t rows, int64_t cols, int64_t row_stride, int64_t col_stride,
                          int64_t *lo, int64_t *hi, int *dense);
/* launches of the fp64 tensor-core kernel (mma.sync DMMA, csrc/gemm_dmma.cuh) since the library was loaded: float64
 * problems whose 128 x 128 tiles fill at least half of the SMs take it instead of the CUDA-core kernel (same FMA chain
 * per element, bit for bit; LASER_B200_F64_DMMA=0 turns it off) -- gemm.nim:234-246, the float64 row of the dispatch */
int64_t laser_b200_debug_f64_dmma_launches(void);

/* ---- synthetic inputs ---------------------------------------------------
 * Counter-based uniform generator, bit-identical to the CPU oracle's
 * (oracle_fill_uniform_f32); stands in for the reference bench's
 * randomize(42) + rand(-0.1..0.1) (benchmarks/gemm/gemm_bench_float32.nim:329,343-344). */
int laser_b200_fill_uniform_f32_dev(float *dst_dev, int64_t n, uint64_t seed, float lo, float hi,
                                    void *stream);

#ifdef __cplusplus
}
#endif
#endif /* LASER_B200_H */
