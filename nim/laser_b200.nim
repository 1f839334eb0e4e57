# laser_b200.nim -- the Nim side of the drop-in boundary.
#
# A thin {.importc.} shim over liblaser_b200.so (C ABI: include/laser_b200.h) that gives Nim
# callers the reference's own API for the hot path:
#
#   gemm_strided(M, N, K, alpha, A, rowStrideA, colStrideA, B, rowStrideB, colStrideB,
#                beta, C, rowStrideC, colStrideC)
#
# with exactly the signature of laser/primitives/matrix_multiplication/gemm.nim:184-193, so
# that `import laser_b200` can replace `import laser/primitives/matrix_multiplication/gemm`
# at a call site such as benchmarks/gemm/gemm_bench_float32.nim:184-189 without touching it.
# FFI idiom: the reference's own (benchmarks/third_party/blas.nim:18-23: importc + dynlib).
#
# NOTE: no Nim toolchain exists in the build image, so this file is shipped untested; every
# symbol it imports is exercised through the identical C ABI by tests/ (ctypes) instead.

const laserB200Lib* {.strdefine.} = "liblaser_b200.so"

type
  LaserB200Error* = object of CatchableError   # cf. LibraryError in laser/cpuinfo.nim:358-359

  GemmPath* {.size: sizeof(cint).} = enum      # LASER_B200_PATH_*
    pathAuto = 0, pathSimt = 1, pathTf32x1 = 2, pathTf32x3 = 3, pathBf16 = 4, pathF16x3 = 7   # 7: the default fp32 mode

{.push importc, cdecl, dynlib: laserB200Lib.}
proc laser_b200_init*(): cint
proc laser_b200_shutdown*()
proc laser_b200_last_error*(): cstring
proc laser_b200_set_f32_mode*(path: cint): cint
proc laser_b200_gemm_strided_f32*(M, N, K: int64, alpha: float32,
    A: ptr float32, rowStrideA, colStrideA: int64,
    B: ptr float32, rowStrideB, colStrideB: int64,
    beta: float32, C: ptr float32, rowStrideC, colStrideC: int64): cint
proc laser_b200_gemm_strided_f64*(M, N, K: int64, alpha: float64,
    A: ptr float64, rowStrideA, colStrideA: int64,
    B: ptr float64, rowStrideB, colStrideB: int64,
    beta: float64, C: ptr float64, rowStrideC, colStrideC: int64): cint
proc laser_b200_gemm_strided_i32*(M, N, K: int64, alpha: int32,
    A: ptr int32, rowStrideA, colStrideA: int64,
    B: ptr int32, rowStrideB, colStrideB: int64,
    beta: int32, C: ptr int32, rowStrideC, colStrideC: int64): cint
proc laser_b200_gemm_strided_i64*(M, N, K: int64, alpha: int64,
    A: ptr int64, rowStrideA, colStrideA: int64,
    B: ptr int64, rowStrideB, colStrideB: int64,
    beta: int64, C: ptr int64, rowStrideC, colStrideC: int64): cint
# bf16 (a dtype the reference does not have: BASELINE.json config 4): buffers hold bf16 bit patterns, alpha / beta and the
# accumulation are float32, C is rounded to nearest-even
proc laser_b200_gemm_strided_bf16*(M, N, K: int64, alpha: float32,
    A: ptr uint16, rowStrideA, colStrideA: int64,
    B: ptr uint16, rowStrideB, colStrideB: int64,
    beta: float32, C: ptr uint16, rowStrideC, colStrideC: int64): cint
proc laser_b200_gemm_strided_bf16_dev*(M, N, K: int64, alpha: float32,
    A: ptr uint16, rowStrideA, colStrideA: int64,
    B: ptr uint16, rowStrideB, colStrideB: int64,
    beta: float32, C: ptr uint16, rowStrideC, colStrideC: int64, stream: pointer): cint
# row panels of C across the GPUs of the box (the `ic` loop of gemm.nim:160-176 with GPUs as workers)
proc laser_b200_comm_get_unique_id*(id128: pointer): cint
proc laser_b200_comm_init_rank*(comm: ptr pointer, nranks, rank: cint, id128: pointer): cint
proc laser_b200_comm_init_all*(comms: ptr pointer, ngpus: cint): cint
proc laser_b200_comm_destroy*(comm: pointer): cint
proc laser_b200_comm_rank*(comm: pointer): cint
proc laser_b200_comm_size*(comm: pointer): cint
proc laser_b200_rowshard_partition*(M: int64, nranks, rank: cint, firstRow, rows: ptr int64)
proc laser_b200_gemm_rowsharded_f32_dev*(comm: pointer, M_local, N, K: int64, alpha: float32,
    A_local: ptr float32, rowStrideA, colStrideA: int64,
    B: ptr float32, rowStrideB, colStrideB: int64, root: cint,
    beta: float32, C_local: ptr float32, rowStrideC, colStrideC: int64, stream: pointer): cint
proc laser_b200_gemm_rowsharded_f32*(ngpus: cint, M, N, K: int64, alpha: float32,
    A: ptr float32, rowStrideA, colStrideA: int64,
    B: ptr float32, rowStrideB, colStrideB: int64,
    beta: float32, C: ptr float32, rowStrideC, colStrideC: int64): cint
proc laser_b200_gemm_strided_f32_dev*(M, N, K: int64, alpha: float32,
    A: ptr float32, rowStrideA, colStrideA: int64,
    B: ptr float32, rowStrideB, colStrideB: int64,
    beta: float32, C: ptr float32, rowStrideC, colStrideC: int64,
    path: cint, stream: pointer): cint
# pre-packed operands (gemm_prepacked.nim:63-292) and fused epilogue (gemm.nim:196 TODO)
proc laser_b200_gemm_prepackA_mem_required_f32*(M, N, K: int64): csize_t
proc laser_b200_gemm_prepackB_mem_required_f32*(M, N, K: int64): csize_t
proc laser_b200_gemm_prepackA_f32_dev*(dst: pointer, M, N, K: int64, A: ptr float32,
    rowStrideA, colStrideA: int64, stream: pointer): cint
proc laser_b200_gemm_prepackB_f32_dev*(dst: pointer, M, N, K: int64, B: ptr float32,
    rowStrideB, colStrideB: int64, stream: pointer): cint
proc laser_b200_gemm_packed_f32_dev*(M, N, K: int64, alpha: float32, packedA, packedB: pointer,
    beta: float32, C: ptr float32, rowStrideC, colStrideC: int64, stream: pointer): cint
proc laser_b200_gemm_packedB_f32_dev*(M, N, K: int64, alpha: float32, A: ptr float32,
    rowStrideA, colStrideA: int64, packedB: pointer, beta: float32, C: ptr float32,
    rowStrideC, colStrideC: int64, stream: pointer): cint
proc laser_b200_malloc*(devPtr: ptr pointer, bytes: csize_t): cint
proc laser_b200_free*(devPtr: pointer): cint
proc laser_b200_memcpy_h2d*(dst, src: pointer, bytes: csize_t): cint
proc laser_b200_memcpy_d2h*(dst, src: pointer, bytes: csize_t): cint
proc laser_b200_memset_zero*(dst: pointer, bytes: csize_t): cint
{.pop.}

template check(code: cint) =
  if code != 0:
    raise newException(LaserB200Error, $laser_b200_last_error())

# ---- bf16 and multi-GPU flavours of the same call ------------------------------------------------------
type BFloat16* = distinct uint16     # bit pattern of a bfloat16

proc gemm_strided*(M, N, K: int, alpha: float32,
                   A: ptr BFloat16, rowStrideA, colStrideA: int,
                   B: ptr BFloat16, rowStrideB, colStrideB: int,
                   beta: float32,
                   C: ptr BFloat16, rowStrideC, colStrideC: int) =
  check laser_b200_gemm_strided_bf16(M, N, K, alpha, cast[ptr uint16](A), rowStrideA, colStrideA,
                                     cast[ptr uint16](B), rowStrideB, colStrideB, beta,
                                     cast[ptr uint16](C), rowStrideC, colStrideC)

proc gemm_strided_rowsharded*(ngpus: int, M, N, K: int, alpha: float32,
                              A: ptr float32, rowStrideA, colStrideA: int,
                              B: ptr float32, rowStrideB, colStrideB: int,
                              beta: float32,
                              C: ptr float32, rowStrideC, colStrideC: int) =
  ## gemm_strided on host matrices with the row blocks of A and C spread over `ngpus` GPUs of this process and one
  ## NCCL broadcast of B (the reference's `ic` loop, gemm.nim:160-176, with GPUs as workers)
  check laser_b200_gemm_rowsharded_f32(ngpus.cint, M, N, K, alpha, A, rowStrideA, colStrideA,
                                       B, rowStrideB, colStrideB, beta, C, rowStrideC, colStrideC)

# ---- the drop-in overloads: same parameter list as gemm.nim:184-193 -------------------
proc gemm_strided*(M, N, K: int, alpha: float32,
                   A: ptr float32, rowStrideA, colStrideA: int,
                   B: ptr float32, rowStrideB, colStrideB: int,
                   beta: float32,
                   C: ptr float32, rowStrideC, colStrideC: int) =
  check laser_b200_gemm_strided_f32(M, N, K, alpha, A, rowStrideA, colStrideA,
                                    B, rowStrideB, colStrideB, beta, C, rowStrideC, colStrideC)

proc gemm_strided*(M, N, K: int, alpha: float64,
                   A: ptr float64, rowStrideA, colStrideA: int,
                   B: ptr float64, rowStrideB, colStrideB: int,
                   beta: float64,
                   C: ptr float64, rowStrideC, colStrideC: int) =
  check laser_b200_gemm_strided_f64(M, N, K, alpha, A, rowStrideA, colStrideA,
                                    B, rowStrideB, colStrideB, beta, C, rowStrideC, colStrideC)

proc gemm_strided*(M, N, K: int, alpha: int32,
                   A: ptr int32, rowStrideA, colStrideA: int,
                   B: ptr int32, rowStrideB, colStrideB: int,
                   beta: int32,
                   C: ptr int32, rowStrideC, colStrideC: int) =
  check laser_b200_gemm_strided_i32(M, N, K, alpha, A, rowStrideA, colStrideA,
                                    B, rowStrideB, colStrideB, beta, C, rowStrideC, colStrideC)

proc gemm_strided*(M, N, K: int, alpha: int,
                   A: ptr int, rowStrideA, colStrideA: int,
                   B: ptr int, rowStrideB, colStrideB: int,
                   beta: int,
                   C: ptr int, rowStrideC, colStrideC: int) =
  check laser_b200_gemm_strided_i64(M, N, K, alpha.int64, cast[ptr int64](A), rowStrideA, colStrideA,
                                    cast[ptr int64](B), rowStrideB, colStrideB, beta.int64,
                                    cast[ptr int64](C), rowStrideC, colStrideC)

# ---- device tensor honouring laser/tensor's contract (datatypes.nim:12-88) -----------
# Same fields and accessors as Tensor[T]; storage lives in HBM.  Metadata mirrors
# DynamicStackArray[int] with LASER_MAXRANK = 6 (laser/dynamic_stack_arrays.nim:6,14-19).
const LASER_MAXRANK* = 6
type
  Metadata* = object
    data*: array[LASER_MAXRANK, int]
    len*: int
  CudaStorage*[T] = ref object
    raw_buffer*: ptr UncheckedArray[T]   # device address
    memowner*: bool
  CudaTensor*[T] = object
    shape*, strides*: Metadata           # strides in elements
    offset*: int
    storage*: CudaStorage[T]

proc finalizer[T](s: CudaStorage[T]) =
  if s.memowner and not s.raw_buffer.isNil: discard laser_b200_free(s.raw_buffer)

func rank*(t: CudaTensor): int {.inline.} = t.shape.len
func size*(t: CudaTensor): int =
  result = 1
  for i in 0 ..< t.shape.len: result *= t.shape.data[i]
func is_C_contiguous*(t: CudaTensor): bool =
  var cur = 1
  for i in countdown(t.rank - 1, 0):
    if t.shape.data[i] != 1 and t.strides.data[i] != cur: return false
    cur *= t.shape.data[i]
  true
func unsafe_raw_data*[T](t: CudaTensor[T]): ptr T {.inline.} =
  ## device address of element [0, ..., 0] (storage + offset), datatypes.nim:64-88
  cast[ptr T](t.storage.raw_buffer[t.offset].addr)

proc newCudaTensor*[T](shape: varargs[int]): CudaTensor[T] =
  ## zero-initialised row-major device tensor (initialization.nim:156-170)
  result.shape.len = shape.len
  result.strides.len = shape.len
  var acc = 1
  for i in countdown(shape.len - 1, 0):
    result.shape.data[i] = shape[i]
    result.strides.data[i] = acc
    acc *= shape[i]
  new(result.storage, finalizer[T])
  var p: pointer
  check laser_b200_malloc(p.addr, csize_t(acc * sizeof(T)))
  check laser_b200_memset_zero(p, csize_t(acc * sizeof(T)))
  result.storage.raw_buffer = cast[ptr UncheckedArray[T]](p)
  result.storage.memowner = true

# ---- pre-packed API with the reference's names (gemm_prepacked.nim) on device tensors ----
proc gemm_prepackB_mem_required*(M, N, K: int): int =
  int laser_b200_gemm_prepackB_mem_required_f32(M, N, K)
proc gemm_prepackA_mem_required*(M, N, K: int): int =
  int laser_b200_gemm_prepackA_mem_required_f32(M, N, K)
proc gemm_prepackB*(dst_packedB: pointer, M, N, K: int, src_B: ptr float32,
                    rowStrideB, colStrideB: int) =
  ## dst_packedB, src_B: device pointers (gemm_prepacked.nim:111-135)
  check laser_b200_gemm_prepackB_f32_dev(dst_packedB, M, N, K, src_B, rowStrideB, colStrideB, nil)
proc gemm_prepackA*(dst_packedA: pointer, M, N, K: int, src_A: ptr float32,
                    rowStrideA, colStrideA: int) =
  check laser_b200_gemm_prepackA_f32_dev(dst_packedA, M, N, K, src_A, rowStrideA, colStrideA, nil)
proc gemm_packed*(M, N, K: int, alpha: float32, packedA, packedB: pointer, beta: float32,
                  C: ptr float32, rowStrideC, colStrideC: int) =
  ## gemm_prepacked.nim:275-292
  check laser_b200_gemm_packed_f32_dev(M, N, K, alpha, packedA, packedB, beta, C, rowStrideC, colStrideC, nil)

proc matmul*(a, b: CudaTensor[float32], c: var CudaTensor[float32],
             alpha = 1'f32, beta = 0'f32, path = pathAuto) =
  ## C <- alpha*A*B + beta*C on device tensors of any strides, as gemm_prepacked.nim:306-307
  ## does with `cast[ptr T](t.unsafe_raw_data)`.
  doAssert a.rank == 2 and b.rank == 2 and c.rank == 2
  check laser_b200_gemm_strided_f32_dev(
    a.shape.data[0], b.shape.data[1], a.shape.data[1], alpha,
    a.unsafe_raw_data, a.strides.data[0], a.strides.data[1],
    b.unsafe_raw_data, b.strides.data[0], b.strides.data[1],
    beta, c.unsafe_raw_data, c.strides.data[0], c.strides.data[1], path.cint, nil)

# ---- the steps either side of the GEMM: transposes (laser/primitives/swapaxes.nim:16-112) and
# ---- im2col convolution (benchmarks/convolution/conv2d_common.nim:6-45, conv2d_im2col.nim:8-166)
{.push importc, cdecl, dynlib: laserB200Lib.}
proc laser_b200_transpose2D_copy*(dst, src: pointer, NR, NC: int64, elemSize: cint): cint
proc laser_b200_transpose2D_batched*(dst, src: pointer, N, NR, NC: int64, elemSize: cint): cint
proc laser_b200_nchw2nhwc*(dst, src: pointer, N, C, H, W: int64, elemSize: cint): cint
proc laser_b200_nhwc2nchw*(dst, src: pointer, N, C, H, W: int64, elemSize: cint): cint
proc laser_b200_conv2d_out_shape*(ishape, kshape: ptr array[4, int64], padding, strides: ptr array[2, int64],
                                  oshape: ptr array[4, int64]): cint
proc laser_b200_conv2d_im2col_f32*(output, input: ptr float32, ishape: ptr array[4, int64], kernel: ptr float32,
                                   kshape: ptr array[4, int64], padding, strides: ptr array[2, int64]): cint
proc laser_b200_conv2d_direct_f32*(output, input: ptr float32, ishape: ptr array[4, int64], kernel: ptr float32,
                                   kshape: ptr array[4, int64], padding, strides: ptr array[2, int64]): cint
proc laser_b200_conv2d_direct_f32_dev*(output, input: ptr float32, ishape: ptr array[4, int64], kernel: ptr float32,
                                       kshape: ptr array[4, int64], padding, strides: ptr array[2, int64],
                                       epi: pointer, stream: pointer): cint
{.pop.}

proc transpose2D_copy*[T](dst, src: ptr (T or UncheckedArray[T]), NR, NC: Natural) =
  ## swapaxes.nim:16-54 (host pointers, synchronous)
  check laser_b200_transpose2D_copy(dst, src, NR, NC, sizeof(T).cint)
proc transpose2D_batched*[T](dst, src: ptr (T or UncheckedArray[T]), N, NR, NC: Natural) =
  ## swapaxes.nim:56-81
  check laser_b200_transpose2D_batched(dst, src, N, NR, NC, sizeof(T).cint)
proc nchw2nhwc*[T](dst_hwnc, src_nchw: ptr (T or UncheckedArray[T]), N, C, H, W: Natural) =
  check laser_b200_nchw2nhwc(dst_hwnc, src_nchw, N, C, H, W, sizeof(T).cint)
proc nhwc2nchw*[T](dst_nchw, src_nhwc: ptr (T or UncheckedArray[T]), N, C, H, W: Natural) =
  check laser_b200_nhwc2nchw(dst_nchw, src_nhwc, N, C, H, W, sizeof(T).cint)

type
  TensorShape* = tuple[n, c, h, w: int]
  KernelShape* = tuple[c_out, c_in, kH, kW: int]
  Padding* = tuple[h, w: int]
  Strides* = tuple[h, w: int]

proc conv2d_im2col*(output: ptr float32, oshape: TensorShape, input: ptr float32, ishape: TensorShape,
                    kernel: ptr float32, kshape: KernelShape, padding: Padding, strides: Strides) =
  ## conv2d_im2col.nim:95-166 without the caller-provided workspace (owned by the library)
  var
    ish = [ishape.n.int64, ishape.c.int64, ishape.h.int64, ishape.w.int64]
    ksh = [kshape.c_out.int64, kshape.c_in.int64, kshape.kH.int64, kshape.kW.int64]
    pad = [padding.h.int64, padding.w.int64]
    st = [strides.h.int64, strides.w.int64]
  check laser_b200_conv2d_im2col_f32(output, input, ish.addr, kernel, ksh.addr, pad.addr, st.addr)

proc conv2d_direct*(output: ptr float32, oshape: TensorShape, input: ptr float32, ishape: TensorShape,
                    kernel: ptr float32, kshape: KernelShape, padding: Padding, strides: Strides) =
  ## conv2d_direct_convolution.nim:8-76 (host pointers, synchronous): no workspace, one kernel launch; `output` is
  ## overwritten (the reference adds into a zeroed one) with the values conv2d_im2col gives on the exact path
  var
    ish = [ishape.n.int64, ishape.c.int64, ishape.h.int64, ishape.w.int64]
    ksh = [kshape.c_out.int64, kshape.c_in.int64, kshape.kH.int64, kshape.kW.int64]
    pad = [padding.h.int64, padding.w.int64]
    st = [strides.h.int64, strides.w.int64]
  check laser_b200_conv2d_direct_f32(output, input, ish.addr, kernel, ksh.addr, pad.addr, st.addr)
