// laser_b200.hpp -- header-only C++ host mirror of the reference's interface for the hot path,
// on top of the C ABI (laser_b200.h).  The reference is Nim, which compiles to C/C++; no Nim
// toolchain exists in the build image, so this is the compiled-language host side: same names,
// argument order and meaning as the Nim procs, errors surfaced as exceptions (the Nim shim in
// nim/laser_b200.nim does the same with LaserB200Error).
//
//   laser::gemm_strided<T>(M, N, K, alpha, A, rowStrideA, colStrideA, B, rowStrideB, colStrideB,
//                          beta, C, rowStrideC, colStrideC)
//        == proc gemm_strided*[T: SomeNumber](...)   laser/primitives/matrix_multiplication/gemm.nim:184-193
//   laser::CudaTensor<T>  (shape / strides / offset / storage; rank, size, is_C_contiguous,
//                          unsafe_raw_data)           laser/tensor/datatypes.nim:12-88
//   laser::newTensor<T>, toTensor<T>, toHost          laser/tensor/initialization.nim:156-202
//   laser::gemm_prepackA/B_mem_required, gemm_prepackA/B, gemm_packed
//                                                     .../gemm_prepacked.nim:63-292
//   laser::transpose2D_copy, transpose2D_batched, nchw2nhwc, nhwc2nchw
//                                                     laser/primitives/swapaxes.nim:16-112
//   laser::TensorShape/KernelShape/Padding/Strides, conv2d_out_shape, im2col_workspace_size,
//   conv2d_im2col                                     benchmarks/convolution/conv2d_common.nim:6-45,
//                                                     conv2d_im2col.nim:8-166
//   conv2d_direct                                     conv2d_direct_convolution.nim:8-76
#pragma once

#include <cstdint>
#include <initializer_list>
#include <memory>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <vector>

#include "laser_b200.h"

namespace laser {

struct LaserB200Error : std::runtime_error {
  int code;
  LaserB200Error(int c, const char *msg) : std::runtime_error(std::string("laser_b200: ") + msg), code(c) {}
};
inline void check(int rc) {
  if (rc != LASER_B200_OK) throw LaserB200Error(rc, laser_b200_last_error());
}

// ---- gemm_strided: host pointers, synchronous (gemm.nim:184-193) -------------------------
inline void gemm_strided(int64_t M, int64_t N, int64_t K, float alpha, const float *A, int64_t rowStrideA,
                         int64_t colStrideA, const float *B, int64_t rowStrideB, int64_t colStrideB, float beta,
                         float *C, int64_t rowStrideC, int64_t colStrideC) {
  check(laser_b200_gemm_strided_f32(M, N, K, alpha, A, rowStrideA, colStrideA, B, rowStrideB, colStrideB, beta, C,
                                    rowStrideC, colStrideC));
}
inline void gemm_strided(int64_t M, int64_t N, int64_t K, double alpha, const double *A, int64_t rowStrideA,
                         int64_t colStrideA, const double *B, int64_t rowStrideB, int64_t colStrideB, double beta,
                         double *C, int64_t rowStrideC, int64_t colStrideC) {
  check(laser_b200_gemm_strided_f64(M, N, K, alpha, A, rowStrideA, colStrideA, B, rowStrideB, colStrideB, beta, C,
                                    rowStrideC, colStrideC));
}
inline void gemm_strided(int64_t M, int64_t N, int64_t K, int32_t alpha, const int32_t *A, int64_t rowStrideA,
                         int64_t colStrideA, const int32_t *B, int64_t rowStrideB, int64_t colStrideB, int32_t beta,
                         int32_t *C, int64_t rowStrideC, int64_t colStrideC) {
  check(laser_b200_gemm_strided_i32(M, N, K, alpha, A, rowStrideA, colStrideA, B, rowStrideB, colStrideB, beta, C,
                                    rowStrideC, colStrideC));
}
inline void gemm_strided(int64_t M, int64_t N, int64_t K, int64_t alpha, const int64_t *A, int64_t rowStrideA,
                         int64_t colStrideA, const int64_t *B, int64_t rowStrideB, int64_t colStrideB, int64_t beta,
                         int64_t *C, int64_t rowStrideC, int64_t colStrideC) {
  check(laser_b200_gemm_strided_i64(M, N, K, alpha, A, rowStrideA, colStrideA, B, rowStrideB, colStrideB, beta, C,
                                    rowStrideC, colStrideC));
}

// ---- device tensor honouring the tensor contract (datatypes.nim:12-88) -------------------
constexpr int LASER_MAXRANK = LASER_B200_MAXRANK;  // laser/dynamic_stack_arrays.nim:6

template <typename T> struct dtype_code;
template <> struct dtype_code<float> { static constexpr int value = 0; };
template <> struct dtype_code<double> { static constexpr int value = 1; };
template <> struct dtype_code<int32_t> { static constexpr int value = 2; };
template <> struct dtype_code<int64_t> { static constexpr int value = 3; };

template <typename T>
struct CudaStorage {  // CpuStorage analogue: raw_buffer + ownership (datatypes.nim:24-30)
  T *raw_buffer = nullptr;
  bool memowner = false;
  explicit CudaStorage(size_t n) {
    void *p = nullptr;
    check(laser_b200_malloc(&p, n * sizeof(T)));
    check(laser_b200_memset_zero(p, n * sizeof(T)));
    raw_buffer = static_cast<T *>(p);
    memowner = true;
  }
  ~CudaStorage() {
    if (memowner && raw_buffer) laser_b200_free(raw_buffer);
  }
  CudaStorage(const CudaStorage &) = delete;
  CudaStorage &operator=(const CudaStorage &) = delete;
};

template <typename T>
struct CudaTensor {
  std::vector<int64_t> shape, strides;  // strides in elements
  int64_t offset = 0;
  std::shared_ptr<CudaStorage<T>> storage;  // reference semantics, like the `ref object` it mirrors

  int rank() const { return static_cast<int>(shape.size()); }
  int64_t size() const {
    int64_t n = 1;
    for (auto s : shape) n *= s;
    return n;
  }
  bool is_C_contiguous() const {  // datatypes.nim:37-47
    int64_t cur = 1;
    for (int i = rank() - 1; i >= 0; --i) {
      if (shape[i] != 1 && strides[i] != cur) return false;
      cur *= shape[i];
    }
    return true;
  }
  T *unsafe_raw_data() const { return storage->raw_buffer + offset; }  // datatypes.nim:64-88
  CudaTensor transpose() const {
    CudaTensor t = *this;
    t.shape = {shape[1], shape[0]};
    t.strides = {strides[1], strides[0]};
    return t;
  }
  laser_b200_tensor_view view() const {
    laser_b200_tensor_view v{};
    v.rank = rank();
    v.dtype = dtype_code<T>::value;
    for (int i = 0; i < rank(); ++i) { v.shape[i] = shape[i]; v.strides[i] = strides[i]; }
    v.offset = offset;
    v.storage = storage->raw_buffer;
    return v;
  }
};

template <typename T>
CudaTensor<T> newTensor(std::initializer_list<int64_t> shape) {  // zero-initialised, row-major
  if (shape.size() > static_cast<size_t>(LASER_MAXRANK)) throw std::invalid_argument("rank > LASER_MAXRANK");
  CudaTensor<T> t;
  t.shape.assign(shape.begin(), shape.end());
  t.strides.assign(t.shape.size(), 1);
  int64_t acc = 1;
  for (int i = t.rank() - 1; i >= 0; --i) { t.strides[i] = acc; acc *= t.shape[i]; }
  t.storage = std::make_shared<CudaStorage<T>>(static_cast<size_t>(acc));
  return t;
}
template <typename T>
CudaTensor<T> toTensor(const T *host, std::initializer_list<int64_t> shape) {
  CudaTensor<T> t = newTensor<T>(shape);
  check(laser_b200_memcpy_h2d(t.unsafe_raw_data(), host, static_cast<size_t>(t.size()) * sizeof(T)));
  return t;
}
template <typename T>
std::vector<T> toHost(const CudaTensor<T> &t) {  // C-contiguous tensors only
  if (!t.is_C_contiguous()) throw std::invalid_argument("toHost needs a C-contiguous tensor");
  std::vector<T> out(static_cast<size_t>(t.size()));
  check(laser_b200_memcpy_d2h(out.data(), t.unsafe_raw_data(), out.size() * sizeof(T)));
  return out;
}

// C <- alpha * A*B + beta * C on rank-2 device tensors of any strides
template <typename T>
void matmul(const CudaTensor<T> &A, const CudaTensor<T> &B, CudaTensor<T> &C, double alpha = 1.0, double beta = 0.0,
            int path = LASER_B200_PATH_AUTO) {
  const laser_b200_tensor_view va = A.view(), vb = B.view();
  laser_b200_tensor_view vc = C.view();
  check(laser_b200_matmul_views(&va, &vb, &vc, alpha, beta, path, nullptr));
}

// dst <- src over a common shape, any strides (copyFrom, initialization.nim:80-112)
template <typename T>
void copyFrom(CudaTensor<T> &dst, const CudaTensor<T> &src) {
  laser_b200_tensor_view vd = dst.view();
  const laser_b200_tensor_view vs = src.view();
  check(laser_b200_copy_views(&vd, &vs, nullptr));
}
// forEach o in out, x in a, y in b, z in c: <body named by op> (foreach.nim:229-251); op = LASER_B200_FOREACH_*
template <typename T>
void forEach(int op, CudaTensor<T> &out, const CudaTensor<T> *x = nullptr, const CudaTensor<T> *y = nullptr,
             const CudaTensor<T> *z = nullptr, double alpha = 0.0) {
  static_assert(std::is_floating_point<T>::value, "forEach opcodes are float32 / float64 only");
  laser_b200_tensor_view vo = out.view(), vx{}, vy{}, vz{};
  if (x) vx = x->view();
  if (y) vy = y->view();
  if (z) vz = z->view();
  check(laser_b200_foreach_views(op, &vo, x ? &vx : nullptr, y ? &vy : nullptr, z ? &vz : nullptr, alpha, nullptr));
}

// ---- pre-packed API (gemm_prepacked.nim:63-292); device pointers --------------------------
inline size_t gemm_prepackA_mem_required(int64_t M, int64_t N, int64_t K) { return laser_b200_gemm_prepackA_mem_required_f32(M, N, K); }
inline size_t gemm_prepackB_mem_required(int64_t M, int64_t N, int64_t K) { return laser_b200_gemm_prepackB_mem_required_f32(M, N, K); }
inline void gemm_prepackA(void *dst_packedA, int64_t M, int64_t N, int64_t K, const float *src_A, int64_t rowStrideA,
                          int64_t colStrideA) {
  check(laser_b200_gemm_prepackA_f32_dev(dst_packedA, M, N, K, src_A, rowStrideA, colStrideA, nullptr));
}
inline void gemm_prepackB(void *dst_packedB, int64_t M, int64_t N, int64_t K, const float *src_B, int64_t rowStrideB,
                          int64_t colStrideB) {
  check(laser_b200_gemm_prepackB_f32_dev(dst_packedB, M, N, K, src_B, rowStrideB, colStrideB, nullptr));
}
inline void gemm_packed(int64_t M, int64_t N, int64_t K, float alpha, const void *packedA, const void *packedB, float beta,
                        float *C, int64_t rowStrideC, int64_t colStrideC) {
  check(laser_b200_gemm_packed_f32_dev(M, N, K, alpha, packedA, packedB, beta, C, rowStrideC, colStrideC, nullptr));
}

// ---- physical transposition (swapaxes.nim:16-112); host pointers, synchronous ---------------
template <typename T>
void transpose2D_copy(T *dst, const T *src, int64_t NR, int64_t NC) {
  check(laser_b200_transpose2D_copy(dst, src, NR, NC, static_cast<int>(sizeof(T))));
}
template <typename T>
void transpose2D_batched(T *dst, const T *src, int64_t N, int64_t NR, int64_t NC) {
  check(laser_b200_transpose2D_batched(dst, src, N, NR, NC, static_cast<int>(sizeof(T))));
}
template <typename T>
void nchw2nhwc(T *dst_nhwc, const T *src_nchw, int64_t N, int64_t C, int64_t H, int64_t W) {
  check(laser_b200_nchw2nhwc(dst_nhwc, src_nchw, N, C, H, W, static_cast<int>(sizeof(T))));
}
template <typename T>
void nhwc2nchw(T *dst_nchw, const T *src_nhwc, int64_t N, int64_t C, int64_t H, int64_t W) {
  check(laser_b200_nhwc2nchw(dst_nchw, src_nhwc, N, C, H, W, static_cast<int>(sizeof(T))));
}

// ---- im2col convolution (conv2d_common.nim:6-45, conv2d_im2col.nim:8-166) ---------------------
struct TensorShape { int64_t n, c, h, w; };          // batch, channels, height, width
struct KernelShape { int64_t c_out, c_in, kH, kW; };
struct Padding { int64_t h, w; };
struct Strides { int64_t h, w; };

inline TensorShape conv2d_out_shape(TensorShape input, KernelShape kernel, Padding padding, Strides strides) {
  const int64_t is[4] = {input.n, input.c, input.h, input.w}, ks[4] = {kernel.c_out, kernel.c_in, kernel.kH, kernel.kW};
  const int64_t pd[2] = {padding.h, padding.w}, st[2] = {strides.h, strides.w};
  int64_t o[4];
  check(laser_b200_conv2d_out_shape(is, ks, pd, st, o));
  return TensorShape{o[0], o[1], o[2], o[3]};
}
inline int64_t im2col_workspace_size(TensorShape ishape, KernelShape kshape, Padding padding, Strides strides) {
  const TensorShape o = conv2d_out_shape(ishape, kshape, padding, strides);
  return ishape.c * kshape.kH * kshape.kW * o.h * o.w;
}
// output / input NCHW, kernel (c_out, c_in, kH, kW); host pointers; output fully overwritten.
// The reference's caller-provided one-image workspace is owned by the library here.
inline void conv2d_im2col(float *output, TensorShape oshape, const float *input, TensorShape ishape,
                          const float *kernel, KernelShape kshape, Padding padding, Strides strides) {
  const TensorShape expect = conv2d_out_shape(ishape, kshape, padding, strides);
  if (expect.n != oshape.n || expect.c != oshape.c || expect.h != oshape.h || expect.w != oshape.w)
    throw std::invalid_argument("conv2d_im2col: oshape does not match conv2d_out_shape");
  const int64_t is[4] = {ishape.n, ishape.c, ishape.h, ishape.w}, ks[4] = {kshape.c_out, kshape.c_in, kshape.kH, kshape.kW};
  const int64_t pd[2] = {padding.h, padding.w}, st[2] = {strides.h, strides.w};
  check(laser_b200_conv2d_im2col_f32(output, input, is, kernel, ks, pd, st));
}
// conv2d_direct_convolution.nim:8-76 with the same arguments: no workspace, one kernel launch, output fully overwritten
// (the reference adds into a zeroed output), bit for bit the values of conv2d_im2col on the exact path.
inline void conv2d_direct(float *output, TensorShape oshape, const float *input, TensorShape ishape, const float *kernel,
                          KernelShape kshape, Padding padding, Strides strides) {
  const TensorShape expect = conv2d_out_shape(ishape, kshape, padding, strides);
  if (expect.n != oshape.n || expect.c != oshape.c || expect.h != oshape.h || expect.w != oshape.w)
    throw std::invalid_argument("conv2d_direct: oshape does not match conv2d_out_shape");
  const int64_t is[4] = {ishape.n, ishape.c, ishape.h, ishape.w}, ks[4] = {kshape.c_out, kshape.c_in, kshape.kH, kshape.kW};
  const int64_t pd[2] = {padding.h, padding.w}, st[2] = {strides.h, strides.w};
  check(laser_b200_conv2d_direct_f32(output, input, is, kernel, ks, pd, st));
}

}  // namespace laser
