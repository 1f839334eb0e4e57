// gemm_simt.cuh -- exact CUDA-core strided GEMM (fp32 FFMA; also f64 / i32 / i64).
//
// The non-tensor-core path: any strides, any alignment, any size.  For float
// types every C[i,j] is produced by the SAME sequence of operations as the
// reference CPU path, so results are bit-identical to it (and to oracle/):
//   - k-sequential FMA chain from 0 inside blocks of kc = min(2048/sizeof(T), K)
//       (gemm_tiling.nim:309-310, gemm_ukernel_generator.nim:196-250)
//   - after every kc block the reference epilogue runs on C itself, with
//       beta' = beta on the first block and 1 afterwards   (gemm.nim:150-158,
//       gemm_ukernel_generic.nim:53-76): beta'==0 -> C not read.
// Integer types wrap (the reference uses mullo + add).
//
// Tiling: (16*TM) x (16*TN) x BK block tile, 256 threads, TM x TN outputs per thread
// in two strided halves so that shared-memory reads are 16-byte broadcasts and the
// C accesses of a warp are contiguous along N.  Global loads of the next k-tile are
// issued into registers before the FMAs of the current one (software pipelining);
// the thread -> element mapping of the loads follows whichever stride of the operand
// is smaller so that HBM accesses coalesce for row-major, transposed and sliced views.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "ptx.cuh"
#include "simt_epilogue.cuh"

namespace lb200 {

template <typename T> struct SimtOps;
template <> struct SimtOps<float> {
  static __device__ __forceinline__ float fma(float a, float b, float c) { return __fmaf_rn(a, b, c); }
  static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
  static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
};
template <> struct SimtOps<double> {
  static __device__ __forceinline__ double fma(double a, double b, double c) { return __fma_rn(a, b, c); }
  static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
  static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
};
template <> struct SimtOps<int32_t> {
  static __device__ __forceinline__ int32_t fma(int32_t a, int32_t b, int32_t c) {
    return static_cast<int32_t>(static_cast<uint32_t>(a) * static_cast<uint32_t>(b) + static_cast<uint32_t>(c));
  }
  static __device__ __forceinline__ int32_t mul(int32_t a, int32_t b) {
    return static_cast<int32_t>(static_cast<uint32_t>(a) * static_cast<uint32_t>(b));
  }
  static __device__ __forceinline__ int32_t add(int32_t a, int32_t b) {
    return static_cast<int32_t>(static_cast<uint32_t>(a) + static_cast<uint32_t>(b));
  }
};
template <> struct SimtOps<int64_t> {
  static __device__ __forceinline__ int64_t fma(int64_t a, int64_t b, int64_t c) {
    return static_cast<int64_t>(static_cast<uint64_t>(a) * static_cast<uint64_t>(b) + static_cast<uint64_t>(c));
  }
  static __device__ __forceinline__ int64_t mul(int64_t a, int64_t b) {
    return static_cast<int64_t>(static_cast<uint64_t>(a) * static_cast<uint64_t>(b));
  }
  static __device__ __forceinline__ int64_t add(int64_t a, int64_t b) {
    return static_cast<int64_t>(static_cast<uint64_t>(a) + static_cast<uint64_t>(b));
  }
};

template <typename T>
struct SimtParams {
  int64_t M, N, K;
  T alpha, beta;
  const T *A; int64_t rsA, csA;
  const T *B; int64_t rsB, csB;
  T *C; int64_t rsC, csC;
  int a_along_m;  // 1: consecutive loader threads walk m (|rsA| < |csA|), 0: walk k
  int b_along_k;  // 1: consecutive loader threads walk k (|rsB| < |csB|), 0: walk n
  int num_m_blocks, num_n_blocks;
  // fused epilogue (float only), applied after the LAST kc block: v -> act(v + bias)
  const float *bias = nullptr;
  int bias_per_row = 0;
  int act = 0;
  // batch of independent problems in one launch: problem b reads A + b*bsA, B + b*bsB and
  // writes C + b*bsC (a stride of 0 shares the operand; outputs must not overlap)
  int64_t batch = 1, bsA = 0, bsB = 0, bsC = 0;
};

// host side: everything but the fused epilogue; returns the number of output tiles
template <typename T, int TM, int TN>
inline int64_t simt_plan(SimtParams<T> &p, int64_t M, int64_t N, int64_t K, T alpha, const T *A, int64_t rsA,
                         int64_t csA, const T *B, int64_t rsB, int64_t csB, T beta, T *C, int64_t rsC,
                         int64_t csC) {
  p.M = M; p.N = N; p.K = K; p.alpha = alpha; p.beta = beta;
  p.A = A; p.rsA = rsA; p.csA = csA;
  p.B = B; p.rsB = rsB; p.csB = csB;
  p.C = C; p.rsC = rsC; p.csC = csC;
  p.a_along_m = ((rsA < 0 ? -rsA : rsA) < (csA < 0 ? -csA : csA)) ? 1 : 0;
  p.b_along_k = ((rsB < 0 ? -rsB : rsB) < (csB < 0 ? -csB : csB)) ? 1 : 0;
  constexpr int BM = 16 * TM, BN = 16 * TN;
  const int64_t mblocks = (M + BM - 1) / BM, nblocks = (N + BN - 1) / BN;
  p.num_m_blocks = static_cast<int>(mblocks);
  p.num_n_blocks = static_cast<int>(nblocks);
  return mblocks * nblocks;
}

#ifndef LB200_SIMT_MINB
#define LB200_SIMT_MINB 1
#endif
#define LB200_SIMT_KERNEL_NAME gemm_simt_kernel
#define LB200_SIMT_BATCHED 0
#include "gemm_simt_kernel.inc"
#undef LB200_SIMT_KERNEL_NAME
#undef LB200_SIMT_BATCHED
#define LB200_SIMT_KERNEL_NAME gemm_simt_batched_kernel
#define LB200_SIMT_BATCHED 1
#include "gemm_simt_kernel.inc"
#undef LB200_SIMT_KERNEL_NAME
#undef LB200_SIMT_BATCHED

// ---------------------------------------------------------------------------
// Skinny GEMM: N <= 4 (matrix x few vectors).  One warp per output row: lanes stride
// over K with coalesced loads of A's row, partial dot products are combined with
// warp shuffles.  Not bit-identical to the reference's k-sequential chain (the
// reduction tree differs) - used only when the caller asks for PATH_AUTO on a
// skinny problem; PATH_SIMT always takes the exact kernel above.
// ---------------------------------------------------------------------------
template <int NV, bool VEC>
__global__ void __launch_bounds__(256)
gemv_warp_kernel(int64_t M, int64_t K, float alpha, const float *__restrict__ A, int64_t rsA,
                 int64_t csA, const float *__restrict__ B, int64_t rsB, int64_t csB, float beta,
                 float *__restrict__ C, int64_t rsC, int64_t csC) {
  const int lane = threadIdx.x & 31;
  const int64_t warps_total = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  for (int64_t row = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; row < M;
       row += warps_total) {
    float acc[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) acc[j] = 0.0f;
    const float *a = A + row * rsA;
    if constexpr (VEC) {
      // A rows contiguous and 16-byte aligned, K % 4 == 0: each lane streams float4s, four
      // independent 16-byte loads in flight per lane (the kernel is pure HBM streaming of A)
      const float4 *a4 = reinterpret_cast<const float4 *>(a);
      const int64_t K4 = K >> 2;
#pragma unroll 4
      for (int64_t q = lane; q < K4; q += 32) {
        const float4 av = __ldg(a4 + q);
        const int64_t k = q << 2;
#pragma unroll
        for (int j = 0; j < NV; ++j) {
          acc[j] = fmaf(av.x, __ldg(B + (k + 0) * rsB + j * csB), acc[j]);
          acc[j] = fmaf(av.y, __ldg(B + (k + 1) * rsB + j * csB), acc[j]);
          acc[j] = fmaf(av.z, __ldg(B + (k + 2) * rsB + j * csB), acc[j]);
          acc[j] = fmaf(av.w, __ldg(B + (k + 3) * rsB + j * csB), acc[j]);
        }
      }
    } else {
#pragma unroll 4
      for (int64_t k = lane; k < K; k += 32) {
        const float av = a[k * csA];
#pragma unroll
        for (int j = 0; j < NV; ++j) acc[j] = fmaf(av, B[k * rsB + j * csB], acc[j]);
      }
    }
#pragma unroll
    for (int j = 0; j < NV; ++j) {
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], off);
    }
    if (lane == 0) {
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        float *c = C + row * rsC + j * csC;
        const float v = alpha * acc[j];
        *c = (beta == 0.0f) ? v : fmaf(beta, *c, v);
      }
    }
  }
}

// Same contract, B (K x NV) staged once per CTA in shared memory, transposed to Bs[j][k] so
// that each 16-byte load of A is matched by NV 16-byte shared loads instead of 4*NV global
// ones.  Needs A rows contiguous + 16-byte aligned, K % 4 == 0 and NV*K*4 bytes of smem.
template <int NV>
__global__ void __launch_bounds__(256)
gemv_warp_smem_kernel(int64_t M, int64_t K, float alpha, const float *__restrict__ A, int64_t rsA,
                      const float *__restrict__ B, int64_t rsB, int64_t csB, float beta,
                      float *__restrict__ C, int64_t rsC, int64_t csC) {
  LB200_DYN_SMEM(float4, gemv_smem4);
  float *Bs = reinterpret_cast<float *>(gemv_smem4);
  for (int64_t i = threadIdx.x; i < K * NV; i += blockDim.x) {
    const int64_t k = i / NV;
    const int j = static_cast<int>(i - k * NV);
    Bs[j * K + k] = B[k * rsB + j * csB];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t warps_total = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int64_t K4 = K >> 2;
  for (int64_t row = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; row < M;
       row += warps_total) {
    float acc[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) acc[j] = 0.0f;
    const float4 *a4 = reinterpret_cast<const float4 *>(A + row * rsA);
#pragma unroll 8
    for (int64_t q = lane; q < K4; q += 32) {
      const float4 av = __ldg(a4 + q);
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        const float4 bv = *reinterpret_cast<const float4 *>(Bs + j * K + (q << 2));
        acc[j] = fmaf(av.x, bv.x, acc[j]);
        acc[j] = fmaf(av.y, bv.y, acc[j]);
        acc[j] = fmaf(av.z, bv.z, acc[j]);
        acc[j] = fmaf(av.w, bv.w, acc[j]);
      }
    }
#pragma unroll
    for (int j = 0; j < NV; ++j) {
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], off);
    }
    if (lane == 0) {
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        float *c = C + row * rsC + j * csC;
        const float v = alpha * acc[j];
        *c = (beta == 0.0f) ? v : fmaf(beta, *c, v);
      }
    }
  }
}

// ---------------------------------------------------------------------------
// Few output ROWS, very wide N: the GEMM of the im2col convolution (conv2d_im2col.nim:150-166: M = filters = 20,
// K = C * kH * kW = 27, N = outH * outW = 49284 per image).  A 128 x 128 tile of the general kernel would compute 84 %
// padding; here a thread owns 4 consecutive columns of ALL rows: per k one 16-byte load of B (coalesced along n), MT / 4
// 16-byte broadcast reads of A's k-th column from shared memory and 4 * MT FMAs -- the kernel streams B and C once.
// Exact: every C[i,j] is the reference's k-sequential FMA chain inside kc = 512 blocks with the reference epilogue per
// block (same statements as gemm_simt_kernel), so results are bit-identical to the general kernel's.  Batched like it.
// MT: rows held in registers (M <= MT, a multiple of 4).
// ---------------------------------------------------------------------------
constexpr int SKINNY_KCHUNK = 64;   // k-columns of A staged in shared memory at a time
// NC: columns per thread (4 for MT <= 16, 2 above: MT * NC running sums per thread must leave room for two CTAs per SM)
template <int MT, int NC>
__global__ void __launch_bounds__(256, 2)
gemm_skinny_m_kernel(const SimtParams<float> p) {
  static_assert(MT % 4 == 0 && MT <= 32 && (NC == 2 || NC == 4), "rows in registers");
  constexpr int64_t KC = 2048 / 4;   // gemm_tiling.nim:310
  constexpr int COLS = 256 * NC;     // columns per CTA and iteration
  __shared__ float4 As4[SKINNY_KCHUNK][MT / 4];   // As[k][m]: the m of one k are contiguous (16-byte broadcast reads)
  float *As = reinterpret_cast<float *>(As4);
  const int tid = threadIdx.x;
  const int64_t nblocks = (p.N + COLS - 1) / COLS;
  const int64_t total = nblocks * p.batch;
  for (int64_t t = blockIdx.x; t < total; t += gridDim.x) {
    const int64_t bi = t / nblocks;
    const int64_t n0 = (t - bi * nblocks) * COLS + NC * tid;
    const float *Ab = p.A + bi * p.bsA;
    const float *Bb = p.B + bi * p.bsB;
    float *Cb = p.C + bi * p.bsC;
    const bool vec_b = p.csB == 1 && n0 + NC <= p.N &&
                       ((reinterpret_cast<uintptr_t>(Bb + n0) | (static_cast<uint64_t>(p.rsB) * 4)) & (4 * NC - 1)) == 0;
    for (int64_t pc = 0; pc < p.K; pc += KC) {  // reference loop 2 (gemm.nim:150)
      const int64_t kend = (pc + KC < p.K) ? pc + KC : p.K;
      float acc[MT][NC];
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NC; ++j) acc[i][j] = 0.0f;
      for (int64_t k0 = pc; k0 < kend; k0 += SKINNY_KCHUNK) {
        const int kn = static_cast<int>(kend - k0 < SKINNY_KCHUNK ? kend - k0 : SKINNY_KCHUNK);
        __syncthreads();   // the previous chunk of A is consumed
        for (int i = tid; i < SKINNY_KCHUNK * MT; i += 256) {
          const int k = i / MT, m = i - k * MT;
          As[i] = (m < p.M && k < kn) ? Ab[m * p.rsA + (k0 + k) * p.csA] : 0.0f;
        }
        __syncthreads();
        if (n0 < p.N) {
          // (k-steps in flight: as many as the register budget of two CTAs per SM allows next to the MT * NC sums)
#pragma unroll(MT * NC > 48 ? 2 : 4)
          for (int k = 0; k < kn; ++k) {
            float b[NC];
            const float *brow = Bb + (k0 + k) * p.rsB + n0 * p.csB;
            if (vec_b) {
              if constexpr (NC == 4) {
                const float4 v = *reinterpret_cast<const float4 *>(brow);
                b[0] = v.x; b[1] = v.y; b[2] = v.z; b[3] = v.w;
              } else {
                const float2 v = *reinterpret_cast<const float2 *>(brow);
                b[0] = v.x; b[1] = v.y;
              }
            } else {
#pragma unroll
              for (int j = 0; j < NC; ++j) b[j] = (n0 + j < p.N) ? brow[j * p.csB] : 0.0f;
            }
#pragma unroll
            for (int i4 = 0; i4 < MT / 4; ++i4) {
              const float4 a = As4[k][i4];
              const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
              for (int e = 0; e < 4; ++e)
#pragma unroll
                for (int j = 0; j < NC; ++j) acc[4 * i4 + e][j] = __fmaf_rn(av[e], b[j], acc[4 * i4 + e][j]);
            }
          }
        }
      }
      // reference epilogue for this kc block (gemm_ukernel_generic.nim:53-76)
      const float beta1 = (pc == 0) ? p.beta : 1.0f;
      const bool has_epi = kend == p.K && (p.bias != nullptr || p.act != 0);
      if (n0 < p.N) {
#pragma unroll
        for (int i = 0; i < MT; ++i) {
          if (i >= p.M) break;
          float *crow = Cb + i * p.rsC + n0 * p.csC;
          float v[NC];
#pragma unroll
          for (int j = 0; j < NC; ++j) {
            if (n0 + j >= p.N) { v[j] = 0.0f; continue; }
            float x;
            if (beta1 == 0.0f) x = 0.0f;
            else if (beta1 != 1.0f) x = __fmul_rn(crow[j * p.csC], beta1);
            else x = crow[j * p.csC];
            if (p.alpha == 1.0f) x = __fadd_rn(x, acc[i][j]);
            else x = __fadd_rn(x, __fmul_rn(p.alpha, acc[i][j]));
            if (has_epi) x = simt_bias_act(x, p.bias, p.bias_per_row, p.act, i, n0 + j);
            v[j] = x;
          }
          if (p.csC == 1 && n0 + NC <= p.N && (reinterpret_cast<uintptr_t>(crow) & (4 * NC - 1)) == 0) {
            if constexpr (NC == 4) *reinterpret_cast<float4 *>(crow) = make_float4(v[0], v[1], v[2], v[3]);
            else *reinterpret_cast<float2 *>(crow) = make_float2(v[0], v[1]);
          } else {
#pragma unroll
            for (int j = 0; j < NC; ++j)
              if (n0 + j < p.N) crow[j * p.csC] = v[j];
          }
        }
      }
    }
  }
}

// The same product with B streamed through shared memory by cp.async: thread t copies exactly the 16 bytes (its 4 columns) of
// each k-row it will consume into a private FIFO of SKA_STAGES x SKA_K rows -- no registers hold data in flight and no barrier
// guards it, so ~100 KB per SM are on their way from HBM at any time (the register-only kernel above keeps 16 KB in flight and
// runs at 1.1 TB/s).  Needs unit column stride and 16-byte aligned rows of B (the host checks); same FMA chains, same results.
constexpr int SKA_K = 8, SKA_STAGES = 4;
template <int MT>
__global__ void __launch_bounds__(256, 1)
gemm_skinny_m_async_kernel(const SimtParams<float> p) {
  static_assert(MT % 4 == 0 && MT <= 32, "rows in registers");
  static_assert(SKINNY_KCHUNK % SKA_K == 0, "whole FIFO stages per chunk of A");
  constexpr int64_t KC = 2048 / 4;   // gemm_tiling.nim:310 (a multiple of SKA_K: stages never straddle a kc block)
  LB200_DYN_SMEM(float4, ska_smem);  // [SKA_STAGES][SKA_K][256] float4 of B, then As4[SKINNY_KCHUNK][MT / 4]
  float4 *Bf = ska_smem;
  float4 *As4 = ska_smem + SKA_STAGES * SKA_K * 256;
  float *As = reinterpret_cast<float *>(As4);
  const int tid = threadIdx.x;
  const int64_t nblocks = (p.N + 1023) / 1024;
  const int64_t total = nblocks * p.batch;
  // The CTA's tiles (1024 columns of one problem each) form ONE stream of FIFO stages, SKA_K k-rows each: the copies of the
  // next tile are in flight while this one is multiplied and stored (with K = 27 a tile is only four stages long)
  const int64_t st_per_tile = (p.K + SKA_K - 1) / SKA_K;
  const int64_t my_tiles = blockIdx.x < total ? (total - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const int64_t total_stages = my_tiles * st_per_tile;
  auto issue = [&](int64_t g) {   // one commit group per call (possibly empty)
    if (g < total_stages) {
      const int64_t it = g / st_per_tile, s = g - it * st_per_tile;
      const int64_t t = blockIdx.x + it * gridDim.x;
      const int64_t bi = t / nblocks;
      const int64_t n0 = (t - bi * nblocks) * 1024 + 4 * tid;
      if (n0 < p.N) {
        const uint32_t src_bytes = static_cast<uint32_t>((p.N - n0 < 4 ? p.N - n0 : 4) * 4);   // ragged right edge: zero fill
        const float *Bb = p.B + bi * p.bsB + n0;
        float4 *dst = Bf + ((g % SKA_STAGES) * SKA_K) * 256 + tid;
#pragma unroll
        for (int r = 0; r < SKA_K; ++r) {
          const int64_t k = s * SKA_K + r;
          if (k < p.K) ptx::cp_async_16(dst + r * 256, Bb + k * p.rsB, src_bytes);
        }
      }
    }
    ptx::cp_async_commit();
  };
#pragma unroll
  for (int s = 0; s < SKA_STAGES - 1; ++s) issue(s);
  int64_t g = 0;   // stage being consumed
  for (int64_t t = blockIdx.x; t < total; t += gridDim.x) {
    const int64_t bi = t / nblocks;
    const int64_t n0 = (t - bi * nblocks) * 1024 + 4 * tid;
    const float *Ab = p.A + bi * p.bsA;
    float *Cb = p.C + bi * p.bsC;
    const bool live = n0 < p.N;
    for (int64_t pc = 0; pc < p.K; pc += KC) {  // reference loop 2 (gemm.nim:150)
      const int64_t kend = (pc + KC < p.K) ? pc + KC : p.K;
      float acc[MT][4];
#pragma unroll
      for (int i = 0; i < MT; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.0f;
      for (int64_t k0 = pc; k0 < kend; k0 += SKINNY_KCHUNK) {
        const int kn = static_cast<int>(kend - k0 < SKINNY_KCHUNK ? kend - k0 : SKINNY_KCHUNK);
        __syncthreads();   // the previous chunk of A is consumed
        for (int i = tid; i < SKINNY_KCHUNK * MT; i += 256) {
          const int k = i / MT, m = i - k * MT;
          As[i] = (m < p.M && k < kn) ? Ab[m * p.rsA + (k0 + k) * p.csA] : 0.0f;
        }
        __syncthreads();
#pragma unroll 1
        for (int kk = 0; kk < kn; kk += SKA_K, ++g) {
          ptx::cp_async_wait<SKA_STAGES - 2>();   // this thread's copies of stage g have landed (nobody else reads them)
          const float4 *bs = Bf + ((g % SKA_STAGES) * SKA_K) * 256 + tid;
          const int kr = kn - kk < SKA_K ? kn - kk : SKA_K;
          if (live) {
#pragma unroll
            for (int r = 0; r < SKA_K; ++r) {
              if (r < kr) {
                const float4 bv = bs[r * 256];
                const float b[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
                for (int i4 = 0; i4 < MT / 4; ++i4) {
                  const float4 a = As4[(kk + r) * (MT / 4) + i4];
                  const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
                  for (int e = 0; e < 4; ++e)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[4 * i4 + e][j] = __fmaf_rn(av[e], b[j], acc[4 * i4 + e][j]);
                }
              }
            }
          }
          issue(g + SKA_STAGES - 1);   // refill the slot consumed one iteration ago (it may belong to the next tile)
        }
      }
      // reference epilogue for this kc block (gemm_ukernel_generic.nim:53-76)
      const float beta1 = (pc == 0) ? p.beta : 1.0f;
      const bool has_epi = kend == p.K && (p.bias != nullptr || p.act != 0);
      // the common case of the convolution (alpha = 1, beta = 0, nothing fused, whole float4 inside C): 0 + sum, one vector
      // store per row -- a few hundred instructions instead of the general store loop below (instruction-cache footprint)
      const bool plain = beta1 == 0.0f && p.alpha == 1.0f && !has_epi && p.csC == 1 && n0 + 4 <= p.N &&
                         ((reinterpret_cast<uintptr_t>(Cb + n0) | (static_cast<uint64_t>(p.rsC) * 4)) & 15) == 0;
      if (live && plain) {
#pragma unroll
        for (int i = 0; i < MT; ++i) {
          if (i < p.M)
            *reinterpret_cast<float4 *>(Cb + i * p.rsC + n0) =
                make_float4(__fadd_rn(0.0f, acc[i][0]), __fadd_rn(0.0f, acc[i][1]), __fadd_rn(0.0f, acc[i][2]), __fadd_rn(0.0f, acc[i][3]));
        }
      } else if (live) {
#pragma unroll
        for (int i = 0; i < MT; ++i) {
          if (i >= p.M) break;
          float *crow = Cb + i * p.rsC + n0 * p.csC;
          float v[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (n0 + j >= p.N) { v[j] = 0.0f; continue; }
            float x;
            if (beta1 == 0.0f) x = 0.0f;
            else if (beta1 != 1.0f) x = __fmul_rn(crow[j * p.csC], beta1);
            else x = crow[j * p.csC];
            if (p.alpha == 1.0f) x = __fadd_rn(x, acc[i][j]);
            else x = __fadd_rn(x, __fmul_rn(p.alpha, acc[i][j]));
            if (has_epi) x = simt_bias_act(x, p.bias, p.bias_per_row, p.act, i, n0 + j);
            v[j] = x;
          }
          if (p.csC == 1 && n0 + 4 <= p.N && (reinterpret_cast<uintptr_t>(crow) & 15) == 0) {
            *reinterpret_cast<float4 *>(crow) = make_float4(v[0], v[1], v[2], v[3]);
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (n0 + j < p.N) crow[j * p.csC] = v[j];
          }
        }
      }
    }
  }
  ptx::cp_async_wait<0>();
}
template <int MT> constexpr size_t ska_smem_bytes() { return (static_cast<size_t>(SKA_STAGES) * SKA_K * 256 + SKINNY_KCHUNK * (MT / 4)) * sizeof(float4); }

}  // namespace lb200
