// simt_epilogue.cuh -- device pieces shared by the exact CUDA-core GEMM (gemm_simt.cuh) and the direct
// convolution (layers.cuh): the bias + activation of the fused epilogue, and the spelling of dynamic shared
// memory.  One definition, so that both produce the same bits for the same value.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace lb200 {

// bias + activation of the fused epilogue, out of line: inlined into the unrolled MT x NC store loops the tanhf / expf bodies
// made the kernels several times larger than the instruction cache (ncu: 58 % of the stall samples "no instruction").
// A host compiler (tests/emu runs these headers on host threads) gets a plain inline function.
#if defined(__CUDACC__) && !defined(LB200_HOST_EMULATION)
static __device__ __noinline__
#else
inline
#endif
float simt_bias_act(float x, const float *bias, int bias_per_row, int act, int64_t row, int64_t col) {
  if (bias) x += bias_per_row ? bias[row] : bias[col];
  if (act == 1) x = fmaxf(x, 0.0f);
  else if (act == 2) x = tanhf(x);
  else if (act == 3) x = 1.0f / (1.0f + expf(-x));
  return x;
}

}  // namespace lb200

// dynamic shared memory (tests/emu runs these headers on host threads, where it is a plain buffer)
#ifndef LB200_DYN_SMEM
#ifdef LB200_HOST_EMULATION
#define LB200_DYN_SMEM(T, name) T *name = reinterpret_cast<T *>(emu::dyn_smem_ptr())
#else
#define LB200_DYN_SMEM(T, name) extern __shared__ T name[]
#endif
#endif
