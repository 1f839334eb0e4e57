// conv2d_direct_emu.cpp -- TEST INFRASTRUCTURE: the direct convolution kernel of laser_b200/csrc/layers.cuh
// (conv2d_direct_kernel) compiled for the host (cuda_emu.h) behind a small C interface for ctypes, launched with the
// plan the library uses (direct_conv_plan) -- either variant of the kernel, on a chosen number of blocks.
#define LB200_HOST_EMULATION 1
#include "cuda_emu.h"

#include "../../laser_b200/csrc/layers.cuh"

using namespace lb200;

extern "C" {

// geom = {C, H, W, Cout, kH, kW, pH, pW, sH, sW, outH, outW}; bias: NULL or Cout values; act 0..3.
// grid <= 0: one block per unit of work (else a grid-stride loop over `grid` blocks); stage_input = 0: the variant that
// reads the input from global memory.  Returns 1 when the staged variant ran, 0 for the other.
int emu_conv2d_direct(float *output, const float *input, const float *kernel, int64_t images, const int64_t geom[12],
                      const float *bias, int act, int grid, int stage_input) {
  DirectConvParams p;
  const bool staged = direct_conv_plan(geom, images, &p, stage_input != 0);
  p.bias = bias;
  p.act = act;
  if (p.total == 0) return staged ? 1 : 0;
  if (grid <= 0 || grid > p.total) grid = static_cast<int>(p.total);
  const bool multi = p.K > DC_KC;
  if (staged) {
    if (multi) emu::launch(grid, 256, [=]() { conv2d_direct_kernel<true, true>(output, input, kernel, p); });
    else emu::launch(grid, 256, [=]() { conv2d_direct_kernel<false, true>(output, input, kernel, p); });
  } else {
    if (multi) emu::launch(grid, 256, [=]() { conv2d_direct_kernel<true, false>(output, input, kernel, p); });
    else emu::launch(grid, 256, [=]() { conv2d_direct_kernel<false, false>(output, input, kernel, p); });
  }
  return staged ? 1 : 0;
}

}  // extern "C"
