// layers.cuh -- the HBM-bound steps either side of the GEMM in the reference's intended use
// (SURVEY.md section 8f, rank 4): physical transposition / NCHW<->NHWC
// (laser/primitives/swapaxes.nim:16-112), im2col (benchmarks/convolution/conv2d_im2col.nim:44-93),
// the direct convolution (benchmarks/convolution/conv2d_direct_convolution.nim:8-76) and the strided N-d copy behind
// copyFrom (laser/tensor/initialization.nim:80-112).
// All of them move each byte once: coalesced 16-byte global accesses where the shapes allow,
// shared-memory tiles for the transposition, grids sized from the SM count by the host.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "simt_epilogue.cuh"

namespace lb200 {

// ---- batched 2-d transposition: dst[n][j][i] = src[n][i][j], src = N x [NR][NC] contiguous ----
// 64 x 64 element tiles through shared memory (row pitch 65 elements: the transposed read hits
// 2-way bank conflicts at worst, far from limiting an HBM-bound kernel).  V = elements per
// global access (4 when NR, NC are multiples of 4 and both bases are aligned to 4 elements,
// else 1).  256 threads: 16 accesses of V=4 per tile row, 16 rows per pass.
template <typename T>
struct alignas(sizeof(T) * 4 > 16 ? 16 : sizeof(T) * 4) Vec4 {
  T v[4];
};

// host side: may the 4-element accesses be used?
template <typename T>
inline bool transpose_can_vec(const void *dst, const void *src, int64_t NR, int64_t NC) {
  const uintptr_t align = sizeof(T) * 4 > 16 ? 16 : sizeof(T) * 4;
  return (NR % 4 == 0) && (NC % 4 == 0) && (reinterpret_cast<uintptr_t>(dst) % align == 0) &&
         (reinterpret_cast<uintptr_t>(src) % align == 0);
}
inline int64_t transpose_tiles(int64_t N, int64_t NR, int64_t NC) { return N * ((NR + 63) / 64) * ((NC + 63) / 64); }

template <typename T, int V>
__global__ void __launch_bounds__(256)
transpose_batched_kernel(T *__restrict__ dst, const T *__restrict__ src, int64_t N, int64_t NR, int64_t NC) {
  constexpr int TILE = 64;
  __shared__ T tile[TILE][TILE + 1];
  const int64_t tiles_r = (NR + TILE - 1) / TILE, tiles_c = (NC + TILE - 1) / TILE;
  const int64_t per_mat = tiles_r * tiles_c, total = per_mat * N;
  const int tid = threadIdx.x;
  for (int64_t t = blockIdx.x; t < total; t += gridDim.x) {
    const int64_t n = t / per_mat, rem = t - n * per_mat;
    const int64_t r0 = (rem / tiles_c) * TILE, c0 = (rem % tiles_c) * TILE;
    const T *s = src + n * NR * NC;
    T *d = dst + n * NR * NC;
    if constexpr (V == 4) {
      const int q = tid & 15, rr = tid >> 4;
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const int r = p * 16 + rr;
        if (r0 + r < NR && c0 + 4 * q < NC) {
          const Vec4<T> v = *reinterpret_cast<const Vec4<T> *>(s + (r0 + r) * NC + c0 + 4 * q);
#pragma unroll
          for (int e = 0; e < 4; ++e) tile[r][4 * q + e] = v.v[e];
        }
      }
      __syncthreads();
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const int j = p * 16 + rr;  // row of dst inside the tile = column of src
        if (c0 + j < NC && r0 + 4 * q < NR) {
          Vec4<T> v;
#pragma unroll
          for (int e = 0; e < 4; ++e) v.v[e] = tile[4 * q + e][j];
          *reinterpret_cast<Vec4<T> *>(d + (c0 + j) * NR + r0 + 4 * q) = v;
        }
      }
    } else {
      const int x = tid & 63, y = tid >> 6;  // 64 x 4
#pragma unroll 4
      for (int p = 0; p < 16; ++p) {
        const int r = p * 4 + y;
        if (r0 + r < NR && c0 + x < NC) tile[r][x] = s[(r0 + r) * NC + c0 + x];
      }
      __syncthreads();
#pragma unroll 4
      for (int p = 0; p < 16; ++p) {
        const int j = p * 4 + y;
        if (c0 + j < NC && r0 + x < NR) d[(c0 + j) * NR + r0 + x] = tile[x][j];
      }
    }
    __syncthreads();
  }
}

// ---- im2col: images x [C][H][W] -> images x [C*kH*kW][outH*outW], zero outside the image ----
struct Im2colParams {
  int C, H, W, kH, kW, pH, pW, sH, sW, outH, outW;
  int K;         // C * kH * kW  (rows of the workspace matrix)
  int outHW;     // columns
  int64_t rows;  // K * images
  int64_t in_image_stride, ws_image_stride;  // elements
  int tx_log2;   // threads along the columns = 1 << tx_log2 (each owns 4 consecutive columns)
  int chunks;    // column chunks of (4 * quads_per_thread << tx_log2) per row
  int quads_per_thread;   // consecutive groups of 4 columns one thread writes (row and column decoded once for all of them)
};

// host side: launch geometry.  geom = {C, H, W, kH, kW, pH, pW, sH, sW, outH, outW} (all < 2^31).
// Returns the number of blocks of 256 threads; *vec4 says whether the float4 store variant applies.
inline int64_t im2col_plan(const int64_t geom[11], int64_t images, const void *workspace, Im2colParams *p,
                           bool *vec4) {
  p->C = (int)geom[0]; p->H = (int)geom[1]; p->W = (int)geom[2]; p->kH = (int)geom[3]; p->kW = (int)geom[4];
  p->pH = (int)geom[5]; p->pW = (int)geom[6]; p->sH = (int)geom[7]; p->sW = (int)geom[8];
  p->outH = (int)geom[9]; p->outW = (int)geom[10];
  p->K = p->C * p->kH * p->kW;
  p->outHW = p->outH * p->outW;
  p->rows = static_cast<int64_t>(p->K) * images;
  p->in_image_stride = geom[0] * geom[1] * geom[2];
  p->ws_image_stride = static_cast<int64_t>(p->K) * p->outHW;
  const int quads = (p->outHW + 3) / 4;
  int tx_log2 = 0;
  while ((1 << tx_log2) < quads && tx_log2 < 8) ++tx_log2;
  p->tx_log2 = tx_log2;
  p->quads_per_thread = quads >= 1024 ? 4 : 1;
  const int per_chunk = p->quads_per_thread << tx_log2;
  p->chunks = (quads + per_chunk - 1) / per_chunk;
  const int rows_per_block = 256 >> tx_log2;
  *vec4 = (p->outHW % 4 == 0) && (reinterpret_cast<uintptr_t>(workspace) % 16 == 0);
  return ((p->rows + rows_per_block - 1) / rows_per_block) * p->chunks;
}

// thread (tx, ty): row = block_row_group * rows_per_block + ty, columns 4*((chunk*U + u)*TX + tx) .. +3 for u < U =
// quads_per_thread.  The row is decoded once per thread (kk -> c, krow, kcol), the column once per 4 outputs.
template <bool VEC4>
__global__ void __launch_bounds__(256)
im2col_kernel(float *__restrict__ ws, const float *__restrict__ in, Im2colParams p) {
  const int tx = threadIdx.x & ((1 << p.tx_log2) - 1), ty = threadIdx.x >> p.tx_log2;
  const int rows_per_block = 256 >> p.tx_log2;
  const int64_t blk = blockIdx.x;
  const int chunk = static_cast<int>(blk % p.chunks);
  const int64_t row = (blk / p.chunks) * rows_per_block + ty;
  if (row >= p.rows) return;
  const int64_t img = row / p.K;
  const int kk = static_cast<int>(row - img * p.K);
  const int khw = p.kH * p.kW;
  const int c = kk / khw, r2 = kk - c * khw;
  const int krow = r2 / p.kW, kcol = r2 - krow * p.kW;
  const float *src = in + img * p.in_image_stride + static_cast<int64_t>(c) * p.H * p.W;
  float *wrow = ws + img * p.ws_image_stride + static_cast<int64_t>(kk) * p.outHW;
  // quad u of this thread: lanes stay next to each other in every store instruction (the row was decoded once above)
  for (int u = 0; u < p.quads_per_thread; ++u) {
    const int p0 = (((chunk * p.quads_per_thread + u) << p.tx_log2) + tx) * 4;
    if (p0 >= p.outHW) return;
    int oh = p0 / p.outW, ow = p0 - oh * p.outW;
    float *dst = wrow + p0;
    float v[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int r = oh * p.sH - p.pH + krow, cc = ow * p.sW - p.pW + kcol;
      const bool inside = (p0 + e < p.outHW) && static_cast<unsigned>(r) < static_cast<unsigned>(p.H) &&
                          static_cast<unsigned>(cc) < static_cast<unsigned>(p.W);
      v[e] = inside ? src[static_cast<int64_t>(r) * p.W + cc] : 0.0f;
      if (++ow == p.outW) { ow = 0; ++oh; }
    }
    if constexpr (VEC4) {
      *reinterpret_cast<float4 *>(dst) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (p0 + e < p.outHW) dst[e] = v[e];
    }
  }
}

// ---- direct convolution: images x [C][H][W] (*) [Cout][C][kH][kW] -> images x [Cout][outH][outW], no workspace ----
// Every output is the value the exact im2col path computes (im2col_kernel, then the exact GEMM with M = Cout, K = C*kH*kW,
// N = outH*outW): one __fmaf_rn chain from +0 over ascending tap kk = (ci*kH + kr)*kW + kc inside blocks of DC_KC taps,
// the blocks summed in order (x = 0 + blk0, x = x + blk1, ...), taps outside the image multiplied as zeros, and the bias +
// activation applied once to the final sum through simt_bias_act (bias per output channel = per GEMM row).
//
// Work unit ("tile"): DC_PIX consecutive output pixels (flattened oh * outW + ow) of one image x DC_CG output channels; a
// 1-d grid strides over images x tiles x channel groups (decoded in 64 bits).  Thread t owns the pixels p0 + t + j*256,
// j < DC_CPT, so every store of a warp writes 32 consecutive floats of one output plane (one 128-byte line) and the
// staged-input reads of a warp hit consecutive shared-memory words.  It keeps DC_CPT x DC_CG running sums (and as many
// block totals when K > DC_KC) in registers.
//   STAGED: per chunk of `cc` input channels the rows the tile's taps touch are copied to shared memory at full padded
//           width, zero outside the image, next to the chunk's weights of the channel group ([tap][co], two 16-byte
//           broadcast reads per tap) and a table of each tap's offset inside the staged window.
//   not STAGED (a single staged channel would exceed DC_SMEM_BYTES: very wide images): weights in 512-tap chunks, input
//           read from global memory with a bounds check per tap.
constexpr int DC_CG = 8;                // output channels per group
constexpr int DC_CPT = 4;               // pixels per thread
constexpr int DC_PIX = 256 * DC_CPT;    // pixels per tile
constexpr int DC_KC = 2048 / 4;         // taps per summation block: the exact GEMM's kc (gemm_tiling.nim:310)
constexpr int DC_SMEM_BYTES = 48 * 1024;   // static shared memory of one block (3 blocks fit an SM's 227 KB)

struct DirectConvParams {
  int C, H, W, Cout, kH, kW, pH, pW, sH, sW, outH, outW;
  int K, khw, outHW;
  int tiles, groups;       // pixel tiles per image, channel groups
  int64_t total;           // images * tiles * groups
  int cc;                  // STAGED: input channels per chunk
  int rows, pitch, plane;  // STAGED: staged rows per channel, row pitch (floats), rows * pitch
  int ws_off, toff_off;    // STAGED: float offsets of the weights and of the tap-offset table in shared memory
  const float *bias;       // NULL or Cout values (device)
  int act;                 // 0 none, 1 relu, 2 tanh, 3 sigmoid
};

// host side: launch geometry.  geom = {C, H, W, Cout, kH, kW, pH, pW, sH, sW, outH, outW} (checked by conv_geom).
// Returns whether the STAGED variant of the kernel applies (always false with stage_input = false: the variant that reads
// the input from global memory, which the library takes only when one staged channel does not fit DC_SMEM_BYTES).
inline bool direct_conv_plan(const int64_t geom[12], int64_t images, DirectConvParams *p, bool stage_input = true) {
  p->C = (int)geom[0]; p->H = (int)geom[1]; p->W = (int)geom[2]; p->Cout = (int)geom[3];
  p->kH = (int)geom[4]; p->kW = (int)geom[5]; p->pH = (int)geom[6]; p->pW = (int)geom[7];
  p->sH = (int)geom[8]; p->sW = (int)geom[9]; p->outH = (int)geom[10]; p->outW = (int)geom[11];
  p->khw = p->kH * p->kW;
  p->K = p->C * p->khw;
  p->outHW = p->outH * p->outW;
  p->tiles = (p->outHW + DC_PIX - 1) / DC_PIX;
  p->groups = (p->Cout + DC_CG - 1) / DC_CG;
  p->total = images * p->tiles * p->groups;
  p->bias = nullptr;
  p->act = 0;
  // output rows a tile of DC_PIX consecutive pixels can touch, hence input rows and the padded width it needs
  const int64_t pix = p->outHW < DC_PIX ? p->outHW : DC_PIX;
  int64_t span = (pix - 1 + p->outW - 1) / p->outW + 1;
  if (span > p->outH) span = p->outH;
  const int64_t rows = (span - 1) * geom[8] + geom[4], pitch = (geom[11] - 1) * geom[9] + geom[5];
  const int64_t plane = rows * pitch, budget = DC_SMEM_BYTES / 4;
  int64_t cc = 0;
  if (stage_input && plane < budget) {
    cc = budget / (plane + static_cast<int64_t>(p->khw) * (DC_CG + 1) + 4);
    if (cc > p->C) cc = p->C;
    while (cc > 0 && (cc * plane + 3) / 4 * 4 + cc * p->khw * (DC_CG + 1) > budget) --cc;
  }
  if (cc == 0) {   // weights + (ci, kr, kc) of each tap of a 512-tap chunk: (8 + 3) * 512 * 4 bytes = 22 KB
    p->cc = 0; p->rows = p->pitch = p->plane = 0;
    p->ws_off = 0;
    p->toff_off = DC_KC * DC_CG;
    return false;
  }
  p->cc = static_cast<int>(cc);
  p->rows = static_cast<int>(rows); p->pitch = static_cast<int>(pitch); p->plane = static_cast<int>(plane);
  p->ws_off = static_cast<int>((cc * plane + 3) / 4 * 4);   // 16-byte aligned weights
  p->toff_off = p->ws_off + static_cast<int>(cc) * p->khw * DC_CG;
  return true;
}

template <bool MULTI, bool STAGED>
__global__ void __launch_bounds__(256)
conv2d_direct_kernel(float *__restrict__ out, const float *__restrict__ in, const float *__restrict__ ker, DirectConvParams p) {
  __shared__ float4 dc_smem4[DC_SMEM_BYTES / 16];
  float *smem = reinterpret_cast<float *>(dc_smem4);
  float *ws = smem + p.ws_off;                                   // [tap][DC_CG] weights of the current chunk
  int *toff = reinterpret_cast<int *>(smem + p.toff_off);        // STAGED: tap -> window offset; else (ci, kr, kc) x 512
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if constexpr (STAGED) {   // the same for every chunk: channel-local tap tl -> (tl / khw) * plane + kr * pitch + kc
    for (int tl = tid; tl < p.cc * p.khw; tl += 256) {
      const int ci = tl / p.khw, r = tl - ci * p.khw, kr = r / p.kW;
      toff[tl] = ci * p.plane + kr * p.pitch + (r - kr * p.kW);
    }
  }
  for (int64_t t = blockIdx.x; t < p.total; t += gridDim.x) {
    const int g = static_cast<int>(t % p.groups);
    const int64_t rest = t / p.groups;
    const int tile = static_cast<int>(rest % p.tiles);
    const int64_t n = rest / p.tiles;
    const int co0 = g * DC_CG, p0 = tile * DC_PIX, oh_a = p0 / p.outW;
    const float *img = in + n * static_cast<int64_t>(p.C) * p.H * p.W;
    const int64_t HW = static_cast<int64_t>(p.H) * p.W;
    int base[DC_CPT], ih0[DC_CPT], iw0[DC_CPT];   // STAGED: window offset of the pixel's first tap; else its image position
    bool live[DC_CPT];
#pragma unroll
    for (int j = 0; j < DC_CPT; ++j) {
      const int pix = p0 + tid + j * 256;
      live[j] = pix < p.outHW;
      const int oh = live[j] ? pix / p.outW : oh_a, ow = live[j] ? pix - oh * p.outW : 0;
      base[j] = (oh - oh_a) * p.sH * p.pitch + ow * p.sW;
      ih0[j] = oh * p.sH - p.pH;
      iw0[j] = ow * p.sW - p.pW;
    }
    float acc[DC_CPT][DC_CG], x[DC_CPT][DC_CG];
#pragma unroll
    for (int j = 0; j < DC_CPT; ++j)
#pragma unroll
      for (int c = 0; c < DC_CG; ++c) { acc[j][c] = 0.0f; x[j][c] = 0.0f; }
    // end of a summation block: x = x + blk (x starts at +0: the exact GEMM's beta = 0 epilogue, then beta' = 1)
    auto flush = [&]() {
#pragma unroll
      for (int j = 0; j < DC_CPT; ++j)
#pragma unroll
        for (int c = 0; c < DC_CG; ++c) { x[j][c] = __fadd_rn(x[j][c], acc[j][c]); acc[j][c] = 0.0f; }
    };
    auto fma_tap = [&](const float *w, const float *v) {
#pragma unroll
      for (int j = 0; j < DC_CPT; ++j)
#pragma unroll
        for (int c = 0; c < DC_CG; ++c) acc[j][c] = __fmaf_rn(w[c], v[j], acc[j][c]);
    };
    if constexpr (STAGED) {
      const int ih_a = oh_a * p.sH - p.pH;
      for (int c0 = 0; c0 < p.C; c0 += p.cc) {
        const int cn = p.C - c0 < p.cc ? p.C - c0 : p.cc;
        __syncthreads();   // the previous chunk (or tile) is consumed
        // input: one warp per staged row, lanes along it (window column q <-> image column q - pW)
        for (int rr = warp; rr < cn * p.rows; rr += 8) {
          const int ci = rr / p.rows, ih = ih_a + (rr - ci * p.rows);
          float *dst = smem + static_cast<int64_t>(rr) * p.pitch;
          if (static_cast<unsigned>(ih) < static_cast<unsigned>(p.H)) {
            const float *src = img + (c0 + ci) * HW + static_cast<int64_t>(ih) * p.W;
            for (int q = lane; q < p.pitch; q += 32) {
              const int iw = q - p.pW;
              dst[q] = static_cast<unsigned>(iw) < static_cast<unsigned>(p.W) ? src[iw] : 0.0f;
            }
          } else {
            for (int q = lane; q < p.pitch; q += 32) dst[q] = 0.0f;
          }
        }
        for (int i = tid; i < cn * p.khw * DC_CG; i += 256) {
          const int tl = i / DC_CG, c = i - tl * DC_CG;
          ws[i] = co0 + c < p.Cout ? ker[static_cast<int64_t>(co0 + c) * p.K + c0 * p.khw + tl] : 0.0f;
        }
        __syncthreads();
        const int taps = cn * p.khw, kk0 = c0 * p.khw;
#pragma unroll 2
        for (int tl = 0; tl < taps; ++tl) {
          const float4 wa = reinterpret_cast<const float4 *>(ws)[2 * tl], wb = reinterpret_cast<const float4 *>(ws)[2 * tl + 1];
          const float w[DC_CG] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
          const int off = toff[tl];
          float v[DC_CPT];
#pragma unroll
          for (int j = 0; j < DC_CPT; ++j) v[j] = smem[base[j] + off];
          fma_tap(w, v);
          if constexpr (MULTI) {
            if (((kk0 + tl + 1) & (DC_KC - 1)) == 0) flush();   // block boundaries follow kk, not the channel chunks
          }
        }
      }
      if constexpr (MULTI) {
        if (p.K & (DC_KC - 1)) flush();   // the last, partial block
      }
    } else {
      int *tci = toff, *tkr = toff + DC_KC, *tkc = toff + 2 * DC_KC;
      for (int k0 = 0; k0 < p.K; k0 += DC_KC) {   // one chunk = one summation block
        const int kn = p.K - k0 < DC_KC ? p.K - k0 : DC_KC;
        __syncthreads();
        for (int i = tid; i < kn * DC_CG; i += 256) {
          const int tl = i / DC_CG, c = i - tl * DC_CG;
          ws[i] = co0 + c < p.Cout ? ker[static_cast<int64_t>(co0 + c) * p.K + k0 + tl] : 0.0f;
        }
        for (int tl = tid; tl < kn; tl += 256) {
          const int kk = k0 + tl, ci = kk / p.khw, r = kk - ci * p.khw, kr = r / p.kW;
          tci[tl] = ci; tkr[tl] = kr; tkc[tl] = r - kr * p.kW;
        }
        __syncthreads();
        for (int tl = 0; tl < kn; ++tl) {
          const float *w = ws + tl * DC_CG;
          const int kr = tkr[tl], kc = tkc[tl];
          const float *plane = img + tci[tl] * HW;
          float v[DC_CPT];
#pragma unroll
          for (int j = 0; j < DC_CPT; ++j) {
            const int ih = ih0[j] + kr, iw = iw0[j] + kc;
            v[j] = live[j] && static_cast<unsigned>(ih) < static_cast<unsigned>(p.H) &&
                           static_cast<unsigned>(iw) < static_cast<unsigned>(p.W)
                       ? plane[static_cast<int64_t>(ih) * p.W + iw]
                       : 0.0f;
          }
          float wr[DC_CG];
#pragma unroll
          for (int c = 0; c < DC_CG; ++c) wr[c] = w[c];
          fma_tap(wr, v);
        }
        if constexpr (MULTI) flush();
      }
    }
    // the single store: act(x + bias[co]) for every live pixel of the group's channels
    const bool has_epi = p.bias != nullptr || p.act != 0;
#pragma unroll
    for (int c = 0; c < DC_CG; ++c) {
      if (co0 + c >= p.Cout) break;
      float *oplane = out + (n * p.Cout + co0 + c) * static_cast<int64_t>(p.outHW);
#pragma unroll
      for (int j = 0; j < DC_CPT; ++j) {
        if (!live[j]) continue;
        float v = MULTI ? x[j][c] : __fadd_rn(0.0f, acc[j][c]);
        if (has_epi) v = simt_bias_act(v, p.bias, 1, p.act, co0 + c, p0 + tid + j * 256);
        oplane[p0 + tid + j * 256] = v;
      }
    }
  }
}

// ---- strided N-d copy (copyFrom): dst[idx] = src[idx] over a common shape, rank <= 6 ----
struct CopyParams {
  int rank;
  int64_t shape[6], dst_strides[6], src_strides[6];  // elements; innermost dimension last
  int64_t total;
};
// host side: merge neighbouring dimensions that are contiguous in both views, drop extents of 1
inline void copy_plan(int rank, const int64_t *shape, const int64_t *dst_strides, const int64_t *src_strides,
                      CopyParams *p) {
  p->rank = 0;
  p->total = 1;
  for (int d = 0; d < rank; ++d) {
    p->total *= shape[d];
    if (shape[d] == 1) continue;
    if (p->rank > 0 && p->dst_strides[p->rank - 1] == dst_strides[d] * shape[d] &&
        p->src_strides[p->rank - 1] == src_strides[d] * shape[d]) {
      p->shape[p->rank - 1] *= shape[d];
      p->dst_strides[p->rank - 1] = dst_strides[d];
      p->src_strides[p->rank - 1] = src_strides[d];
    } else {
      p->shape[p->rank] = shape[d];
      p->dst_strides[p->rank] = dst_strides[d];
      p->src_strides[p->rank] = src_strides[d];
      ++p->rank;
    }
  }
  for (int d = p->rank; d < 6; ++d) { p->shape[d] = 1; p->dst_strides[d] = 0; p->src_strides[d] = 0; }
}

template <typename T>
__global__ void __launch_bounds__(256)
copy_strided_kernel(T *__restrict__ dst, const T *__restrict__ src, CopyParams p) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < p.total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    int64_t rem = i, od = 0, os = 0;
#pragma unroll
    for (int d = 5; d >= 0; --d) {
      if (d < p.rank) {
        const int64_t q = rem / p.shape[d], x = rem - q * p.shape[d];
        od += x * p.dst_strides[d];
        os += x * p.src_strides[d];
        rem = q;
      }
    }
    dst[od] = src[os];
  }
}


// ---- forEach over up to four equal-shape strided views (laser/strided_iteration/foreach.nim:229-251) ----
// `forEach o in out, x in a, y in b, z in c: <body>` -- the body cannot cross a C ABI, so the bodies
// the reference's own code, docs and iteration benchmark use are provided as opcodes.
enum ForeachOp : int {
  FE_COPY = 0,    // o = x                      (copyFrom / deepCopy, initialization.nim:68,104)
  FE_FILL = 1,    // o = alpha
  FE_SCALE = 2,   // o = alpha * x
  FE_ADD = 3,     // o = x + y
  FE_SUB = 4,     // o = x - y
  FE_MUL = 5,     // o = x * y
  FE_FMA = 6,     // o = x + y * z               (`x += y * z`, foreach.nim:231-232, with o aliasing x)
  FE_AXPY = 7,    // o = alpha * x + y
  FE_BENCH = 8,   // o = x + y - sin(z)          (benchmarks/loop_iteration/iter_bench_prod.nim:88-90)
  FE_NUM_OPS = 9
};
struct ForeachParams {
  int rank;
  int64_t shape[6];
  int64_t strides[4][6];   // o, x, y, z (elements; 0 for unused operands)
  int64_t total;
};
// host side: merge neighbouring dimensions contiguous in every operand, drop extents of 1
inline void foreach_plan(int rank, const int64_t *shape, const int64_t *const strides[4], ForeachParams *p) {
  p->rank = 0;
  p->total = 1;
  for (int d = 0; d < rank; ++d) {
    p->total *= shape[d];
    if (shape[d] == 1) continue;
    bool merge = p->rank > 0;
    for (int t = 0; t < 4 && merge; ++t)
      merge = p->strides[t][p->rank - 1] == (strides[t] ? strides[t][d] : 0) * shape[d];
    if (merge) {
      p->shape[p->rank - 1] *= shape[d];
      for (int t = 0; t < 4; ++t) p->strides[t][p->rank - 1] = strides[t] ? strides[t][d] : 0;
    } else {
      p->shape[p->rank] = shape[d];
      for (int t = 0; t < 4; ++t) p->strides[t][p->rank] = strides[t] ? strides[t][d] : 0;
      ++p->rank;
    }
  }
  for (int d = p->rank; d < 6; ++d) {
    p->shape[d] = 1;
    for (int t = 0; t < 4; ++t) p->strides[t][d] = 0;
  }
}
template <typename T> __device__ __forceinline__ T fe_sin(T v);
template <> __device__ __forceinline__ float fe_sin<float>(float v) { return sinf(v); }
template <> __device__ __forceinline__ double fe_sin<double>(double v) { return sin(v); }

template <typename T, int OP>
__global__ void __launch_bounds__(256)
foreach_strided_kernel(T *o, const T *x, const T *y, const T *z, ForeachParams p, T alpha) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < p.total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    int64_t rem = i, off[4] = {0, 0, 0, 0};
#pragma unroll
    for (int d = 5; d >= 0; --d) {
      if (d < p.rank) {
        const int64_t q = rem / p.shape[d], c = rem - q * p.shape[d];
#pragma unroll
        for (int t = 0; t < 4; ++t) off[t] += c * p.strides[t][d];
        rem = q;
      }
    }
    T v;
    if constexpr (OP == FE_COPY) v = x[off[1]];
    else if constexpr (OP == FE_FILL) v = alpha;
    else if constexpr (OP == FE_SCALE) v = alpha * x[off[1]];
    else if constexpr (OP == FE_ADD) v = x[off[1]] + y[off[2]];
    else if constexpr (OP == FE_SUB) v = x[off[1]] - y[off[2]];
    else if constexpr (OP == FE_MUL) v = x[off[1]] * y[off[2]];
    else if constexpr (OP == FE_FMA) v = x[off[1]] + y[off[2]] * z[off[3]];
    else if constexpr (OP == FE_AXPY) v = alpha * x[off[1]] + y[off[2]];
    else v = x[off[1]] + y[off[2]] - fe_sin<T>(z[off[3]]);
    o[off[0]] = v;
  }
}
// operands an opcode reads (bit 0: x, bit 1: y, bit 2: z)
inline int foreach_operands(int op) {
  switch (op) {
    case FE_COPY: case FE_SCALE: return 1;
    case FE_FILL: return 0;
    case FE_ADD: case FE_SUB: case FE_MUL: case FE_AXPY: return 3;
    case FE_FMA: case FE_BENCH: return 7;
    default: return -1;
  }
}

}  // namespace lb200
