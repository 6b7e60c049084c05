// PSNR, SSIM and MS-SSIM of the evaluation loop (compress.py --metrics): src/helpers/metrics.py:7-18 (psnr), 37-63
// (gaussian_filter), 66-103 (_ssim), 106-161 (ssim), 164-236 (ms_ssim).
//
// ssim_level_kernel: one SSIM level.  CTA = one (n, c) plane x one 32 x 64 tile of valid outputs.  It stages the tile plus
// its (win - 1) halo of X and Y (and one leading zero row / column: the top / left padding of an odd dimension's pooling)
// in shared memory, runs the separable window over the five moments x, y, x^2, y^2, xy (vertical pass first, as the
// reference's conv2d pair does; both passes register-blocked, taps in registers), forms ssim / cs per output pixel and
// writes the CTA's double partial sums to its own workspace slot.  The same CTA writes pooled tile (ty, tx) (16 x 32
// pooled pixels) of this level's 2x2 average pool, the next level's input: every pooled pixel has exactly one owner.
// ssim_finalize_kernel: one CTA sums the partials in a fixed order (no float atomics: results are bit-reproducible and do
// not depend on the batch size) and forms the per-plane and per-image / batch values.
// psnr_*: per-image sum of (x - y)^2 in fp64, fixed-order two-launch reduction, fp64 log10.
//
// Backward (2 * levels + 1 launches, coarse level first):
// ssim_grad_coeffs_kernel: per (plane, level) the weights alpha / beta of each output's ssim / cs in the upstream
// gradient, from the per-plane level sums the forward's finalize left in the workspace and the upstream gradient on the
// device (no host read).
// ssim_level_kernel<MAXW, true>: the forward's staging and filter passes again (the same instantiated code, so the same
// moments bit for bit), then the four gradient maps d/d(mu1, mu2, exx = eyy, exy) per valid output (16 B each).
// ssim_level_bwd_kernel: CTA = one (n, c) plane x one 32 x 64 tile of the level's INPUT.  It stages the four maps with a
// (win - 1) halo before the tile, applies the adjoint window (flipped taps, vertical then horizontal), combines with x and
// y, adds 0.25 x the next level's input gradient at the pooled pixel that read this one, and writes dx / dy.  Every input
// pixel has one owner and no float atomics are used: the gradients are bit-reproducible and independent of the batch.
#include "hfc_internal.h"
#include "ssim_math.cuh"

namespace hfc {

constexpr int kSsimThreads = 256;
constexpr int kVertRows = 4;          // vertical pass: outputs per thread along h
constexpr int kHorzCols = 8;          // horizontal pass: outputs per thread along w
static_assert(kSsimTileH * (kSsimTileW / kHorzCols) == kSsimThreads, "one horizontal item per thread");

struct SsimLevelArgs {
  const float* x;
  const float* y;
  float* px;                  // pooled outputs (nullptr at the last level)
  float* py;
  const float* taps;          // [c][win]
  double* partials;           // [planes][tiles][2]
  int c, win;
  float c1, c2;
  SsimLevelGeom g;
  // gradient maps (GRAD instantiation only)
  const float* coef;          // [planes][levels][2] (alpha, beta)
  float4* maps;               // [planes][ho][wo] (gmu1, gmu2, gE, gXY)
  int level, levels;
};

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

template <int MAXW, bool GRAD>
__global__ void __launch_bounds__(kSsimThreads)
ssim_level_kernel(SsimLevelArgs a) {
  extern __shared__ float smem[];
  __shared__ float staps[2][MAXW];
  __shared__ double red[kSsimThreads / 32][2];
  const SsimLevelGeom& g = a.g;
  const int SR = ssim_stage_rows(g), SC = ssim_stage_cols(g);
  const int VC = kSsimTileW + g.ww - 1, VP = VC | 1;          // odd pitch: the horizontal pass reads down columns
  float* sx = smem;
  float* sy = sx + SR * SC;
  float* sv = sy + SR * SC;                                     // [5][TH][VP] vertically filtered moments
  const int64_t plane = blockIdx.y;
  const int tile = blockIdx.x, ty = tile / g.tiles_x, tx = tile - ty * g.tiles_x;
  const int r0 = ty * kSsimTileH, c0 = tx * kSsimTileW;
  const int tid = threadIdx.x;
  const int64_t base = plane * static_cast<int64_t>(g.h) * g.w;
  const int ch = static_cast<int>(plane % a.c);
  if constexpr (GRAD) {
    if (r0 >= g.ho || c0 >= g.wo) return;                       // a tile the grid has only for the pooled plane
  }

  if (tid < MAXW) {
    const float t = tid < a.win ? a.taps[static_cast<int64_t>(ch) * a.win + tid] : 0.f;
    staps[0][tid] = g.wh == 1 ? (tid == 0 ? 1.f : 0.f) : t;
    staps[1][tid] = g.ww == 1 ? (tid == 0 ? 1.f : 0.f) : t;
  }
  for (int i = tid; i < SR * SC; i += kSsimThreads) {
    const int rr = i / SC, cc = i - rr * SC;
    const int gr = r0 - 1 + rr, gc = c0 - 1 + cc;
    const bool in = gr >= 0 && gr < g.h && gc >= 0 && gc < g.w;
    const int64_t off = base + static_cast<int64_t>(gr) * g.w + gc;
    sx[i] = in ? __ldg(a.x + off) : 0.f;
    sy[i] = in ? __ldg(a.y + off) : 0.f;
  }
  __syncthreads();

  // vertical pass: item = (group of kVertRows output rows, one column of the halo-wide tile)
  {
    float w[MAXW];
#pragma unroll
    for (int k = 0; k < MAXW; ++k) w[k] = staps[0][k];
    const int items = (kSsimTileH / kVertRows) * VC;
    for (int it = tid; it < items; it += kSsimThreads) {
      const int rg = it / VC, j = it - rg * VC;
      float acc[5][kVertRows];
#pragma unroll
      for (int m = 0; m < 5; ++m)
#pragma unroll
        for (int r = 0; r < kVertRows; ++r) acc[m][r] = 0.f;
#pragma unroll
      for (int t = 0; t < kVertRows + MAXW - 1; ++t) {
        if (t < kVertRows + g.wh - 1) {
          const int s = (rg * kVertRows + t + 1) * SC + j + 1;
          const float xv = sx[s], yv = sy[s];
          const float v[5] = {xv, yv, mul_rn(xv, xv), mul_rn(yv, yv), mul_rn(xv, yv)};
#pragma unroll
          for (int r = 0; r < kVertRows; ++r) {
            const int k = t - r;
            if (k >= 0 && k < MAXW && k < g.wh) {
#pragma unroll
              for (int m = 0; m < 5; ++m) acc[m][r] = fmaf(w[k < 0 ? 0 : k], v[m], acc[m][r]);
            }
          }
        }
      }
#pragma unroll
      for (int m = 0; m < 5; ++m)
#pragma unroll
        for (int r = 0; r < kVertRows; ++r) sv[(m * kSsimTileH + rg * kVertRows + r) * VP + j] = acc[m][r];
    }
  }
  __syncthreads();

  // horizontal pass + per-pixel ssim / cs: item = (output row, group of kHorzCols output columns)
  double s_acc = 0.0, c_acc = 0.0;
  {
    float w[MAXW];
#pragma unroll
    for (int k = 0; k < MAXW; ++k) w[k] = staps[1][k];
    const int i = tid % kSsimTileH, j0 = (tid / kSsimTileH) * kHorzCols;
    float acc[5][kHorzCols];
#pragma unroll
    for (int m = 0; m < 5; ++m)
#pragma unroll
      for (int r = 0; r < kHorzCols; ++r) acc[m][r] = 0.f;
#pragma unroll
    for (int t = 0; t < kHorzCols + MAXW - 1; ++t) {
      if (t < kHorzCols + g.ww - 1) {
        float v[5];
#pragma unroll
        for (int m = 0; m < 5; ++m) v[m] = sv[(m * kSsimTileH + i) * VP + j0 + t];
#pragma unroll
        for (int r = 0; r < kHorzCols; ++r) {
          const int k = t - r;
          if (k >= 0 && k < MAXW && k < g.ww) {
#pragma unroll
            for (int m = 0; m < 5; ++m) acc[m][r] = fmaf(w[k < 0 ? 0 : k], v[m], acc[m][r]);
          }
        }
      }
    }
    if constexpr (GRAD) {
      const float* cf = a.coef + (plane * a.levels + a.level) * 2;
      const float alpha = cf[0], beta = cf[1];
      if (r0 + i < g.ho) {
        float4* dst = a.maps + (plane * g.ho + r0 + i) * static_cast<int64_t>(g.wo) + c0 + j0;
#pragma unroll
        for (int r = 0; r < kHorzCols; ++r) {
          if (c0 + j0 + r < g.wo) {
            float4 m;
            ssim_grad_maps(acc[0][r], acc[1][r], acc[2][r], acc[3][r], acc[4][r], a.c1, a.c2, alpha, beta, &m.x, &m.y,
                           &m.z, &m.w);
            dst[r] = m;
          }
        }
      }
      return;
    } else if (r0 + i < g.ho) {
#pragma unroll
      for (int r = 0; r < kHorzCols; ++r) {
        if (c0 + j0 + r < g.wo) {
          float s, c;
          ssim_from_moments(acc[0][r], acc[1][r], acc[2][r], acc[3][r], acc[4][r], a.c1, a.c2, &s, &c);
          s_acc += static_cast<double>(s);
          c_acc += static_cast<double>(c);
        }
      }
    }
  }

  // 2x2 average pool of the staged tile: pooled tile (ty, tx)
  if (a.px) {
    const int64_t pbase = plane * static_cast<int64_t>(g.hp) * g.wp;
    const int ph = g.h & 1, pw = g.w & 1;
    constexpr int PH = kSsimTileH / 2, PW = kSsimTileW / 2;
    for (int it = tid; it < PH * PW; it += kSsimThreads) {
      const int pi = it / PW, pj = it - pi * PW;
      const int gpi = ty * PH + pi, gpj = tx * PW + pj;
      if (gpi < g.hp && gpj < g.wp) {
        const int s = pooled_stage_index(pi, ph) * SC + pooled_stage_index(pj, pw);
        const int64_t o = pbase + static_cast<int64_t>(gpi) * g.wp + gpj;
        a.px[o] = pool4(sx[s], sx[s + 1], sx[s + SC], sx[s + SC + 1]);
        a.py[o] = pool4(sy[s], sy[s + 1], sy[s + SC], sy[s + SC + 1]);
      }
    }
  }

  s_acc = warp_sum_d(s_acc);
  c_acc = warp_sum_d(c_acc);
  const int warp = tid >> 5, lane = tid & 31;
  if (lane == 0) {
    red[warp][0] = s_acc;
    red[warp][1] = c_acc;
  }
  __syncthreads();
  if (tid == 0) {
    double s = 0.0, c = 0.0;
    for (int k = 0; k < kSsimThreads / 32; ++k) {
      s += red[k][0];
      c += red[k][1];
    }
    double* dst = a.partials + (plane * ssim_level_tiles(g) + tile) * 2;
    dst[0] = s;
    dst[1] = c;
  }
}

struct SsimFinalArgs {
  double* ws;
  int64_t planes;
  int n, c, h0, w0, win, levels, relu_last, size_average;
  float weights[kSsimMaxLevels];
  float* out;
};

constexpr int kFinalThreads = 1024;

__global__ void __launch_bounds__(kFinalThreads) ssim_finalize_kernel(SsimFinalArgs a) {
  __shared__ double red[kFinalThreads / 32];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  double* plane_sums = a.ws + ssim_partials_offset(a.planes, a.h0, a.w0, a.win, a.levels);
  double* vals = plane_sums + a.planes * a.levels * 2;
  // per (plane, level): a warp sums the level's tile partials, lane-strided then a fixed shuffle tree
  for (int64_t q = warp; q < a.planes * a.levels; q += kFinalThreads / 32) {
    const int64_t p = q / a.levels;
    const int l = static_cast<int>(q - p * a.levels);
    const int64_t tiles = ssim_level_tiles(ssim_level_geom(a.h0, a.w0, a.win, l));
    const double* src = a.ws + ssim_partials_offset(a.planes, a.h0, a.w0, a.win, l) + p * tiles * 2;
    double s = 0.0, c = 0.0;
    for (int64_t t = lane; t < tiles; t += 32) {
      s += src[2 * t];
      c += src[2 * t + 1];
    }
    s = warp_sum_d(s);
    c = warp_sum_d(c);
    if (lane == 0) {
      plane_sums[(p * a.levels + l) * 2] = s;
      plane_sums[(p * a.levels + l) * 2 + 1] = c;
    }
  }
  __syncthreads();
  for (int64_t p = tid; p < a.planes; p += kFinalThreads)
    vals[p] = ssim_plane_value(plane_sums + p * a.levels * 2, a.weights, a.levels, a.h0, a.w0, a.win, a.relu_last);
  __syncthreads();
  if (a.size_average) {
    double s = 0.0;
    for (int64_t p = tid; p < a.planes; p += kFinalThreads) s += vals[p];
    s = warp_sum_d(s);
    if (lane == 0) red[warp] = s;
    __syncthreads();
    if (tid == 0) {
      double t = 0.0;
      for (int k = 0; k < kFinalThreads / 32; ++k) t += red[k];
      a.out[0] = static_cast<float>(t / static_cast<double>(a.planes));
    }
  } else {
    for (int i = tid; i < a.n; i += kFinalThreads) {
      double s = 0.0;
      for (int ch = 0; ch < a.c; ++ch) s += vals[static_cast<int64_t>(i) * a.c + ch];
      a.out[i] = static_cast<float>(s / a.c);
    }
  }
}

struct SsimGradCoefArgs {
  const double* plane_sums;   // [planes][levels][2]
  const float* grad_out;      // [1] (size_average) or [n]
  float* coef;                // [planes][levels][2]
  int64_t planes;
  int c, h0, w0, win, levels, relu_last, size_average;
  float weights[kSsimMaxLevels];
};

__global__ void ssim_grad_coeffs_kernel(SsimGradCoefArgs a) {
  for (int64_t p = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; p < a.planes;
       p += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const double dv = ssim_grad_dv(a.grad_out, p, a.planes, a.c, a.size_average);
    ssim_grad_coeffs(a.plane_sums + p * a.levels * 2, a.weights, a.levels, a.h0, a.w0, a.win, a.relu_last, dv,
                     a.coef + p * a.levels * 2);
  }
}

struct SsimLevelBwdArgs {
  const float* x;
  const float* y;
  const float4* maps;         // [planes][ho][wo]
  const float* taps;          // [c][win]
  const float* dx_coarse;     // [planes][hp][wp] or nullptr (last level)
  const float* dy_coarse;
  float* dx;                  // [planes][h][w] or nullptr (not needed)
  float* dy;
  int c, win;
  SsimLevelGeom g;
};

constexpr int kBwdMaps = 4;

template <int MAXW>
__global__ void __launch_bounds__(kSsimThreads)
ssim_level_bwd_kernel(SsimLevelBwdArgs a) {
  extern __shared__ float smem[];
  __shared__ float staps[2][MAXW];
  const SsimLevelGeom& g = a.g;
  const int SR = ssim_bwd_stage_rows(g), SC = ssim_bwd_stage_cols(g), VP = SC | 1;
  float* sm = smem;                                             // [4][SR][SC] staged maps
  float* sv = sm + kBwdMaps * SR * SC;                          // [4][TH][VP] vertically filtered maps
  const int64_t plane = blockIdx.y;
  const int tile = blockIdx.x, ty = tile / ssim_bwd_tiles_x(g), tx = tile - ty * ssim_bwd_tiles_x(g);
  const int r0 = ty * kSsimTileH, c0 = tx * kSsimTileW;
  const int tid = threadIdx.x;
  const int ch = static_cast<int>(plane % a.c);

  if (tid < MAXW) {                                             // flipped taps; a 1-tap identity where not smoothed
    const float t = tid < a.win ? a.taps[static_cast<int64_t>(ch) * a.win + (a.win - 1 - tid)] : 0.f;
    staps[0][tid] = g.wh == 1 ? (tid == 0 ? 1.f : 0.f) : t;
    staps[1][tid] = g.ww == 1 ? (tid == 0 ? 1.f : 0.f) : t;
  }
  const int64_t mbase = plane * static_cast<int64_t>(g.ho) * g.wo;
  for (int i = tid; i < SR * SC; i += kSsimThreads) {
    const int rr = i / SC, cc = i - rr * SC;
    const int orow = r0 - (g.wh - 1) + rr, ocol = c0 - (g.ww - 1) + cc;
    const bool in = orow >= 0 && orow < g.ho && ocol >= 0 && ocol < g.wo;
    const float4 m = in ? __ldg(a.maps + mbase + static_cast<int64_t>(orow) * g.wo + ocol) : make_float4(0.f, 0.f, 0.f, 0.f);
    sm[i] = m.x;
    sm[SR * SC + i] = m.y;
    sm[2 * SR * SC + i] = m.z;
    sm[3 * SR * SC + i] = m.w;
  }
  __syncthreads();

  // vertical adjoint pass: item = (group of kVertRows input rows, one column of the halo-wide tile)
  {
    float w[MAXW];
#pragma unroll
    for (int k = 0; k < MAXW; ++k) w[k] = staps[0][k];
    const int items = (kSsimTileH / kVertRows) * SC;
    for (int it = tid; it < items; it += kSsimThreads) {
      const int rg = it / SC, j = it - rg * SC;
      float acc[kBwdMaps][kVertRows];
#pragma unroll
      for (int m = 0; m < kBwdMaps; ++m)
#pragma unroll
        for (int r = 0; r < kVertRows; ++r) acc[m][r] = 0.f;
#pragma unroll
      for (int t = 0; t < kVertRows + MAXW - 1; ++t) {
        if (t < kVertRows + g.wh - 1) {
          const int s = (rg * kVertRows + t) * SC + j;
          float v[kBwdMaps];
#pragma unroll
          for (int m = 0; m < kBwdMaps; ++m) v[m] = sm[m * SR * SC + s];
#pragma unroll
          for (int r = 0; r < kVertRows; ++r) {
            const int k = t - r;
            if (k >= 0 && k < MAXW && k < g.wh) {
#pragma unroll
              for (int m = 0; m < kBwdMaps; ++m) acc[m][r] = fmaf(w[k < 0 ? 0 : k], v[m], acc[m][r]);
            }
          }
        }
      }
#pragma unroll
      for (int m = 0; m < kBwdMaps; ++m)
#pragma unroll
        for (int r = 0; r < kVertRows; ++r) sv[(m * kSsimTileH + rg * kVertRows + r) * VP + j] = acc[m][r];
    }
  }
  __syncthreads();

  // horizontal adjoint pass + combine: item = (input row, group of kHorzCols input columns)
  float w[MAXW];
#pragma unroll
  for (int k = 0; k < MAXW; ++k) w[k] = staps[1][k];
  const int i = tid % kSsimTileH, j0 = (tid / kSsimTileH) * kHorzCols;
  float acc[kBwdMaps][kHorzCols];
#pragma unroll
  for (int m = 0; m < kBwdMaps; ++m)
#pragma unroll
    for (int r = 0; r < kHorzCols; ++r) acc[m][r] = 0.f;
#pragma unroll
  for (int t = 0; t < kHorzCols + MAXW - 1; ++t) {
    if (t < kHorzCols + g.ww - 1) {
      float v[kBwdMaps];
#pragma unroll
      for (int m = 0; m < kBwdMaps; ++m) v[m] = sv[(m * kSsimTileH + i) * VP + j0 + t];
#pragma unroll
      for (int r = 0; r < kHorzCols; ++r) {
        const int k = t - r;
        if (k >= 0 && k < MAXW && k < g.ww) {
#pragma unroll
          for (int m = 0; m < kBwdMaps; ++m) acc[m][r] = fmaf(w[k < 0 ? 0 : k], v[m], acc[m][r]);
        }
      }
    }
  }
  const int gi = r0 + i;
  if (gi >= g.h) return;
  const int64_t base = plane * static_cast<int64_t>(g.h) * g.w + static_cast<int64_t>(gi) * g.w;
  const int64_t pbase = (plane * static_cast<int64_t>(g.hp) + pooled_index_of(gi, g.h & 1)) * g.wp;
#pragma unroll
  for (int r = 0; r < kHorzCols; ++r) {
    const int gj = c0 + j0 + r;
    if (gj < g.w) {
      const float xv = __ldg(a.x + base + gj), yv = __ldg(a.y + base + gj);
      const int64_t po = pbase + pooled_index_of(gj, g.w & 1);
      if (a.dx) a.dx[base + gj] = ssim_grad_combine(acc[0][r], acc[2][r], acc[3][r], xv, yv, a.dx_coarse ? __ldg(a.dx_coarse + po) : 0.f);
      if (a.dy) a.dy[base + gj] = ssim_grad_combine(acc[1][r], acc[2][r], acc[3][r], yv, xv, a.dy_coarse ? __ldg(a.dy_coarse + po) : 0.f);
    }
  }
}

constexpr int kPsnrThreads = 256;
constexpr int kPsnrUnroll = 4;

static int psnr_blocks(int64_t per_image) {
  const int64_t b = (per_image + kPsnrThreads * 16 - 1) / (kPsnrThreads * 16);
  return static_cast<int>(std::min<int64_t>(std::max<int64_t>(b, 1), 256));
}

__global__ void __launch_bounds__(kPsnrThreads)
psnr_partial_kernel(const float* __restrict__ a, const float* __restrict__ b, int64_t per_image, double* partials) {
  __shared__ double red[kPsnrThreads / 32];
  const int64_t base = static_cast<int64_t>(blockIdx.y) * per_image;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kPsnrThreads;
  double acc = 0.0;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * kPsnrThreads + threadIdx.x; i < per_image; i += stride * kPsnrUnroll) {
    float va[kPsnrUnroll], vb[kPsnrUnroll];
#pragma unroll
    for (int u = 0; u < kPsnrUnroll; ++u) {
      const int64_t k = i + u * stride;
      va[u] = k < per_image ? __ldg(a + base + k) : 0.f;
      vb[u] = k < per_image ? __ldg(b + base + k) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < kPsnrUnroll; ++u) {
      const double d = static_cast<double>(va[u]) - static_cast<double>(vb[u]);
      acc = fma(d, d, acc);
    }
  }
  acc = warp_sum_d(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int k = 0; k < kPsnrThreads / 32; ++k) s += red[k];
    partials[static_cast<int64_t>(blockIdx.y) * gridDim.x + blockIdx.x] = s;
  }
}

__global__ void psnr_finalize_kernel(const double* __restrict__ partials, int n, int blocks, int64_t per_image,
                                     double max_val, double* __restrict__ out) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    double s = 0.0;
    for (int k = 0; k < blocks; ++k) s += partials[static_cast<int64_t>(i) * blocks + k];
    const double mse = s / static_cast<double>(per_image);
    out[i] = 20.0 * log10(max_val) - 10.0 * log10(mse);
  }
}

}  // namespace hfc

using namespace hfc;

static size_t ssim_smem_bytes(const SsimLevelGeom& g) {
  const int VP = (kSsimTileW + g.ww - 1) | 1;
  return sizeof(float) * (2 * static_cast<size_t>(ssim_stage_rows(g)) * ssim_stage_cols(g) + 5 * kSsimTileH * VP);
}

template <int MAXW, bool GRAD>
static int launch_ssim_level(const SsimLevelArgs& a, int64_t planes, cudaStream_t st) {
  const size_t smem = ssim_smem_bytes(a.g);
  SsimLevelGeom big{};                 // the largest window's requirement (host-side attribute, no synchronisation)
  big.wh = big.ww = MAXW;
  cudaError_t e = cudaFuncSetAttribute(ssim_level_kernel<MAXW, GRAD>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(ssim_smem_bytes(big)));
  if (e != cudaSuccess) return set_error(HFC_ERR_LAUNCH, "ssim_level: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  dim3 grid(static_cast<unsigned>(ssim_level_tiles(a.g)), static_cast<unsigned>(planes));
  ssim_level_kernel<MAXW, GRAD><<<grid, kSsimThreads, smem, st>>>(a);
  return HFC_OK;
}

static size_t ssim_bwd_smem_bytes(const SsimLevelGeom& g) {
  const int SR = ssim_bwd_stage_rows(g), SC = ssim_bwd_stage_cols(g);
  return sizeof(float) * kBwdMaps * (static_cast<size_t>(SR) * SC + static_cast<size_t>(kSsimTileH) * (SC | 1));
}

template <int MAXW>
static int launch_ssim_level_bwd(const SsimLevelBwdArgs& a, int64_t planes, cudaStream_t st) {
  SsimLevelGeom big{};
  big.wh = big.ww = MAXW;
  cudaError_t e = cudaFuncSetAttribute(ssim_level_bwd_kernel<MAXW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(ssim_bwd_smem_bytes(big)));
  if (e != cudaSuccess)
    return set_error(HFC_ERR_LAUNCH, "ssim_level_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  dim3 grid(static_cast<unsigned>(ssim_bwd_tiles_y(a.g) * ssim_bwd_tiles_x(a.g)), static_cast<unsigned>(planes));
  ssim_level_bwd_kernel<MAXW><<<grid, kSsimThreads, ssim_bwd_smem_bytes(a.g), st>>>(a);
  return HFC_OK;
}

static int ssim_check(int32_t n, int32_t c, int32_t h0, int32_t w0, int32_t win, int32_t levels, const char* what) {
  if (n <= 0 || c <= 0 || h0 <= 0 || w0 <= 0) return set_error(HFC_ERR_INVALID, "%s: empty input", what);
  if (win < 1 || win % 2 == 0) return set_error(HFC_ERR_INVALID, "%s: window size must be odd", what);
  if (win > kSsimMaxWin) return set_error(HFC_ERR_UNSUPPORTED, "%s: window size %d > %d", what, win, kSsimMaxWin);
  if (levels < 1 || levels > kSsimMaxLevels)
    return set_error(HFC_ERR_UNSUPPORTED, "%s: 1..%d levels", what, kSsimMaxLevels);
  if (static_cast<int64_t>(n) * c > 65535) return set_error(HFC_ERR_UNSUPPORTED, "%s: n * c > 65535 planes", what);
  return HFC_OK;
}

extern "C" int64_t hfc_ssim_ws_bytes(int32_t n, int32_t c, int32_t h, int32_t w, int32_t win, int32_t levels) {
  if (ssim_check(n, c, h, w, win, levels, "ssim_ws_bytes") != HFC_OK) return -1;
  return ssim_ws_doubles(static_cast<int64_t>(n) * c, h, w, win, levels) * static_cast<int64_t>(sizeof(double));
}

extern "C" int hfc_ssim_level(const float* x, const float* y, int32_t n, int32_t c, int32_t h0, int32_t w0, int32_t level,
                              const float* taps, int32_t win, float c1, float c2, float* x_pooled, float* y_pooled,
                              void* ws, int64_t ws_bytes, void* stream) {
  int rc = ssim_check(n, c, h0, w0, win, level + 1, "ssim_level");
  if (rc != HFC_OK) return rc;
  if (!x || !y || !taps || !ws || (!x_pooled) != (!y_pooled))
    return set_error(HFC_ERR_INVALID, "ssim_level: null pointer");
  const int64_t planes = static_cast<int64_t>(n) * c;
  if (ws_bytes < ssim_partials_offset(planes, h0, w0, win, level + 1) * static_cast<int64_t>(sizeof(double)))
    return set_error(HFC_ERR_INVALID, "ssim_level: workspace too small");
  int sms = 0;
  rc = device_sm_count(&sms);
  if (rc != HFC_OK) return rc;
  SsimLevelArgs a;
  a.x = x;
  a.y = y;
  a.px = x_pooled;
  a.py = y_pooled;
  a.taps = taps;
  a.partials = static_cast<double*>(ws) + ssim_partials_offset(planes, h0, w0, win, level);
  a.c = c;
  a.win = win;
  a.c1 = c1;
  a.c2 = c2;
  a.g = ssim_level_geom(h0, w0, win, level);
  a.coef = nullptr;
  a.maps = nullptr;
  a.level = level;
  a.levels = level + 1;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = win <= 11 ? launch_ssim_level<11, false>(a, planes, st) : launch_ssim_level<kSsimMaxWin, false>(a, planes, st);
  if (rc != HFC_OK) return rc;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(HFC_ERR_LAUNCH, "ssim_level launch: %s", cudaGetErrorString(e));
  note_launch();
  return HFC_OK;
}

extern "C" int hfc_ssim_finalize(int32_t n, int32_t c, int32_t h0, int32_t w0, int32_t win, int32_t levels,
                                 const float* weights_host, int32_t relu_last, int32_t size_average, void* ws,
                                 int64_t ws_bytes, float* out, void* stream) {
  int rc = ssim_check(n, c, h0, w0, win, levels, "ssim_finalize");
  if (rc != HFC_OK) return rc;
  if (!weights_host || !ws || !out) return set_error(HFC_ERR_INVALID, "ssim_finalize: null pointer");
  const int64_t planes = static_cast<int64_t>(n) * c;
  if (ws_bytes < ssim_ws_doubles(planes, h0, w0, win, levels) * static_cast<int64_t>(sizeof(double)))
    return set_error(HFC_ERR_INVALID, "ssim_finalize: workspace too small");
  int sms = 0;
  rc = device_sm_count(&sms);
  if (rc != HFC_OK) return rc;
  SsimFinalArgs a;
  a.ws = static_cast<double*>(ws);
  a.planes = planes;
  a.n = n;
  a.c = c;
  a.h0 = h0;
  a.w0 = w0;
  a.win = win;
  a.levels = levels;
  a.relu_last = relu_last;
  a.size_average = size_average;
  for (int l = 0; l < kSsimMaxLevels; ++l) a.weights[l] = l < levels ? weights_host[l] : 0.f;
  a.out = out;
  ssim_finalize_kernel<<<1, kFinalThreads, 0, static_cast<cudaStream_t>(stream)>>>(a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(HFC_ERR_LAUNCH, "ssim_finalize launch: %s", cudaGetErrorString(e));
  note_launch();
  return HFC_OK;
}

extern "C" int64_t hfc_ssim_grad_maps_bytes(int32_t n, int32_t c, int32_t h0, int32_t w0, int32_t win, int32_t levels) {
  if (ssim_check(n, c, h0, w0, win, levels, "ssim_grad_maps_bytes") != HFC_OK) return -1;
  int64_t most = 0;
  for (int l = 0; l < levels; ++l) {
    const SsimLevelGeom g = ssim_level_geom(h0, w0, win, l);
    most = std::max<int64_t>(most, static_cast<int64_t>(g.ho) * g.wo);
  }
  return static_cast<int64_t>(n) * c * most * static_cast<int64_t>(sizeof(float4));
}

extern "C" int hfc_ssim_grad_coeffs(int32_t n, int32_t c, int32_t h0, int32_t w0, int32_t win, int32_t levels,
                                    const float* weights_host, int32_t relu_last, int32_t size_average, const void* ws,
                                    int64_t ws_bytes, const float* grad_out, float* coeffs, void* stream) {
  int rc = ssim_check(n, c, h0, w0, win, levels, "ssim_grad_coeffs");
  if (rc != HFC_OK) return rc;
  if (!weights_host || !ws || !grad_out || !coeffs) return set_error(HFC_ERR_INVALID, "ssim_grad_coeffs: null pointer");
  const int64_t planes = static_cast<int64_t>(n) * c;
  if (ws_bytes < ssim_ws_doubles(planes, h0, w0, win, levels) * static_cast<int64_t>(sizeof(double)))
    return set_error(HFC_ERR_INVALID, "ssim_grad_coeffs: workspace too small");
  SsimGradCoefArgs a;
  a.plane_sums = static_cast<const double*>(ws) + ssim_partials_offset(planes, h0, w0, win, levels);
  a.grad_out = grad_out;
  a.coef = coeffs;
  a.planes = planes;
  a.c = c;
  a.h0 = h0;
  a.w0 = w0;
  a.win = win;
  a.levels = levels;
  a.relu_last = relu_last;
  a.size_average = size_average;
  for (int l = 0; l < kSsimMaxLevels; ++l) a.weights[l] = l < levels ? weights_host[l] : 0.f;
  const int threads = 128;
  const int blocks = static_cast<int>(std::min<int64_t>((planes + threads - 1) / threads, 1024));
  ssim_grad_coeffs_kernel<<<blocks, threads, 0, static_cast<cudaStream_t>(stream)>>>(a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(HFC_ERR_LAUNCH, "ssim_grad_coeffs launch: %s", cudaGetErrorString(e));
  note_launch();
  return HFC_OK;
}

extern "C" int hfc_ssim_grad_maps(const float* x, const float* y, int32_t n, int32_t c, int32_t h0, int32_t w0,
                                  int32_t level, int32_t levels, const float* taps, int32_t win, float c1, float c2,
                                  const float* coeffs, float* maps, int64_t maps_bytes, void* stream) {
  int rc = ssim_check(n, c, h0, w0, win, levels, "ssim_grad_maps");
  if (rc != HFC_OK) return rc;
  if (level < 0 || level >= levels) return set_error(HFC_ERR_INVALID, "ssim_grad_maps: level out of range");
  if (!x || !y || !taps || !coeffs || !maps) return set_error(HFC_ERR_INVALID, "ssim_grad_maps: null pointer");
  if (reinterpret_cast<uintptr_t>(maps) % 16 != 0) return set_error(HFC_ERR_INVALID, "ssim_grad_maps: maps not 16-byte aligned");
  const int64_t planes = static_cast<int64_t>(n) * c;
  SsimLevelArgs a;
  a.g = ssim_level_geom(h0, w0, win, level);
  if (maps_bytes < planes * a.g.ho * a.g.wo * static_cast<int64_t>(sizeof(float4)))
    return set_error(HFC_ERR_INVALID, "ssim_grad_maps: maps buffer too small");
  a.x = x;
  a.y = y;
  a.px = nullptr;
  a.py = nullptr;
  a.taps = taps;
  a.partials = nullptr;
  a.c = c;
  a.win = win;
  a.c1 = c1;
  a.c2 = c2;
  a.coef = coeffs;
  a.maps = reinterpret_cast<float4*>(maps);
  a.level = level;
  a.levels = levels;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = win <= 11 ? launch_ssim_level<11, true>(a, planes, st) : launch_ssim_level<kSsimMaxWin, true>(a, planes, st);
  if (rc != HFC_OK) return rc;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(HFC_ERR_LAUNCH, "ssim_grad_maps launch: %s", cudaGetErrorString(e));
  note_launch();
  return HFC_OK;
}

extern "C" int hfc_ssim_level_bwd(const float* x, const float* y, const float* maps, int32_t n, int32_t c, int32_t h0,
                                  int32_t w0, int32_t level, const float* taps, int32_t win, const float* dx_coarse,
                                  const float* dy_coarse, float* dx, float* dy, void* stream) {
  int rc = ssim_check(n, c, h0, w0, win, level + 1, "ssim_level_bwd");
  if (rc != HFC_OK) return rc;
  if (!x || !y || !maps || !taps) return set_error(HFC_ERR_INVALID, "ssim_level_bwd: null pointer");
  if (reinterpret_cast<uintptr_t>(maps) % 16 != 0)
    return set_error(HFC_ERR_INVALID, "ssim_level_bwd: maps not 16-byte aligned");
  if (!dx && !dy) return HFC_OK;
  const int64_t planes = static_cast<int64_t>(n) * c;
  SsimLevelBwdArgs a;
  a.x = x;
  a.y = y;
  a.maps = reinterpret_cast<const float4*>(maps);
  a.taps = taps;
  a.dx_coarse = dx_coarse;
  a.dy_coarse = dy_coarse;
  a.dx = dx;
  a.dy = dy;
  a.c = c;
  a.win = win;
  a.g = ssim_level_geom(h0, w0, win, level);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = win <= 11 ? launch_ssim_level_bwd<11>(a, planes, st) : launch_ssim_level_bwd<kSsimMaxWin>(a, planes, st);
  if (rc != HFC_OK) return rc;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(HFC_ERR_LAUNCH, "ssim_level_bwd launch: %s", cudaGetErrorString(e));
  note_launch();
  return HFC_OK;
}

extern "C" int64_t hfc_psnr_ws_bytes(int32_t n, int64_t per_image) {
  if (n <= 0 || per_image <= 0) return -1;
  return static_cast<int64_t>(n) * psnr_blocks(per_image) * static_cast<int64_t>(sizeof(double));
}

extern "C" int hfc_psnr(const float* a, const float* b, int32_t n, int64_t per_image, double max_val, void* ws,
                        int64_t ws_bytes, double* out, void* stream) {
  if (!a || !b || !ws || !out || n <= 0 || per_image <= 0)
    return set_error(HFC_ERR_INVALID, "psnr: null pointer or empty input");
  if (n > 65535) return set_error(HFC_ERR_UNSUPPORTED, "psnr: more than 65535 images");
  const int blocks = psnr_blocks(per_image);
  if (ws_bytes < static_cast<int64_t>(n) * blocks * static_cast<int64_t>(sizeof(double)))
    return set_error(HFC_ERR_INVALID, "psnr: workspace too small");
  int sms = 0;
  int rc = device_sm_count(&sms);
  if (rc != HFC_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  double* partials = static_cast<double*>(ws);
  psnr_partial_kernel<<<dim3(blocks, n), kPsnrThreads, 0, st>>>(a, b, per_image, partials);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(HFC_ERR_LAUNCH, "psnr launch: %s", cudaGetErrorString(e));
  note_launch();
  psnr_finalize_kernel<<<(n + 127) / 128, 128, 0, st>>>(partials, n, blocks, per_image, max_val, out);
  e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(HFC_ERR_LAUNCH, "psnr finalize launch: %s", cudaGetErrorString(e));
  note_launch();
  return HFC_OK;
}
