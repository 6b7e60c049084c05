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
};

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

template <int MAXW>
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
    if (r0 + i < g.ho) {
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

template <int MAXW>
static int launch_ssim_level(const SsimLevelArgs& a, int64_t planes, cudaStream_t st) {
  const size_t smem = ssim_smem_bytes(a.g);
  SsimLevelGeom big{};                 // the largest window's requirement (host-side attribute, no synchronisation)
  big.wh = big.ww = MAXW;
  cudaError_t e = cudaFuncSetAttribute(ssim_level_kernel<MAXW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       static_cast<int>(ssim_smem_bytes(big)));
  if (e != cudaSuccess) return set_error(HFC_ERR_LAUNCH, "ssim_level: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  dim3 grid(static_cast<unsigned>(ssim_level_tiles(a.g)), static_cast<unsigned>(planes));
  ssim_level_kernel<MAXW><<<grid, kSsimThreads, smem, st>>>(a);
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
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  rc = win <= 11 ? launch_ssim_level<11>(a, planes, st) : launch_ssim_level<kSsimMaxWin>(a, planes, st);
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
