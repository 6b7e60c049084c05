// Per-pixel, per-pooled-pixel and per-plane code of the SSIM / MS-SSIM kernels (csrc/ssim.cu).  Shared by the CUDA kernels
// and by the host harness tests/ssim_math_host.cpp, which compiles THIS file with g++ so that the arithmetic, the tiling and
// the pooling ownership the GPU runs are checked on the CPU.  Reference: src/helpers/metrics.py:37-63 (gaussian_filter),
// 66-103 (_ssim), 164-236 (ms_ssim).
//
// Every rounding step is explicit (mul_rn / add_rn / fmaf), so nvcc's FMA contraction cannot make the device differ from
// the host build: both produce the same bits for every filtered moment, pooled pixel and per-pixel ssim / cs value.
#pragma once
#include <math.h>
#include <stdint.h>

#ifdef __CUDACC__
#define HFC_HD __host__ __device__ __forceinline__
#else
#define HFC_HD inline
#endif

namespace hfc {

constexpr int kSsimTileH = 32;        // valid outputs per CTA (rows x cols); the pooled tile is half of it each way
constexpr int kSsimTileW = 64;
constexpr int kSsimMaxWin = 31;       // largest window the level kernel is instantiated for
constexpr int kSsimMaxLevels = 8;

HFC_HD float mul_rn(float a, float b) {
#ifdef __CUDA_ARCH__
  return __fmul_rn(a, b);
#else
  return a * b;
#endif
}
HFC_HD float add_rn(float a, float b) {
#ifdef __CUDA_ARCH__
  return __fadd_rn(a, b);
#else
  return a + b;
#endif
}
HFC_HD float sub_rn(float a, float b) {
#ifdef __CUDA_ARCH__
  return __fsub_rn(a, b);
#else
  return a - b;
#endif
}
HFC_HD float div_rn(float a, float b) {
#ifdef __CUDA_ARCH__
  return __fdiv_rn(a, b);
#else
  return a / b;
#endif
}

// Geometry of one level.  A spatial size smaller than the window is not smoothed along that dimension (the reference's
// gaussian_filter skips it with a warning): its window is then one tap of 1.0, which is an exact identity.
struct SsimLevelGeom {
  int h, w;            // input plane
  int wh, ww;          // window length along h / w (win, or 1 when skipped)
  int ho, wo;          // valid outputs
  int hp, wp;          // 2x2 average-pooled plane (padding h % 2, w % 2)
  int tiles_y, tiles_x;
};

HFC_HD int pooled_size(int s) { return (s + 1) / 2; }   // avg_pool2d(kernel 2, stride 2, padding s % 2)

HFC_HD int ceil_div(int a, int b) { return (a + b - 1) / b; }

HFC_HD SsimLevelGeom ssim_level_geom(int h0, int w0, int win, int level) {
  SsimLevelGeom g;
  g.h = h0;
  g.w = w0;
  for (int l = 0; l < level; ++l) {
    g.h = pooled_size(g.h);
    g.w = pooled_size(g.w);
  }
  g.wh = g.h >= win ? win : 1;
  g.ww = g.w >= win ? win : 1;
  g.ho = g.h - g.wh + 1;
  g.wo = g.w - g.ww + 1;
  g.hp = pooled_size(g.h);
  g.wp = pooled_size(g.w);
  // One CTA owns output tile (ty, tx) AND pooled tile (ty, tx); the grid covers whichever of the two needs more tiles.
  const int ty_s = ceil_div(g.ho, kSsimTileH), ty_p = ceil_div(g.hp, kSsimTileH / 2);
  const int tx_s = ceil_div(g.wo, kSsimTileW), tx_p = ceil_div(g.wp, kSsimTileW / 2);
  g.tiles_y = ty_s > ty_p ? ty_s : ty_p;
  g.tiles_x = tx_s > tx_p ? tx_s : tx_p;
  return g;
}

HFC_HD int64_t ssim_level_tiles(const SsimLevelGeom& g) { return static_cast<int64_t>(g.tiles_y) * g.tiles_x; }

// Workspace (in doubles): per level, [planes][tiles][2] partial sums (ssim, cs), then [planes][levels][2] per-plane sums,
// then [planes] per-plane values.  `ssim_partials_offset(..., level)` is where level `level`'s partials start.
HFC_HD int64_t ssim_partials_offset(int64_t planes, int h0, int w0, int win, int level) {
  int64_t off = 0;
  for (int l = 0; l < level; ++l) off += planes * ssim_level_tiles(ssim_level_geom(h0, w0, win, l)) * 2;
  return off;
}
HFC_HD int64_t ssim_ws_doubles(int64_t planes, int h0, int w0, int win, int levels) {
  return ssim_partials_offset(planes, h0, w0, win, levels) + planes * levels * 2 + planes;
}

// The input region a CTA stages: rows [r0 - 1, r0 + TH + wh - 1), cols [c0 - 1, c0 + TW + ww - 1), zero outside the
// plane.  Staged row k is input row r0 - 1 + k: the extra leading row / column is the top / left zero padding of an odd
// dimension's pooling.
HFC_HD int ssim_stage_rows(const SsimLevelGeom& g) { return kSsimTileH + g.wh; }
HFC_HD int ssim_stage_cols(const SsimLevelGeom& g) { return kSsimTileW + g.ww; }

// Pooled pixel (pi, pj) of a tile (tile-local) reads staged rows / cols sr, sr + 1 and sc, sc + 1.  Its input row is
// 2 * (ty * TH/2 + pi) - (h % 2) = r0 + 2 pi - (h % 2), i.e. staged row 2 pi + 1 - (h % 2).
HFC_HD int pooled_stage_index(int p_local, int odd) { return 2 * p_local + 1 - odd; }

// F.avg_pool2d(kernel 2, count_include_pad=True): ((x00 + x01) + x10) + x11, divided by 4 (exact: a power of two)
HFC_HD float pool4(float x00, float x01, float x10, float x11) {
  return mul_rn(add_rn(add_rn(add_rn(x00, x01), x10), x11), 0.25f);
}

// The five filtered moments of one output pixel -> (ssim, cs), the reference's expressions in its fp32 rounding order:
//   cs = (2 s12 + C2) / (s1 + s2 + C2),  ssim = ((2 mu1 mu2 + C1) / (mu1^2 + mu2^2 + C1)) * cs
HFC_HD void ssim_from_moments(float mu1, float mu2, float exx, float eyy, float exy, float c1, float c2, float* ssim,
                              float* cs) {
  const float mu1_sq = mul_rn(mu1, mu1), mu2_sq = mul_rn(mu2, mu2), mu1_mu2 = mul_rn(mu1, mu2);
  const float s1 = sub_rn(exx, mu1_sq), s2 = sub_rn(eyy, mu2_sq), s12 = sub_rn(exy, mu1_mu2);
  const float c = div_rn(add_rn(mul_rn(2.f, s12), c2), add_rn(add_rn(s1, s2), c2));
  const float l = div_rn(add_rn(mul_rn(2.f, mu1_mu2), c1), add_rn(add_rn(mu1_sq, mu2_sq), c1));
  *cs = c;
  *ssim = mul_rn(l, c);
}

// One filter tap after another, starting from 0: acc = fma(w[k], v[k], acc) for k = 0 .. n-1.  The kernel's register
// blocking performs exactly this sequence for every output.
HFC_HD float filter_taps(const float* v, int64_t stride, const float* taps, int n) {
  float acc = 0.f;
  for (int k = 0; k < n; ++k) acc = fmaf(taps[k], v[k * stride], acc);
  return acc;
}

HFC_HD float relu_keep_nan(float v) { return v < 0.f ? 0.f : v; }   // torch.relu: NaN stays NaN

// One plane's final value from its per-level sums (sums[2 l] = sum of ssim, sums[2 l + 1] = sum of cs over the level's
// valid outputs): mean per level in double, rounded to fp32 like the reference's fp32 mean; relu(cs) below the last level,
// relu(ssim) at the last level when relu_last; then prod_l value_l ** weight_l in fp32, level after level.
HFC_HD float ssim_plane_value(const double* sums, const float* weights, int levels, int h0, int w0, int win,
                              int relu_last) {
  float prod = 1.f;
  for (int l = 0; l < levels; ++l) {
    const SsimLevelGeom g = ssim_level_geom(h0, w0, win, l);
    const double count = static_cast<double>(g.ho) * g.wo;
    const bool last = l == levels - 1;
    float v = static_cast<float>(sums[2 * l + (last ? 0 : 1)] / count);
    if (!last || relu_last) v = relu_keep_nan(v);
    const float f = weights[l] == 1.f ? v : powf(v, weights[l]);
    prod = l == 0 ? f : mul_rn(prod, f);
  }
  return prod;
}

}  // namespace hfc
