// TEST INFRASTRUCTURE: runs the per-CTA work of csrc/ssim.cu on the host with the functions the kernels call
// (csrc/ssim_math.cuh, compiled here with g++): the tile grid, the staged region with its zero padding, the filter taps,
// the per-pixel ssim / cs, the 2x2 pooling and its ownership, and the per-plane finalisation (tests/test_metrics_cpu.py).
// Not covered: the kernels' register blocking (it applies the same taps in the same order) and their in-CTA reductions.
#include <vector>

#include "../high-fidelity-generative-compression_b200/csrc/ssim_math.cuh"

using namespace hfc;

// One level over all planes.  partials[(plane * tiles + tile) * 2 + {0, 1}] = the tile's sums of (ssim, cs);
// out_cover / pool_cover count how often each valid output / pooled pixel is produced (each must be exactly 1).
extern "C" void ssim_level_host(const float* x, const float* y, int planes, int c, int h0, int w0, int level,
                                const float* taps, int win, float c1, float c2, float* px, float* py, double* partials,
                                int* out_cover, int* pool_cover) {
  const SsimLevelGeom g = ssim_level_geom(h0, w0, win, level);
  const int SR = ssim_stage_rows(g), SC = ssim_stage_cols(g), VC = kSsimTileW + g.ww - 1;
  const int64_t tiles = ssim_level_tiles(g);
  std::vector<float> st[5], sv[5];
  for (int m = 0; m < 5; ++m) {
    st[m].resize(static_cast<size_t>(SR) * SC);
    sv[m].resize(static_cast<size_t>(kSsimTileH) * VC);
  }
  const float one = 1.f;
  for (int64_t p = 0; p < planes; ++p) {
    const float* tv = g.wh == 1 ? &one : taps + (p % c) * win;
    const float* th = g.ww == 1 ? &one : taps + (p % c) * win;
    const int64_t base = p * static_cast<int64_t>(g.h) * g.w;
    for (int64_t tile = 0; tile < tiles; ++tile) {
      const int ty = static_cast<int>(tile / g.tiles_x), tx = static_cast<int>(tile % g.tiles_x);
      const int r0 = ty * kSsimTileH, c0 = tx * kSsimTileW;
      for (int rr = 0; rr < SR; ++rr)
        for (int cc = 0; cc < SC; ++cc) {
          const int gr = r0 - 1 + rr, gc = c0 - 1 + cc;
          const bool in = gr >= 0 && gr < g.h && gc >= 0 && gc < g.w;
          const float xv = in ? x[base + static_cast<int64_t>(gr) * g.w + gc] : 0.f;
          const float yv = in ? y[base + static_cast<int64_t>(gr) * g.w + gc] : 0.f;
          const int s = rr * SC + cc;
          st[0][s] = xv;
          st[1][s] = yv;
          st[2][s] = mul_rn(xv, xv);
          st[3][s] = mul_rn(yv, yv);
          st[4][s] = mul_rn(xv, yv);
        }
      for (int m = 0; m < 5; ++m)
        for (int i = 0; i < kSsimTileH; ++i)
          for (int j = 0; j < VC; ++j) sv[m][i * VC + j] = filter_taps(&st[m][(i + 1) * SC + j + 1], SC, tv, g.wh);
      double s_sum = 0.0, c_sum = 0.0;
      for (int i = 0; i < kSsimTileH; ++i)
        for (int j = 0; j < kSsimTileW; ++j) {
          const int oi = r0 + i, oj = c0 + j;
          if (oi >= g.ho || oj >= g.wo) continue;
          float mo[5];
          for (int m = 0; m < 5; ++m) mo[m] = filter_taps(&sv[m][i * VC + j], 1, th, g.ww);
          float s, cs;
          ssim_from_moments(mo[0], mo[1], mo[2], mo[3], mo[4], c1, c2, &s, &cs);
          s_sum += s;
          c_sum += cs;
          ++out_cover[(p * g.ho + oi) * g.wo + oj];
        }
      partials[(p * tiles + tile) * 2] = s_sum;
      partials[(p * tiles + tile) * 2 + 1] = c_sum;
      if (!px) continue;
      for (int pi = 0; pi < kSsimTileH / 2; ++pi)
        for (int pj = 0; pj < kSsimTileW / 2; ++pj) {
          const int gpi = ty * (kSsimTileH / 2) + pi, gpj = tx * (kSsimTileW / 2) + pj;
          if (gpi >= g.hp || gpj >= g.wp) continue;
          const int s = pooled_stage_index(pi, g.h & 1) * SC + pooled_stage_index(pj, g.w & 1);
          const int64_t o = (p * g.hp + gpi) * static_cast<int64_t>(g.wp) + gpj;
          px[o] = pool4(st[0][s], st[0][s + 1], st[0][s + SC], st[0][s + SC + 1]);
          py[o] = pool4(st[1][s], st[1][s + 1], st[1][s + SC], st[1][s + SC + 1]);
          ++pool_cover[o];
        }
    }
  }
}

extern "C" void ssim_level_geom_host(int h0, int w0, int win, int level, int* out) {
  const SsimLevelGeom g = ssim_level_geom(h0, w0, win, level);
  const int v[] = {g.h, g.w, g.wh, g.ww, g.ho, g.wo, g.hp, g.wp, g.tiles_y, g.tiles_x};
  for (int i = 0; i < 10; ++i) out[i] = v[i];
}

// sums: [levels][2] per plane (the finalize kernel's per-plane sums)
extern "C" float ssim_plane_value_host(const double* sums, const float* weights, int levels, int h0, int w0, int win,
                                       int relu_last) {
  return ssim_plane_value(sums, weights, levels, h0, w0, win, relu_last);
}
