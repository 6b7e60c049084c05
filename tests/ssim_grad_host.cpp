// TEST INFRASTRUCTURE: runs the backward of csrc/ssim.cu on the host with the functions its kernels call
// (csrc/ssim_math.cuh, compiled here with g++): the pooled pyramid, the per-plane level sums, the coefficients, the four
// gradient maps per valid output, and the level-backward tiles (staged maps with their zero halo, the adjoint window with
// flipped taps, the combine step and the pooled gradient of the next level), coarsest level first
// (tests/test_metrics_grad_cpu.py).  Not covered: the kernels' register blocking (it applies the same taps in the same
// order) and their in-CTA reductions of the forward sums (summed here in another order).
#include <vector>

#include "../high-fidelity-generative-compression_b200/csrc/ssim_math.cuh"

using namespace hfc;

namespace {

// The five filtered moments of every valid output of one plane, vertical pass first (the forward's order).
void plane_moments(const float* x, const float* y, const SsimLevelGeom& g, const float* tv, const float* th,
                   std::vector<float> mo[5]) {
  std::vector<float> p[5], v[5];
  const size_t hw = static_cast<size_t>(g.h) * g.w;
  for (int m = 0; m < 5; ++m) {
    p[m].resize(hw);
    v[m].resize(static_cast<size_t>(g.ho) * g.w);
    mo[m].assign(static_cast<size_t>(g.ho) * g.wo, 0.f);
  }
  for (size_t i = 0; i < hw; ++i) {
    p[0][i] = x[i];
    p[1][i] = y[i];
    p[2][i] = mul_rn(x[i], x[i]);
    p[3][i] = mul_rn(y[i], y[i]);
    p[4][i] = mul_rn(x[i], y[i]);
  }
  for (int m = 0; m < 5; ++m) {
    for (int i = 0; i < g.ho; ++i)
      for (int j = 0; j < g.w; ++j) v[m][i * g.w + j] = filter_taps(&p[m][i * g.w + j], g.w, tv, g.wh);
    for (int i = 0; i < g.ho; ++i)
      for (int j = 0; j < g.wo; ++j) mo[m][i * g.wo + j] = filter_taps(&v[m][i * g.w + j], 1, th, g.ww);
  }
}

float at(const float* p, int h, int w, int r, int c) { return r >= 0 && r < h && c >= 0 && c < w ? p[r * w + c] : 0.f; }

}  // namespace

// Whole backward of one call over all planes.  x, y: (planes, h0, w0); grad_out: [1] (size_average) or [planes / c];
// dx, dy: (planes, h0, w0) outputs.  cover[l] (planes * h_l * w_l ints each, laid out level after level) counts how
// often a level-backward tile writes each input pixel of level l (each must be exactly 1).
extern "C" void ssim_grad_host(const float* x, const float* y, int planes, int c, int h0, int w0, int levels,
                               const float* taps, int win, float c1, float c2, const float* weights, int relu_last,
                               int size_average, const float* grad_out, float* dx, float* dy, int* cover) {
  std::vector<std::vector<float>> px(levels), py(levels), gx(levels), gy(levels);
  std::vector<SsimLevelGeom> geo(levels);
  for (int l = 0; l < levels; ++l) geo[l] = ssim_level_geom(h0, w0, win, l);
  px[0].assign(x, x + static_cast<size_t>(planes) * h0 * w0);
  py[0].assign(y, y + static_cast<size_t>(planes) * h0 * w0);
  for (int l = 0; l + 1 < levels; ++l) {                       // the forward's pooled pyramid
    const SsimLevelGeom& g = geo[l];
    px[l + 1].resize(static_cast<size_t>(planes) * g.hp * g.wp);
    py[l + 1].resize(px[l + 1].size());
    for (int p = 0; p < planes; ++p)
      for (int i = 0; i < g.hp; ++i)
        for (int j = 0; j < g.wp; ++j) {
          const int r = 2 * i - (g.h & 1), cc = 2 * j - (g.w & 1);
          const float* a = &px[l][static_cast<size_t>(p) * g.h * g.w];
          const float* b = &py[l][static_cast<size_t>(p) * g.h * g.w];
          const size_t o = (static_cast<size_t>(p) * g.hp + i) * g.wp + j;
          px[l + 1][o] = pool4(at(a, g.h, g.w, r, cc), at(a, g.h, g.w, r, cc + 1), at(a, g.h, g.w, r + 1, cc),
                               at(a, g.h, g.w, r + 1, cc + 1));
          py[l + 1][o] = pool4(at(b, g.h, g.w, r, cc), at(b, g.h, g.w, r, cc + 1), at(b, g.h, g.w, r + 1, cc),
                               at(b, g.h, g.w, r + 1, cc + 1));
        }
  }
  const float one = 1.f;
  std::vector<double> sums(static_cast<size_t>(planes) * levels * 2);
  std::vector<std::vector<float>> moments(static_cast<size_t>(planes) * levels * 5);
  for (int p = 0; p < planes; ++p)
    for (int l = 0; l < levels; ++l) {
      const SsimLevelGeom& g = geo[l];
      const float* tv = g.wh == 1 ? &one : taps + (p % c) * win;
      const float* th = g.ww == 1 ? &one : taps + (p % c) * win;
      std::vector<float>* mo = &moments[(static_cast<size_t>(p) * levels + l) * 5];
      const size_t off = static_cast<size_t>(p) * g.h * g.w;
      plane_moments(&px[l][off], &py[l][off], g, tv, th, mo);
      double s = 0.0, cs = 0.0;
      for (size_t o = 0; o < mo[0].size(); ++o) {
        float sv, cv;
        ssim_from_moments(mo[0][o], mo[1][o], mo[2][o], mo[3][o], mo[4][o], c1, c2, &sv, &cv);
        s += sv;
        cs += cv;
      }
      sums[(static_cast<size_t>(p) * levels + l) * 2] = s;
      sums[(static_cast<size_t>(p) * levels + l) * 2 + 1] = cs;
    }
  std::vector<float> coef(static_cast<size_t>(planes) * levels * 2);
  for (int p = 0; p < planes; ++p)
    ssim_grad_coeffs(&sums[static_cast<size_t>(p) * levels * 2], weights, levels, h0, w0, win, relu_last,
                     ssim_grad_dv(grad_out, p, planes, c, size_average), &coef[static_cast<size_t>(p) * levels * 2]);

  int* cov = cover;
  std::vector<int*> cover_of(levels);
  for (int l = 0; l < levels; ++l) {
    cover_of[l] = cov;
    cov += static_cast<size_t>(planes) * geo[l].h * geo[l].w;
  }
  for (int l = levels - 1; l >= 0; --l) {
    const SsimLevelGeom& g = geo[l];
    gx[l].assign(static_cast<size_t>(planes) * g.h * g.w, 0.f);
    gy[l].assign(gx[l].size(), 0.f);
    const int SR = ssim_bwd_stage_rows(g), SC = ssim_bwd_stage_cols(g);
    std::vector<float> st[4], sv[4];
    for (int m = 0; m < 4; ++m) {
      st[m].resize(static_cast<size_t>(SR) * SC);
      sv[m].resize(static_cast<size_t>(kSsimTileH) * SC);
    }
    for (int p = 0; p < planes; ++p) {
      float flipped[2][kSsimMaxWin];
      for (int k = 0; k < win; ++k) flipped[0][k] = flipped[1][k] = taps[(p % c) * win + (win - 1 - k)];
      const float* tv = g.wh == 1 ? &one : flipped[0];
      const float* th = g.ww == 1 ? &one : flipped[1];
      // the four maps of this plane and level (the grad-maps kernel's per-output work)
      const std::vector<float>* mo = &moments[(static_cast<size_t>(p) * levels + l) * 5];
      const float alpha = coef[(static_cast<size_t>(p) * levels + l) * 2];
      const float beta = coef[(static_cast<size_t>(p) * levels + l) * 2 + 1];
      std::vector<float> maps[4];
      for (int m = 0; m < 4; ++m) maps[m].resize(mo[0].size());
      for (size_t o = 0; o < mo[0].size(); ++o)
        ssim_grad_maps(mo[0][o], mo[1][o], mo[2][o], mo[3][o], mo[4][o], c1, c2, alpha, beta, &maps[0][o], &maps[1][o],
                       &maps[2][o], &maps[3][o]);
      const size_t off = static_cast<size_t>(p) * g.h * g.w;
      for (int ty = 0; ty < ssim_bwd_tiles_y(g); ++ty)
        for (int tx = 0; tx < ssim_bwd_tiles_x(g); ++tx) {
          const int r0 = ty * kSsimTileH, c0 = tx * kSsimTileW;
          for (int rr = 0; rr < SR; ++rr)
            for (int cc = 0; cc < SC; ++cc)
              for (int m = 0; m < 4; ++m)
                st[m][rr * SC + cc] = at(maps[m].data(), g.ho, g.wo, r0 - (g.wh - 1) + rr, c0 - (g.ww - 1) + cc);
          for (int m = 0; m < 4; ++m)
            for (int i = 0; i < kSsimTileH; ++i)
              for (int j = 0; j < SC; ++j) sv[m][i * SC + j] = filter_taps(&st[m][i * SC + j], SC, tv, g.wh);
          for (int i = 0; i < kSsimTileH; ++i)
            for (int j = 0; j < kSsimTileW; ++j) {
              const int gi = r0 + i, gj = c0 + j;
              if (gi >= g.h || gj >= g.w) continue;
              float t[4];
              for (int m = 0; m < 4; ++m) t[m] = filter_taps(&sv[m][i * SC + j], 1, th, g.ww);
              const size_t o = off + static_cast<size_t>(gi) * g.w + gj;
              float cx = 0.f, cy = 0.f;
              if (l + 1 < levels) {
                const size_t po = (static_cast<size_t>(p) * g.hp + pooled_index_of(gi, g.h & 1)) * g.wp +
                                  pooled_index_of(gj, g.w & 1);
                cx = gx[l + 1][po];
                cy = gy[l + 1][po];
              }
              gx[l][o] = ssim_grad_combine(t[0], t[2], t[3], px[l][o], py[l][o], cx);
              gy[l][o] = ssim_grad_combine(t[1], t[2], t[3], py[l][o], px[l][o], cy);
              ++cover_of[l][o];
            }
        }
    }
  }
  for (size_t i = 0; i < gx[0].size(); ++i) {
    dx[i] = gx[0][i];
    dy[i] = gy[0][i];
  }
}
