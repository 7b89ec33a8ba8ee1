// Host-only check of the proto.up -> proto.cv2 weight merge (conv_tma.cuh merge_upconv_weights; no GPU needed):
//   nvcc -std=c++17 -gencode arch=compute_100a,code=sm_100a --expt-relaxed-constexpr -o /tmp/merge_check tools/merge_check.cu -lcuda
//   /tmp/merge_check pack.xrsw [seed]
// Reads the n-scale weight pack, merges the two layers in fp64 and evaluates both forms on a random 80x80x64 map in fp64:
// cv2(convT(x)) directly (the ConvTranspose, then the zero-padded 3x3 on the 160x160 map, no activation) against the four
// parity convolutions with the merged weights and border biases.  Prints one line of key=value pairs: the largest error
// relative to the largest output, the same per border class, max |Wm|, and the relative error of Wm rounded to fp16 once.
#include <math.h>

#include <fstream>
#include <iterator>
#include <random>

#include "../xr_image_segmentation_b200/csrc/conv_tma.cuh"
#include "../xr_image_segmentation_b200/csrc/model.cuh"
using namespace xrseg;

int main(int argc, char** argv) {
  if (argc < 2) { fprintf(stderr, "usage: merge_check pack.xrsw [seed]\n"); return 2; }
  std::ifstream f(argv[1], std::ios::binary);
  std::vector<char> data((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  const unsigned seed = argc > 2 ? static_cast<unsigned>(atoi(argv[2])) : 0u;
  Net net('n', 1);
  std::vector<HostLayerWeights> hw;
  xrsw_load(data.data(), data.size(), net.layers, 'n', hw);
  int iu = -1, i2 = -1;
  for (size_t i = 0; i < net.layers.size(); ++i) {
    if (net.layers[i].name == "proto.up") iu = static_cast<int>(i);
    if (net.layers[i].name == "proto.cv2") i2 = static_cast<int>(i);
  }
  if (iu < 0 || i2 < 0) { fprintf(stderr, "layers not found\n"); return 1; }
  const int C = 64, H = 80, W = 80, Ho = 160, Wo = 160;
  const float *wt = hw[iu].w.data(), *bt = hw[iu].b.data(), *w2 = hw[i2].w.data(), *b2 = hw[i2].b.data();
  std::vector<double> wm, bm;
  merge_upconv_weights(wt, bt, w2, b2, C, C, C, wm, bm);

  std::mt19937 rng(seed);
  std::normal_distribution<double> nd(0.0, 1.0);
  std::vector<double> x(static_cast<size_t>(H) * W * C);
  for (double& v : x) v = nd(rng);
  // direct: u = convT(x) + bt on 160x160, z = conv3x3(u) + b2 with zero padding
  std::vector<double> u(static_cast<size_t>(Ho) * Wo * C), z(static_cast<size_t>(Ho) * Wo * C), zm(z.size());
  for (int oy = 0; oy < Ho; ++oy)
    for (int ox = 0; ox < Wo; ++ox)
      for (int c = 0; c < C; ++c) {
        double s = bt[c];
        const int y = oy / 2, xx = ox / 2, a = oy % 2, b = ox % 2;
        for (int i = 0; i < C; ++i) s += x[(static_cast<size_t>(y) * W + xx) * C + i] * wt[((static_cast<size_t>(i) * C + c) * 2 + a) * 2 + b];
        u[(static_cast<size_t>(oy) * Wo + ox) * C + c] = s;
      }
  for (int oy = 0; oy < Ho; ++oy)
    for (int ox = 0; ox < Wo; ++ox)
      for (int o = 0; o < C; ++o) {
        double s = b2[o];
        for (int kh = 0; kh < 3; ++kh)
          for (int kw = 0; kw < 3; ++kw) {
            const int iy = oy + kh - 1, ix = ox + kw - 1;
            if (iy < 0 || iy >= Ho || ix < 0 || ix >= Wo) continue;
            const double* up = &u[(static_cast<size_t>(iy) * Wo + ix) * C];
            for (int c = 0; c < C; ++c) s += w2[(static_cast<size_t>(o) * C + c) * 9 + kh * 3 + kw] * up[c];
          }
        z[(static_cast<size_t>(oy) * Wo + ox) * C + o] = s;
      }
  // merged: parity (dy, dx) of output (2y + dy, 2x + dx) reads input (y + dy + th - 1, x + dx + tw - 1)
  for (int oy = 0; oy < Ho; ++oy)
    for (int ox = 0; ox < Wo; ++ox) {
      const int dy = oy & 1, dx = ox & 1, y = oy >> 1, xx = ox >> 1;
      const int cls = 3 * (oy == 0 ? 1 : (oy == Ho - 1 ? 2 : 0)) + (ox == 0 ? 1 : (ox == Wo - 1 ? 2 : 0));
      for (int o = 0; o < C; ++o) {
        double s = bm[o] + (cls ? bm[static_cast<size_t>(C) * (1 + cls) + o] : 0.0);
        for (int th = 0; th < 2; ++th)
          for (int tw = 0; tw < 2; ++tw) {
            const int iy = y + dy + th - 1, ix = xx + dx + tw - 1;
            if (iy < 0 || iy >= H || ix < 0 || ix >= W) continue;
            const double* wr = &wm[((static_cast<size_t>(((dy * 2 + dx) * 2 + th) * 2 + tw)) * C + o) * C];
            const double* xp = &x[(static_cast<size_t>(iy) * W + ix) * C];
            for (int i = 0; i < C; ++i) s += wr[i] * xp[i];
          }
        zm[(static_cast<size_t>(oy) * Wo + ox) * C + o] = s;
      }
    }
  double zmax = 0, err = 0, cls_err[9] = {0};
  int cls_n[9] = {0};
  for (int oy = 0; oy < Ho; ++oy)
    for (int ox = 0; ox < Wo; ++ox) {
      const int cls = 3 * (oy == 0 ? 1 : (oy == Ho - 1 ? 2 : 0)) + (ox == 0 ? 1 : (ox == Wo - 1 ? 2 : 0));
      ++cls_n[cls];
      for (int o = 0; o < C; ++o) {
        const size_t k = (static_cast<size_t>(oy) * Wo + ox) * C + o;
        zmax = fmax(zmax, fabs(z[k]));
        const double e = fabs(z[k] - zm[k]);
        err = fmax(err, e);
        cls_err[cls] = fmax(cls_err[cls], e);
      }
    }
  double wmax = 0, werr = 0;
  for (double v : wm) {
    wmax = fmax(wmax, fabs(v));
    werr = fmax(werr, fabs(static_cast<double>(__half2float(__double2half(v))) - v));
  }
  printf("rel_err %.3e out_max %.6g wm_max %.6g wm_f16_rel_err %.3e", err / zmax, zmax, wmax, werr / wmax);
  for (int c = 0; c < 9; ++c) printf(" cls%d %.3e n%d %d", c, cls_err[c] / zmax, c, cls_n[c]);
  printf("\n");
  return 0;
}
