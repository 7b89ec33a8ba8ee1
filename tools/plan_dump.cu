// Host-only developer tool: prints the launch plan of every convolution of the network (no GPU needed).
//   nvcc -std=c++17 -gencode arch=compute_100a,code=sm_100a --expt-relaxed-constexpr -o /tmp/plan_dump tools/plan_dump.cu -lcuda
//   /tmp/plan_dump [batch] [n|s] [ops] [up] [num_classes]
//   up: the runner's launch list, with proto.up merged into proto.cv2's launch (model.cuh fuse_up_conv)
//   The launch list follows the fusion switches the runner reads at create time: XRSEG_FUSE, XRSEG_FUSE_BNECK (read here as
//   xrseg_create reads them), XRSEG_FUSE_PE, XRSEG_FUSE_TAIL and XRSEG_FUSE_UP (read by model.cuh itself).
#include <math.h>
#include <string.h>
#include "../xr_image_segmentation_b200/csrc/conv_tma.cuh"
#include "../xr_image_segmentation_b200/csrc/model.cuh"
using namespace xrseg;
int main(int argc, char** argv) {
  const int B = argc > 1 ? atoi(argv[1]) : 64;
  const int scale = argc > 2 ? argv[2][0] : 'n';
  bool ops = false, up = false;
  int nc = 80;
  for (int i = 3; i < argc; ++i) {
    if (argv[i][0] == 'o') ops = true;
    else if (strcmp(argv[i], "up") == 0) up = true;
    else nc = atoi(argv[i]);
  }
  if (ops) {   // "ops": the fused launch list (one line per network launch) instead of the conv plans
    const char* fuse_env = getenv("XRSEG_FUSE");
    const char* bneck_env = getenv("XRSEG_FUSE_BNECK");
    Net fused(scale, B, 640, !(fuse_env && fuse_env[0] == '0'), !(bneck_env && bneck_env[0] == '0'), nc, up);
    const char* kind_name[] = {"stem", "conv", "dw", "sppf", "up", "attn", "bneck"};
    for (const Op& o : fused.ops) {
      std::string name = o.layer >= 0 ? fused.layers[o.layer].name : std::string("-");
      if (o.kind == OP_CONV && o.layer2 >= 0) name += "+" + fused.layers[o.layer2].name;
      printf("op %-6s %-28s in %3dx%-3d c%-3d out c%-3d res %d branch %d\n", kind_name[o.kind], name.c_str(), o.x.H, o.x.W, o.x.Cp,
             o.y.Cp, o.has_res ? 1 : 0, o.branch);
      if (o.kind == OP_CONV && o.up_layer >= 0) printf("   (merged: %s runs inside this launch)\n", fused.layers[o.up_layer].name.c_str());
      if (o.kind == OP_CONV && o.tail_layer >= 0) printf("   (tail: %s runs inside this launch)\n", fused.layers[o.tail_layer].name.c_str());
    }
    return 0;
  }
  Net net(scale, B, 640, true, false, nc, up);   // Bottleneck fusion off: every convolution keeps its own plan
  const char* mode_name[] = {"gather", "halo", "halo_tma", "flat_tma", "s2_tma"};
  long total_smem_small = 0;
  for (const Op& o : net.ops) {
    if (o.kind != OP_CONV) continue;
    const LayerRec& l = net.layers[o.layer];
    ConvDesc cd{};
    cd.B = B; cd.H = o.x.H; cd.W = o.x.W; cd.Cin = o.x.Cp; cd.in_pitch = o.x.pitch; cd.Cout = o.y.Cp + (o.layer2 >= 0 ? o.y2.Cp : 0); cd.out_pitch = o.y.pitch;
    cd.k = o.k; cd.stride = o.stride; cd.act = o.act; cd.transposed = o.transposed; cd.res_pitch = o.has_res ? o.res.pitch : 0;
    cd.upm = o.up_layer >= 0 ? 1 : 0;
    ConvParams p;
    if (!plan_conv_halo_tma(cd, 148, p) && !plan_conv_flat_tma(cd, 148, p) && !plan_conv_s2_tma(cd, 148, p)) p = plan_conv(cd, 148, 0);
    const int work = p.m_tiles * p.n_tiles;
    printf("%-16s %3dx%-3d %3d->%-3d k%d s%d %-8s cb %2d kps %d nks %2d R %2d nsub %d S %d smem %6d tmem %3d items %5d (%.1f/CTA) bres %d",
           (o.layer2 >= 0 ? l.name + "+" : l.name).c_str(), o.x.H, o.x.W, l.cin,
           l.cout + (o.layer2 >= 0 ? net.layers[o.layer2].cout : 0), o.k, o.stride, mode_name[p.mode], p.cb, p.kps, p.nks, p.R, p.nsub, p.S,
           p.smem_bytes, p.tmem_cols, work, static_cast<double>(work) / p.grid, p.b_resident);
    {
      // estimated per-CTA time of the three engines, in us at 1.9 GHz: TMA = 1.5 cycles per box row (tools/probe_tma_rate.cu),
      // tensor = 128 x N x 16 MACs per MMA at 4096 MACs / cycle, HBM = algorithmic bytes at 6.5 TB/s over the whole chip
      const int kps = p.kps > 1 ? p.kps : 1;
      const double rows_item = p.mode == MODE_FLAT_TMA ? static_cast<double>(p.slots) * kps * p.nks
                               : p.mode == MODE_S2_TMA ? (p.pair ? 2.0 : 4.0) * p.slots * p.nks : static_cast<double>(p.slots) * p.nks;
      const double per_cta = ceil(static_cast<double>(work) / p.grid);
      const double tma_us = rows_item * 1.5 * per_cta / 1900.0;
      const double mma_item = static_cast<double>(p.nsub) * (p.upm ? p.taps / 2 : p.taps) * (p.mode == MODE_FLAT_TMA ? kps * p.nks : p.nks) * (p.cb / 16) * (p.Ntile / 2.0 > 16 ? p.Ntile / 2.0 : 16);
      const double mma_us = mma_item * per_cta / 1900.0;
      printf("  est_us tma %.1f mma %.1f  ntiles %d%s", tma_us, mma_us, p.n_tiles, p.pair ? "  pixel-pair rows" : "");
      // merged ConvTranspose: nsub counts (128-row sub-tile, column parity) pairs; items alternate the two row parities
      if (p.upm) printf("  merged %s: %d sub-tiles x 2 column parities, 2 row parities", net.layers[o.up_layer].name.c_str(), p.nsub / 2);
      printf("\n");
    }
    if (p.smem_bytes <= 113 * 1024) ++total_smem_small;
  }
  printf("layers with <= 113 KB shared memory: %ld\n", total_smem_small);
  return 0;
}
