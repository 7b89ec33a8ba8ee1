// Host-only developer tool: prints the launch plan of every convolution of the network (no GPU needed).
//   nvcc -std=c++17 -gencode arch=compute_100a,code=sm_100a --expt-relaxed-constexpr -o /tmp/plan_dump tools/plan_dump.cu -lcuda
//   /tmp/plan_dump [batch] [n|s] [ops] [up] [num_classes]
//   up: the runner's launch list, with proto.up merged into proto.cv2's launch (model.cuh fuse_up_conv)
//   The launch list follows the fusion switches the runner reads at create time: XRSEG_FUSE, XRSEG_FUSE_BNECK (read here as
//   xrseg_create reads them), XRSEG_FUSE_PE, XRSEG_FUSE_TAIL and XRSEG_FUSE_UP (read by model.cuh itself).
//
//   /tmp/plan_dump sig <scales> <micro-batches> <chunks> <class counts> [uniq]
//   One line per launch of the runner's list, with the parameters it runs with on 148 SMs (model.cuh plan_conv_op +
//   conv_launch_params, as xrseg_api.cu derives them), for every combination of
//     scales        n, s or ns
//     micro-batches 64, 1-512 or a comma list of those: the runner's micro-batch mb (the layers are planned for it)
//     chunks        comma list of nb = frames of the chunk that runs: a number, "mb" or "mb-1" (nb < mb: a partial chunk)
//     class counts  comma list
//   Line: "sig <scale> <mb> <nb> <nc> <kind> <launch> | <signature> | <geometry>".  The signature holds what selects a code
//   path (for a convolution: mode, K-blocks, rows per item, sub-tiles, stages, N tiles, pixel pairs, resident weights, the
//   merged / tail epilogues, accumulator sets, and whether the CTAs run 1, 2 or more rounds of the item loop, whether the
//   last round is ragged and whether the last item is a partial tile); the geometry holds the grid, the work items and the
//   frames (first:last, chunk-relative) the rows of item 0, of item `grid` (the first of the second round) and of the last item
//   belong to.  The last line of a combination is the post-processing's decode variant.  uniq: print a (scale, launch,
//   signature) only the first time it appears.
#include <math.h>
#include <string.h>
#include <set>
#include <string>
#include <vector>
#include "../xr_image_segmentation_b200/csrc/conv_tma.cuh"
#include "../xr_image_segmentation_b200/csrc/model.cuh"
using namespace xrseg;

namespace {
constexpr int SMS = 148;

std::vector<int> parse_list(const char* s, int mb = 0) {   // "1-512,600", "mb", "mb-1"
  std::vector<int> v;
  for (const char* p = s; *p;) {
    const char* e = strchr(p, ',');
    const std::string t(p, e ? e - p : strlen(p));
    if (t == "mb") v.push_back(mb);
    else if (t == "mb-1") v.push_back(mb - 1);
    else if (t.find('-') != std::string::npos) {
      for (int i = atoi(t.c_str()), hi = atoi(t.c_str() + t.find('-') + 1); i <= hi; ++i) v.push_back(i);
    } else v.push_back(atoi(t.c_str()));
    p = e ? e + 1 : p + t.size();
  }
  return v;
}

// Frames (first:last, chunk-relative) that the rows of work item w of a convolution launch belong to.  The item -> tile
// decomposition is the kernel's own (conv_tma.cuh, tma_kernel's producer loop: "tile = w >> ..." / "b = fd_div(p.fd_hp1,
// tile)", and the epilogue loop tma_epilogue_loop: the same two lines; flat mode: rows [tile * slots, + slots) of the
// [B*H*W, C] matrix).  Halo / s2 / merged: frame = tile / tpi (tiles per image); flat: row / (H*W).
std::string item_frames(const ConvParams& p, bool tma, long w, int nb) {
  if (!tma) return "0:" + std::to_string(nb - 1);     // thread-gather kernel: no persistent item loop over frames
  const int shift = p.upm ? 1 : (p.n_tiles == 4 ? 2 : (p.n_tiles == 2 ? 1 : 0));
  const long tile = w >> shift;
  long f0, f1;
  if (p.mode == MODE_FLAT_TMA) {
    const long hw = static_cast<long>(p.H) * p.W;
    const long r0 = tile * p.slots, r1 = std::min<long>(r0 + p.slots, p.flat_rows) - 1;
    f0 = r0 / hw; f1 = r1 / hw;
  } else {
    f0 = f1 = tile / p.tpi;
  }
  return std::to_string(f0) + ":" + std::to_string(f1);
}

std::string conv_line(const ConvParams& p, bool tma, int nb) {
  static const char* mode_name[] = {"gather", "halo", "halo_tma", "flat_tma", "s2_tma"};
  const long items = static_cast<long>(p.m_tiles) * p.n_tiles;
  const long rounds = (items + p.grid - 1) / p.grid;
  int partial = 0;                                      // the last item is a partial tile
  if (p.mode == MODE_FLAT_TMA) partial = p.flat_rows % p.slots != 0;
  // items tile the rows of p.H: the output rows in s2 mode (plan_conv_s2_tma_impl sets p.H = Ho), the input rows of the merged
  // ConvTranspose, the map's rows otherwise
  else if (p.mode == MODE_HALO_TMA || p.mode == MODE_S2_TMA) partial = p.H % p.R != 0;
  char b[512];
  snprintf(b, sizeof b, "mode %s cb %d kps %d nks %d R %d nsub %d S %d Ntile %d n_tiles %d pair %d bres %d upm %d tail %d nbuf %d "
           "rounds %s ragged %d partial %d | grid %d items %ld tpi %d frames %s %s %s",
           mode_name[p.mode], p.cb, p.kps, p.nks, p.R, p.nsub, p.S, p.Ntile, p.n_tiles, p.pair, p.b_resident, p.upm,
           p.tail_n > 0 ? 1 : 0, p.nbuf, rounds >= 3 ? "3+" : (rounds == 2 ? "2" : "1"), items % p.grid != 0 ? 1 : 0, partial,
           p.grid, items, p.tpi, item_frames(p, tma, 0, nb).c_str(),
           items > p.grid ? item_frames(p, tma, p.grid, nb).c_str() : "-", item_frames(p, tma, items - 1, nb).c_str());
  return b;
}

// The other launches: grid and tiling as xrseg_api.cu add_network_launches builds them (one CTA per tile of one frame,
// frame = blockIdx.z, except the SPPF pool: frame = blockIdx.x / (C / 8), and attention: frame = blockIdx.x / heads), so a
// launch is one round and its last tile holds the last frame.  These grids restate the launch code of the cases OP_STEM
// (stem_rows_kernel), OP_DW, OP_BNECK (bneck_grid), OP_UP, OP_SPPF and OP_ATTN there; tests/test_plan_coverage.py asserts
// on the GPU that every launch but the stem (whose kernel is chosen when it is launched) runs exactly this grid.
std::string other_line(const Op& o, int nb) {
  char b[512];
  const std::string ends = "| grid %ld items %ld tpi 0 frames 0:0 - " + std::to_string(nb - 1) + ":" + std::to_string(nb - 1);
  long gx = 1, gy = 1, per_frame = 1;
  std::string sig;
  switch (o.kind) {
    case OP_STEM: {                                     // stem_rows_kernel (640x640 frames): 64 x 16 output pixels per CTA
      gx = ceil_div(o.x.W / 2, 64); gy = ceil_div(o.x.H / 2, 16);
      snprintf(b, sizeof b, "tile 64x16 ragged_x %d ragged_y %d ", (o.x.W / 2) % 64 != 0, (o.x.H / 2) % 16 != 0);
      break;
    }
    case OP_DW: {                                       // dwconv3x3_kernel: 128 x 8 channels of a row band of `rows` rows
      const int rows = o.x.H >= 40 ? 16 : 10, lanes = o.x.W * (o.y.Cp / 8);
      gx = ceil_div(lanes, 128); gy = ceil_div(o.x.H, rows);
      snprintf(b, sizeof b, "rows %d ragged_x %d ragged_y %d ", rows, lanes % 128 != 0, o.x.H % rows != 0);
      break;
    }
    case OP_BNECK: {                                    // bottleneck_mma_kernel: 14 x 14 output pixels
      gx = ceil_div(o.x.W, 14); gy = ceil_div(o.x.H, 14);
      snprintf(b, sizeof b, "tile 14x14 c %d ragged_x %d ragged_y %d ", o.x.Cp, o.x.W % 14 != 0, o.x.H % 14 != 0);
      break;
    }
    case OP_UP: {                                       // upsample2x_kernel: 256 x 8 channels of one input row
      const int lanes = o.x.W * (o.x.Cp / 8);
      gx = ceil_div(lanes, 256); gy = o.x.H;
      snprintf(b, sizeof b, "ragged_x %d ", lanes % 256 != 0);
      break;
    }
    case OP_SPPF:                                       // sppf_pool_kernel: 8 channels of one frame
      per_frame = o.x.Cp / 4 / 8;
      snprintf(b, sizeof b, "c %d ", o.x.Cp / 4);
      break;
    case OP_ATTN: {                                     // attention_kernel: (frame, head) x 13 warps of 16 queries
      const int n = o.x.H * o.x.W;
      per_frame = o.heads; gy = ceil_div(n / 16, 13);
      snprintf(b, sizeof b, "heads %d tokens %d pe %d ragged_q %d ", o.heads, n, o.layer >= 0, (n / 16) % 13 != 0);
      break;
    }
    default: snprintf(b, sizeof b, "? ");
  }
  sig = b;
  const long grid = gx * gy * per_frame * nb;
  snprintf(b, sizeof b, ends.c_str(), grid, grid);
  return sig + b;
}
}  // namespace

int sig_main(int argc, char** argv) {
  if (argc < 6) { fprintf(stderr, "usage: plan_dump sig <n|s|ns> <micro-batches> <chunks> <class counts> [uniq]\n"); return 2; }
  const bool uniq = argc > 6 && strcmp(argv[6], "uniq") == 0;
  const char* fuse_env = getenv("XRSEG_FUSE");
  const char* bneck_env = getenv("XRSEG_FUSE_BNECK");
  const bool fuse = !(fuse_env && fuse_env[0] == '0'), bneck = !(bneck_env && bneck_env[0] == '0');
  const char* kind_name[] = {"stem", "conv", "dw", "sppf", "up", "attn", "bneck"};
  std::set<std::string> seen;
  for (const char* sc = argv[2]; *sc; ++sc)
    for (int mb : parse_list(argv[3]))
      for (int nc : parse_list(argv[5])) {
        Net net(*sc, mb, 640, fuse, bneck, nc, true);   // the runner's list (xrseg_create)
        std::vector<ConvParams> plan(net.ops.size());
        std::vector<char> tma(net.ops.size(), 0);
        for (size_t i = 0; i < net.ops.size(); ++i)
          if (net.ops[i].kind == OP_CONV) {
            tma[i] = plan_conv_op(net.ops[i], mb, SMS, plan[i]);
            if (net.ops[i].tail_layer >= 0) plan[i].tail_n = net.ops[i].ytail.Cp;   // xrseg_api.cu upload_layers
          }
        std::set<int> chunks;
        for (int nb : parse_list(argv[4], mb))
          if (nb >= 1 && nb <= mb) chunks.insert(nb);
        for (int nb : chunks) {
          int ups = 0;
          auto emit = [&](const std::string& launch, const char* kind, const std::string& rest) {
            const size_t bar = rest.find('|');
            if (uniq && !seen.insert(std::string(1, *sc) + " " + launch + " " + rest.substr(0, bar)).second) return;
            printf("sig %c %d %d %d %s %s | %s\n", *sc, mb, nb, nc, kind, launch.c_str(), rest.c_str());
          };
          for (size_t i = 0; i < net.ops.size(); ++i) {
            const Op& o = net.ops[i];
            std::string name = o.layer >= 0 ? net.layers[o.layer].name : std::string("-");
            if (o.kind == OP_CONV && o.layer2 >= 0) name += "+" + net.layers[o.layer2].name;
            if (o.kind == OP_UP) name = "up#" + std::to_string(ups++);
            if (o.kind == OP_SPPF) name = "sppf";
            if (o.kind == OP_ATTN && o.layer < 0) name = "attn";
            if (o.kind == OP_CONV) emit(name, "conv", conv_line(conv_launch_params(plan[i], tma[i], nb, SMS), tma[i], nb));
            else emit(name, kind_name[o.kind], other_line(o, nb));
          }
          // post.decode of the network's fp16 class tensor (xrseg_api.cu add_post_launches: 8 halves per 16-byte chunk)
          static const char* variant_name[] = {"80", "table", "wide"};
          const int pitch = class_pitch(nc);
          char b[128];
          snprintf(b, sizeof b, "decode %s pitch %d | grid %d", variant_name[decode_variant(nc, pitch, 8)], pitch, nb);
          emit("post.decode", "post", b);
        }
      }
  return 0;
}

int main(int argc, char** argv) {
  if (argc > 1 && strcmp(argv[1], "sig") == 0) return sig_main(argc, argv);
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
    ConvParams p;
    plan_conv_op(o, B, SMS, p);
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
