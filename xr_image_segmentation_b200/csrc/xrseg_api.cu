// xrseg_api.cu -- C ABI of libxrseg.so (include/xrseg.h): runner lifecycle, the per-frame pipeline
// (copy -> preprocess -> network -> decode -> NMS -> gather -> masks) on one CUDA stream, CUDA-graph replay, and the
// parity / debug entry points.  One runner per GPU; no CPU fallback anywhere on this path.
#include "../../include/xrseg.h"
#ifdef XRSEG_DEBUG_API
#include "../../include/xrseg_debug.h"
#endif

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <functional>
#include <memory>
#include <type_traits>

#include "common.cuh"
#include "conv_tma.cuh"
#include "conv_umma.cuh"
#include "kernels_misc.cuh"
#include "model.cuh"
#include "post.cuh"
#include "sentis.cuh"
#include "bottleneck.cuh"

using namespace xrseg;
static_assert(NC == 80, "model.cuh decode_variant names the class count decode_filter_kernel is specialised for");

namespace {

thread_local std::string g_create_error;

struct DevLayer {
  // OP_CONV (UMMA)
  ConvParams cp{};
  bool use_tma = false;            // 3x3 stride-1 layers: halo fetched by TMA (conv_tma.cuh)
  TmapSet tmaps{};
  __half* wpack = nullptr;
  float* bias = nullptr;
  // OP_CONV (direct) / OP_DW / OP_STEM
  __half* w16 = nullptr;
  float* w32 = nullptr;
  float* w32_u8 = nullptr;         // stem weights / 255 for the fused uint8 path
  uint2* wfrag = nullptr;          // OP_BNECK: mma.sync B-fragment order (bottleneck.cuh)
  __half* tail_w = nullptr;        // fused trailing 1x1 (Op::tail_layer): its [32][64] weights, 128-byte swizzle; bias in tail_bias
  float* tail_bias = nullptr;
  __half* w16_rows = nullptr;      // stem_rows_kernel weights
};

// ---- fused Bottleneck (bottleneck.cuh): one instantiation per supported channel triple ---------------------------------
constexpr int BNECK_TH = 14;   // output rows per CTA of every instantiation
dim3 bneck_grid(const BneckParams& p, int th) { return dim3(ceil_div(p.W, BNECK_TW), ceil_div(p.H, th), p.B); }
template <int C1, int CM, int C2, int TH>
void bneck_launch_t(const BneckParams& p, bool res, cudaStream_t st) {
  using Cfg = BneckCfg<C1, CM, C2, TH>;
  const dim3 grid = bneck_grid(p, TH);
  if (res) launch_k(bottleneck_mma_kernel<C1, CM, C2, TH, true>, grid, 256, Cfg::SMEM_BYTES, st, p);
  else launch_k(bottleneck_mma_kernel<C1, CM, C2, TH, false>, grid, 256, Cfg::SMEM_BYTES, st, p);
}
template <int C1, int CM, int C2, int TH>
void bneck_prepare_t() {
  using Cfg = BneckCfg<C1, CM, C2, TH>;
  XR_CUDA(cudaFuncSetAttribute(bottleneck_mma_kernel<C1, CM, C2, TH, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  XR_CUDA(cudaFuncSetAttribute(bottleneck_mma_kernel<C1, CM, C2, TH, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
}
void bneck_prepare_device() {
  bneck_prepare_t<16, 8, 16, BNECK_TH>();
  bneck_prepare_t<32, 16, 32, BNECK_TH>();
}
void launch_bneck(int c1, int cm, int c2, const BneckParams& p, bool res, cudaStream_t st) {
  if (c1 == 16 && cm == 8 && c2 == 16) bneck_launch_t<16, 8, 16, BNECK_TH>(p, res, st);
  else if (c1 == 32 && cm == 16 && c2 == 32) bneck_launch_t<32, 16, 32, BNECK_TH>(p, res, st);
  else XR_CHECK(false, "no fused Bottleneck kernel for %d-%d-%d channels", c1, cm, c2);
}

bool branches_disabled() {   // XRSEG_BRANCHES=0: everything on one stream (A/B measurements)
  const char* e = getenv("XRSEG_BRANCHES");
  return e && e[0] == '0';
}
bool mask_mma_enabled() {
  const char* e = getenv("XRSEG_MASK_MMA");
  return !(e && e[0] == '0');
}

template <typename T>
T* dev_alloc(size_t n) {
  T* p = nullptr;
  XR_CUDA(cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T)));
  return p;
}
template <typename T>
T* dev_upload(const std::vector<T>& v) {
  T* p = dev_alloc<T>(v.size());
  if (!v.empty()) XR_CUDA(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  return p;
}

// Scale and class count of an XRSW pack or .sentis asset: the scale from the first convolution's width (16 outputs: 'n',
// 32: 's'), the class count from the three *.cls.2 convolutions (canonical indices of that scale's topology), which must agree.
void weights_info(const void* data, size_t bytes, int& scale, int& nc) {
  XR_CHECK(data != nullptr, "no weights");
  std::vector<int> couts;   // output channels of every convolution, canonical order
  if (looks_like_sentis(data, bytes)) {
    const SentisWeights sw = sentis_load(data, bytes);
    for (const SentisConv& cv : sw.convs) couts.push_back(cv.w_shape.size() == 4 ? cv.w_shape[cv.transposed ? 1 : 0] : -1);
  } else {
    XR_CHECK(bytes >= sizeof(XrswHeader), "weight pack too small");
    XrswHeader h;
    memcpy(&h, data, sizeof(h));
    XR_CHECK(memcmp(h.magic, "XRSW", 4) == 0 && h.version == 1, "neither an XRSW v1 pack nor a .sentis asset");
    XR_CHECK(h.n_layers <= 4096 && bytes >= sizeof(XrswHeader) + static_cast<size_t>(h.n_layers) * sizeof(XrswLayer), "truncated pack");
    for (uint32_t i = 0; i < h.n_layers; ++i) {
      XrswLayer l;
      memcpy(&l, static_cast<const uint8_t*>(data) + sizeof(XrswHeader) + i * sizeof(XrswLayer), sizeof(l));
      couts.push_back(static_cast<int>(l.cout));
    }
  }
  XR_CHECK(!couts.empty() && (couts[0] == 16 || couts[0] == 32), "the first convolution has %d outputs: neither the n (16) nor the s (32) scale",
           couts.empty() ? 0 : couts[0]);
  scale = couts[0] == 16 ? 'n' : 's';
  const Net net(scale, 1);                                   // layer names and order do not depend on the class count
  XR_CHECK(couts.size() == net.layers.size(), "weights have %zu convolutions, the '%c' topology has %zu", couts.size(),
           static_cast<char>(scale), net.layers.size());
  std::vector<int> ncs;
  for (size_t i = 0; i < net.layers.size(); ++i)
    if (net.layers[i].name.size() > 6 && net.layers[i].name.compare(net.layers[i].name.size() - 6, 6, ".cls.2") == 0) ncs.push_back(couts[i]);
  XR_CHECK(ncs.size() == 3 && ncs[0] == ncs[1] && ncs[1] == ncs[2], "the class convolutions disagree: %d / %d / %d classes", ncs[0],
           ncs[1], ncs[2]);
  XR_CHECK(ncs[0] >= NC_MIN && ncs[0] <= NC_MAX, "%d classes: supported are %d..%d", ncs[0], NC_MIN, NC_MAX);
  nc = ncs[0];
}

}  // namespace

struct xrseg_runner {
  xrseg_config cfg{};
  int device = 0, num_sms = 148;
  std::string err;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev_done = nullptr, ev[6] = {}, user_ev[8] = {};
  std::unique_ptr<Net> net;
  int mb = 1;                      // frames per network pass
  int A = 8400;
  int nc = 80;                     // classes of the model (from the weights)
  std::vector<DevLayer> dl;
  __half* arena = nullptr;
  uint8_t* d_frames = nullptr;
  size_t d_frames_cap = 0;
  // post-processing state (sized for max_batch)
  float *d_boxes = nullptr, *d_scores = nullptr;
  int* d_labels = nullptr;
  unsigned long long* d_keys = nullptr;
  int *d_cand_count = nullptr, *d_n_cand = nullptr, *d_sorted_idx = nullptr, *d_overflow = nullptr, *d_filt_list = nullptr;
  float4* d_sorted_corners = nullptr;
  unsigned long long* d_mask = nullptr;
  int *d_keep_idx = nullptr, *d_keep_n = nullptr, *d_offsets = nullptr, *d_done = nullptr;
  float *o_boxes = nullptr, *o_coefs = nullptr, *o_scores = nullptr, *o_probs = nullptr;
  int *o_labels = nullptr, *o_anchor = nullptr, *o_frame = nullptr;
  // debug staging for xrseg_debug_post / xrseg_debug_nms
  float *dbg_box = nullptr, *dbg_cls = nullptr, *dbg_coef = nullptr, *dbg_proto = nullptr, *dbg_corners = nullptr;
  __half* dbg_h16 = nullptr;        // xrseg_debug_post_f16: [box | cls | coef | protos NHWC] rounded to fp16
  // host mirrors
  int *h_counts = nullptr, *h_offsets = nullptr;   // pinned
  int batch = 0;                   // batch of the scheduled / finished run
  int state = 0;                   // 0 idle, 1 scheduled, 2 done
  int words = 0, max_cand = 0, max_det = 0;
  struct ChunkGraph { int b0, nb; cudaGraphExec_t exec; };
  std::vector<ChunkGraph> graphs;     // one captured pipeline per (first frame, frame count) chunk
  cudaStream_t copy_stream = nullptr; // host->device frame copies, overlapped chunk by chunk with compute
  cudaStream_t side[4] = {};          // head / prototype branches inside the captured graph
  cudaEvent_t ev_tag[16] = {}, ev_join[4] = {};
  std::vector<cudaEvent_t> ev_copy;
  struct ChunkLaunches { int b0, nb; void* list; };   // list: std::vector<Launch>* (type local to this file)
  std::vector<ChunkLaunches> launch_cache;
  void* scratch = nullptr;            // grow-only device scratch for xrseg_decode / xrseg_masks results
  size_t scratch_cap = 0;
  int launches = 0, chunk_launches = 0;
  float timings[5] = {};
  std::vector<std::pair<std::string, std::pair<float, double>>> post_times;   // xrseg_debug_post under XRSEG_DBG_TIME: name, ms, bytes
  bool timed = false;
  // fused preprocess + stem: set by do_schedule when the frames are 640x640 (no resample), consumed by OP_STEM
  const uint8_t* fused_src = nullptr;
  int fused_stride = 0, fused_bpp = 0, fused_flip = 0;
  // NHWC fp16 prototypes the last post-processing stage read, which xrseg_masks' 640-px mode reads again: the network arena
  // after xrseg_schedule*, the caller's tensors after xrseg_debug_post_f16.  ptr == nullptr: none usable, `why` says why.
  struct ProtoSrc {
    const __half* ptr = nullptr;
    long bstride = 0;
    int pitch = 0;
    const char* why = "no run scheduled";
  } mask_protos;
  int* h_overflow = nullptr;         // pinned: bit 0 = more candidates than max_candidates, bit 1 = more kept boxes than max_det

  ~xrseg_runner();
};

namespace {

inline __half* ptr_of(xrseg_runner* r, const TV& t) { return r->arena + t.off; }

// ------------------------------------------------------------------------------------------------
// weights -> device, per layer kind
// ------------------------------------------------------------------------------------------------
void upload_layers(xrseg_runner* r, const std::vector<HostLayerWeights>& hw) {
  Net& net = *r->net;
  r->dl.resize(net.layers.size());
  for (size_t oi = 0; oi < net.ops.size(); ++oi) {
    const Op& o = net.ops[oi];
    if (o.layer < 0) continue;
    const LayerRec& l = net.layers[o.layer];
    const HostLayerWeights& w = hw[o.layer];
    DevLayer& d = r->dl[o.layer];
    if (o.kind == OP_STEM) {
      const int co = o.y.Cp;
      std::vector<float> ws(36 * co, 0.f), bs(co, 0.f);
      for (int n = 0; n < l.cout; ++n) {
        for (int ci = 0; ci < 3; ++ci)
          for (int t = 0; t < 9; ++t) ws[(t * 4 + ci) * co + n] = w.w[(static_cast<size_t>(n) * 3 + ci) * 9 + t];
        bs[n] = w.b[n];
      }
      d.w32 = dev_upload(ws);
      d.bias = dev_upload(bs);
      std::vector<__half> wt(static_cast<size_t>(co) * 48, __half(0.f));     // [Cout][12 taps][RGBX] for stem_mma_kernel
      for (int n = 0; n < l.cout; ++n)
        for (int ci = 0; ci < 3; ++ci)
          for (int t = 0; t < 9; ++t) wt[(static_cast<size_t>(n) * 12 + t) * 4 + ci] = __half(w.w[(static_cast<size_t>(n) * 3 + ci) * 9 + t]);
      d.w16 = dev_upload(wt);
      std::vector<__half> wr(static_cast<size_t>(co) * 48, __half(0.f));     // [Cout][kh][16]: k = 3 kw + c < 9 for stem_rows_kernel
      for (int n = 0; n < l.cout; ++n)
        for (int ci = 0; ci < 3; ++ci)
          for (int t = 0; t < 9; ++t)
            wr[(static_cast<size_t>(n) * 3 + t / 3) * 16 + 3 * (t % 3) + ci] = __half(w.w[(static_cast<size_t>(n) * 3 + ci) * 9 + t]);
      d.w16_rows = dev_upload(wr);
      for (float& v : ws) v = v / 255.0f;
      d.w32_u8 = dev_upload(ws);
    } else if (o.kind == OP_DW || o.kind == OP_ATTN) {   // OP_ATTN with a layer: the fused positional encoding's depthwise weights
      const int c = o.y.Cp;
      std::vector<float> ws(9 * c, 0.f), bs(c, 0.f);
      for (int n = 0; n < l.cout; ++n) {
        for (int t = 0; t < 9; ++t) ws[t * c + n] = w.w[static_cast<size_t>(n) * 9 + t];
        bs[n] = w.b[n];
      }
      d.w32 = dev_upload(ws);
      d.bias = dev_upload(bs);
    } else if (o.kind == OP_BNECK) {
      const LayerRec& l2 = net.layers[o.layer2];
      const HostLayerWeights& w2 = hw[o.layer2];
      DevLayer& d2 = r->dl[o.layer2];
      const int cm = round_up(l.cout, 8);
      std::vector<uint32_t> f1, f2;
      pack_bneck_weights(w.w.data(), l.cin, l.cout, o.x.Cp, cm, f1);
      pack_bneck_weights(w2.w.data(), l2.cin, l2.cout, cm, o.y.Cp, f2);
      std::vector<float> b1(cm, 0.f), b2(o.y.Cp, 0.f);
      std::copy(w.b.begin(), w.b.end(), b1.begin());
      std::copy(w2.b.begin(), w2.b.end(), b2.begin());
      d.wfrag = reinterpret_cast<uint2*>(dev_upload(f1));
      d.bias = dev_upload(b1);
      d2.wfrag = reinterpret_cast<uint2*>(dev_upload(f2));
      d2.bias = dev_upload(b2);
    } else if (o.kind == OP_CONV) {
      // sibling fusion: one weight matrix [Cout_a padded to 16 | Cout_b] x Cin x k x k, one bias vector
      HostLayerWeights fused;
      int cout_real = l.cout;
      if (o.layer2 >= 0) {
        const LayerRec& l2 = net.layers[o.layer2];
        const HostLayerWeights& w2 = hw[o.layer2];
        const size_t per = static_cast<size_t>(l.cin) * l.k * l.k;
        fused.w.assign((static_cast<size_t>(o.y.Cp) + l2.cout) * per, 0.f);
        fused.b.assign(static_cast<size_t>(o.y.Cp) + l2.cout, 0.f);
        std::copy(w.w.begin(), w.w.end(), fused.w.begin());
        std::copy(w.b.begin(), w.b.end(), fused.b.begin());
        std::copy(w2.w.begin(), w2.w.end(), fused.w.begin() + static_cast<size_t>(o.y.Cp) * per);
        std::copy(w2.b.begin(), w2.b.end(), fused.b.begin() + o.y.Cp);
        cout_real = o.y.Cp + l2.cout;
      }
      const HostLayerWeights& wsrc = o.layer2 >= 0 ? fused : w;
      d.use_tma = r->cfg.conv_impl == XRSEG_CONV_UMMA && plan_conv_op(o, r->mb, r->num_sms, d.cp);
      XR_CHECK(o.up_layer < 0 || (d.use_tma && d.cp.upm), "no launch plan for the merged ConvTranspose (%s)", l.name.c_str());
      if (d.use_tma && d.cp.mode == MODE_HALO_TMA) {
        d.tmaps.m[0] = make_halo_tensor_map(ptr_of(r, o.x), r->mb, o.x.H, o.x.W, o.x.Cp, o.x.pitch, d.cp.Wp, d.cp.hbox,
                                            d.cp.sw ? d.cp.cb : 8, d.cp.sw);
      } else if (d.use_tma && d.cp.mode == MODE_FLAT_TMA) {
        d.tmaps.m[0] = make_flat_tensor_map(ptr_of(r, o.x), static_cast<long>(r->mb) * o.x.H * o.x.W, o.x.Cp, o.x.pitch, d.cp);
      } else if (d.use_tma) {
        d.tmaps = make_s2_tensor_maps(ptr_of(r, o.x), r->mb, o.x.H, o.x.W, o.x.Cp, o.x.pitch, d.cp);
      }
      if (o.tail_layer >= 0) {
        // fused trailing 1x1 (model.cuh: fuse_tail_1x1): W2 as the 128-byte-swizzled image of a 1x1 layer with Ntile = 32, cb = 64
        const LayerRec& lt = net.layers[o.tail_layer];
        const HostLayerWeights& wt = hw[o.tail_layer];
        const int N1 = d.cp.Ntile, N2 = o.ytail.Cp;
        XR_CHECK(d.use_tma && d.cp.mode == MODE_HALO_TMA && d.cp.sw && N1 == 64 && N2 == 32 && d.cp.n_tiles == 1 && d.cp.b_resident &&
                     d.cp.nbuf == 2 && lt.cin <= N1,
                 "fused trailing 1x1 needs a halo TMA plan with Ntile 64, a 32-channel 1x1, resident weights and two accumulator sets (%s)",
                 l.name.c_str());
        ConvParams t{};
        t.Ntile = N2; t.n_tiles = 1; t.cb = N1; t.sw = N1 == 64 ? 3 : 2; t.taps = 1; t.nks = 1; t.kps = 1; t.b_stage_bytes = N2 * N1 * 2;
        t.Cout = N2;
        std::vector<__half> wp2;
        std::vector<float> bp2;
        pack_conv_weights_sw<__half>(t, wt.w.data(), wt.b.data(), lt.cin, lt.cout, wp2, bp2);
        r->dl[o.tail_layer].tail_w = dev_upload(wp2);
        r->dl[o.tail_layer].tail_bias = dev_upload(bp2);
        d.cp.tail_n = N2;
        d.cp.tail_act = o.tail_act;
        d.cp.smem_off_w2 = round_up(d.cp.smem_bytes, 1024);
        d.cp.smem_bytes = d.cp.smem_off_w2 + N2 * N1 * 2;
        XR_CHECK(d.cp.smem_bytes <= CONV_SMEM_MAX, "no room for the tail's weights (%s)", l.name.c_str());
      }
      if (r->cfg.conv_impl == XRSEG_CONV_UMMA) {
        std::vector<__half> wp;
        std::vector<float> bp;
        XR_CHECK(o.layer2 < 0 || (d.use_tma && d.cp.sw), "fused siblings need the TMA kernel (%s)", l.name.c_str());
        if (o.up_layer >= 0) {
          // merged ConvTranspose (model.cuh fuse_up_conv): parity weights and border biases from the dequantized fp32 weights in
          // fp64, each weight rounded to fp16 once; bias = [64 interior | 9 x 64 border corrections]
          const LayerRec& lu = net.layers[o.up_layer];
          const HostLayerWeights& wu = hw[o.up_layer];
          XR_CHECK(lu.cin == 64 && lu.cout == l.cin && l.cout == 64 && !w.b.empty() && !wu.b.empty(),
                   "merged ConvTranspose: unexpected shapes (%s)", l.name.c_str());
          std::vector<double> wm, bm;
          merge_upconv_weights(wu.w.data(), wu.b.data(), w.w.data(), w.b.data(), lu.cin, lu.cout, l.cout, wm, bm);
          pack_upmerge_weights_sw(d.cp, wm, lu.cin, l.cout, wp);
          bp.assign(bm.begin(), bm.end());
        } else if (d.use_tma && d.cp.sw) pack_conv_weights_sw<__half>(d.cp, wsrc.w.data(), wsrc.b.data(), l.cin, cout_real, wp, bp);
        else pack_conv_weights<__half>(d.cp, wsrc.w.data(), wsrc.b.data(), l.cin, cout_real, wp, bp);
        d.wpack = dev_upload(wp);
        d.bias = dev_upload(bp);
      } else {
        // direct layout: [Cout_p][k*k][Cin_p] or [4][Cout_p][Cin_p]
        const int cin_p = o.x.Cp, cout_p = o.y.Cp;
        const int taps = o.transposed ? 4 : o.k * o.k;
        std::vector<__half> wd(static_cast<size_t>(cout_p) * taps * cin_p, __half(0.f));
        std::vector<float> bs(cout_p, 0.f);
        for (int co = 0; co < l.cout; ++co) {
          bs[co] = w.b[co];
          for (int ci = 0; ci < l.cin; ++ci)
            for (int t = 0; t < taps; ++t) {
              if (o.transposed)
                wd[(static_cast<size_t>(t) * cout_p + co) * cin_p + ci] =
                    __half(w.w[(static_cast<size_t>(ci) * l.cout + co) * 4 + t]);
              else
                wd[(static_cast<size_t>(co) * taps + t) * cin_p + ci] =
                    __half(w.w[(static_cast<size_t>(co) * l.cin + ci) * taps + t]);
            }
        }
        d.w16 = dev_upload(wd);
        d.bias = dev_upload(bs);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// A run is a flat list of kernel launches (network, then post-processing); the normal path enqueues them in order,
// xrseg_profile_ops replays them one by one between CUDA events.
// ------------------------------------------------------------------------------------------------
struct Launch {
  std::string name;
  std::function<void(cudaStream_t)> fn;
  double flops = 0, bytes = 0;   // algorithmic work of the launch (real channel counts, fp16 activations)
  int branch = 0, wait_tag = 0, signal_tag = 0;   // see model.cuh Op::branch
  int grid = 0, items = 0, mode = -1;            // CTAs, work items and conv mode (-1: not a convolution) for xrseg_debug_launches
};

void add_network_launches(xrseg_runner* r, int nb, std::vector<Launch>& out) {
  Net& net = *r->net;
  for (size_t oi = 0; oi < net.ops.size(); ++oi) {
    const Op& o = net.ops[oi];
    Launch L;
    const double px_in = static_cast<double>(nb) * o.x.H * o.x.W, px_out = static_cast<double>(nb) * o.y.H * o.y.W;
    switch (o.kind) {
      case OP_STEM: {
        const LayerRec& l = net.layers[o.layer];
        StemParams p{ptr_of(r, o.x), ptr_of(r, o.y), r->dl[o.layer].w32, r->dl[o.layer].bias, nb, o.x.H, o.x.W, o.y.Cp,
                     o.y.pitch};
        const long total = static_cast<long>(nb) * (o.x.H / 2) * (o.x.W / 2) * (o.y.Cp / 16);
        const size_t smem = (37 * o.y.Cp) * sizeof(float);
        L.name = l.name;
        L.flops = 2.0 * px_out * l.cout * 27;
        L.bytes = px_in * 3 + px_out * l.cout * 2;     // the fused stem reads the caller's uint8 RGB frame (3 B per pixel)
        StemU8Params q{};
        q.out = ptr_of(r, o.y); q.out_pitch = o.y.pitch; q.w = r->dl[o.layer].w32_u8; q.bias = r->dl[o.layer].bias;
        q.B = nb; q.H = o.x.H; q.W = o.x.W; q.Cout = o.y.Cp;
        const size_t smem_u8 = smem + 33 * 33 * 4;
        // b0_off: frame offset of this chunk inside the scheduled batch (fused path reads the caller's frames directly)
        StemMmaParams mq{};
        mq.out = q.out; mq.out_pitch = q.out_pitch; mq.w16 = r->dl[o.layer].w16; mq.bias = q.bias;
        mq.B = nb; mq.H = o.x.H; mq.W = o.x.W; mq.in_scale = 1.0f / 255.0f;
        const int nt = o.y.Cp / 8;
        const __half* w16_rows = r->dl[o.layer].w16_rows;
        L.fn = [r, p, q, mq, nt, total, smem, smem_u8, nb, w16_rows](cudaStream_t st) {
          const bool aligned = (reinterpret_cast<uintptr_t>(r->fused_src) % 4 == 0) && (r->fused_stride % 4 == 0);
          const bool wide = (reinterpret_cast<uintptr_t>(r->fused_src) % 16 == 0) && (r->fused_stride % 16 == 0) &&
                            (mq.W * 3) % 16 == 0 && r->fused_bpp == 3;
          if (r->fused_src && wide && (nt == 2 || nt == 4) && r->cfg.conv_impl == XRSEG_CONV_UMMA) {
            StemMmaParams u = mq;                        // packed RGB rows: raw-byte staging (stem_rows_kernel)
            u.src = r->fused_src; u.stride_bytes = r->fused_stride; u.bpp = 3; u.w16 = w16_rows; u.flip = r->fused_flip;
            const dim3 grid(ceil_div(u.W / 2, STEM2_COLS), ceil_div(u.H / 2, STEM2_ROWS), nb);
            if (nt == 2) launch_k(stem_rows_kernel<2>, grid, 256, 0, st, u);
            else launch_k(stem_rows_kernel<4>, grid, 256, 0, st, u);
          } else if (r->fused_src && aligned && (nt == 2 || nt == 4) && r->cfg.conv_impl == XRSEG_CONV_UMMA) {
            StemMmaParams u = mq;
            u.src = r->fused_src; u.stride_bytes = r->fused_stride; u.bpp = r->fused_bpp; u.flip = r->fused_flip;
            const dim3 grid(ceil_div(u.W / 2, 32), ceil_div(u.H / 2, 8), nb);
            if (nt == 2) launch_k(stem_mma_kernel<2>, grid, 256, 0, st, u);
            else launch_k(stem_mma_kernel<4>, grid, 256, 0, st, u);
          } else if (r->fused_src) {
            StemU8Params u = q;
            u.src = r->fused_src; u.stride_bytes = r->fused_stride; u.bpp = r->fused_bpp; u.flip = r->fused_flip;
            launch_k(stem_u8_kernel, dim3(ceil_div(u.W / 2, 16), ceil_div(u.H / 2, 16), nb), 256, smem_u8, st, u);
          } else {
            launch_k(stem_conv_kernel, grid_for(total), 256, smem, st, p);
          }
        };
        break;
      }
      case OP_CONV: {
        const LayerRec& l = net.layers[o.layer];
        DevLayer& d = r->dl[o.layer];
        L.name = l.name;
        const double taps = o.transposed ? 1.0 : static_cast<double>(o.k) * o.k;
        int cout_alg = l.cout;                       // algorithmic output channels (both siblings of a fused launch)
        if (o.layer2 >= 0) {
          cout_alg += net.layers[o.layer2].cout;
          L.name = l.name + "+" + net.layers[o.layer2].name.substr(net.layers[o.layer2].name.find('.') + 1);
          if (L.name.size() > 31) L.name.resize(31);
        }
        // merged ConvTranspose: 4 taps per output pixel, weights of four parities x four taps
        const bool upm = o.up_layer >= 0;
        const double wtaps = upm ? 16.0 : static_cast<double>(o.k) * o.k;
        L.flops = 2.0 * (o.transposed ? px_in * 4 : px_out) * cout_alg * l.cin * (upm ? 4.0 : taps);
        L.bytes = (px_in * l.cin + px_out * cout_alg * (o.has_res ? 2 : 1) + static_cast<double>(cout_alg) * l.cin * wtaps) * 2;
        if (r->cfg.conv_impl == XRSEG_CONV_UMMA) {
          ConvParams p = conv_launch_params(d.cp, d.use_tma, nb, r->num_sms);
          L.grid = p.grid; L.items = p.m_tiles * p.n_tiles; L.mode = p.mode;
          p.in = ptr_of(r, o.x); p.out = ptr_of(r, o.y);
          if (o.layer2 >= 0) { p.out2 = ptr_of(r, o.y2); p.split_n = o.y.Cp; p.out2_pitch = o.y2.pitch; }
          p.res = o.has_res ? ptr_of(r, o.res) : nullptr;
          p.wpack = d.wpack; p.bias = d.bias;
          if (o.tail_layer >= 0) {                    // the launch's destination is the fused 1x1's
            const LayerRec& lt = net.layers[o.tail_layer];
            p.out = ptr_of(r, o.ytail); p.out_pitch = o.ytail.pitch;
            p.tail_w = r->dl[o.tail_layer].tail_w; p.tail_bias = r->dl[o.tail_layer].tail_bias;
            L.name = l.name + "+" + lt.name.substr(lt.name.find('.') + 1);
            if (upm) L.name = net.layers[o.up_layer].name + "+" + L.name.substr(L.name.find('.') + 1);   // "proto.up+cv2+cv3"
            L.flops += 2.0 * px_out * lt.cout * lt.cin;
            L.bytes = (px_in * l.cin + px_out * lt.cout + static_cast<double>(cout_alg) * l.cin * wtaps + static_cast<double>(lt.cout) * lt.cin) * 2;
          }
          if (d.use_tma) {
            const TmapSet maps = d.tmaps;
            L.fn = [p, maps](cudaStream_t st) { launch_conv_halo_tma(p, maps, st); };
          } else {
            L.fn = [p](cudaStream_t st) { launch_conv_umma(p, st); };
          }
        } else {
          DirectParams p{};
          p.in = ptr_of(r, o.x); p.in_pitch = o.x.pitch; p.out = ptr_of(r, o.y); p.out_pitch = o.y.pitch;
          p.res = o.has_res ? ptr_of(r, o.res) : nullptr; p.res_pitch = o.has_res ? o.res.pitch : 0;
          p.w = d.w16; p.bias = d.bias;
          p.B = nb; p.H = o.x.H; p.W = o.x.W; p.Cin = o.x.Cp; p.Ho = o.y.H; p.Wo = o.y.W; p.Cout = o.y.Cp;
          p.k = o.k; p.stride = o.stride; p.pad = o.k / 2; p.act = o.act; p.transposed = o.transposed;
          const long total = static_cast<long>(nb) * o.y.H * o.y.W * o.y.Cp;
          L.fn = [p, total](cudaStream_t st) { conv_direct_kernel<<<grid_for(total, 256, 148 * 32), 256, 0, st>>>(p); };
        }
        break;
      }
      case OP_BNECK: {
        const LayerRec &l = net.layers[o.layer], &l2 = net.layers[o.layer2];
        BneckParams p{};
        p.in = ptr_of(r, o.x); p.in_pitch = o.x.pitch; p.out = ptr_of(r, o.y); p.out_pitch = o.y.pitch;
        p.w1 = r->dl[o.layer].wfrag; p.b1 = r->dl[o.layer].bias; p.w2 = r->dl[o.layer2].wfrag; p.b2 = r->dl[o.layer2].bias;
        p.B = nb; p.H = o.x.H; p.W = o.x.W;
        const int c1 = o.x.Cp, cm = round_up(l.cout, 8), c2 = o.y.Cp;
        const bool res = o.has_res;
        L.name = l.name.substr(0, l.name.size() - 4);          // "b2.m0"
        L.flops = 2.0 * px_out * 9 * (static_cast<double>(l.cin) * l.cout + static_cast<double>(l2.cin) * l2.cout);
        L.bytes = (px_in * l.cin + px_out * l2.cout + 9.0 * (l.cin * l.cout + l2.cin * l2.cout)) * 2;
        {
          const dim3 g = bneck_grid(p, BNECK_TH);
          L.grid = L.items = static_cast<int>(g.x * g.y * g.z);
        }
        L.fn = [p, c1, cm, c2, res](cudaStream_t st) { launch_bneck(c1, cm, c2, p, res, st); };
        break;
      }
      case OP_DW: {
        const LayerRec& l = net.layers[o.layer];
        DwParams p{};
        p.in = ptr_of(r, o.x); p.in_pitch = o.x.pitch; p.out = ptr_of(r, o.y); p.out_pitch = o.y.pitch;
        p.res = o.has_res ? ptr_of(r, o.res) : nullptr; p.res_pitch = o.has_res ? o.res.pitch : 0;
        p.w = r->dl[o.layer].w32; p.bias = r->dl[o.layer].bias;
        p.B = nb; p.H = o.x.H; p.W = o.x.W; p.C = o.y.Cp; p.act = o.act;
        p.in_grp = o.in_grp; p.in_grp_stride = o.in_grp_stride; p.in_grp_off = o.in_grp_off;
        p.rows = o.x.H >= 40 ? 16 : 10;
        L.name = l.name;
        L.flops = 2.0 * px_out * l.cout * 9;
        L.bytes = (px_in * l.cin + px_out * l.cout * (o.has_res ? 2 : 1)) * 2;
        const dim3 grid(ceil_div(p.W * (p.C / 8), 128), ceil_div(p.H, p.rows), nb);
        L.grid = L.items = static_cast<int>(grid.x * grid.y * grid.z);
        L.fn = [p, grid](cudaStream_t st) { launch_k(dwconv3x3_kernel<4>, grid, 128, 0, st, p); };
        break;
      }
      case OP_SPPF: {
        SppfParams p{ptr_of(r, o.x), nb, o.x.H, o.x.W, o.x.Cp / 4, o.x.pitch};
        const size_t smem = static_cast<size_t>(o.x.H) * o.x.W * 32;
        L.name = "sppf.pool";
        L.bytes = px_in * p.C * 4 * 2;
        const int ctas = nb * (p.C / 8);
        L.grid = L.items = ctas;
        L.fn = [p, ctas, smem](cudaStream_t st) { launch_k(sppf_pool_kernel, ctas, 256, smem, st, p); };
        break;
      }
      case OP_UP: {
        UpParams p{ptr_of(r, o.x), o.x.pitch, ptr_of(r, o.y), o.y.pitch, nb, o.x.H, o.x.W, o.x.Cp};
        const dim3 grid(ceil_div(o.x.W * (o.x.Cp / 8), 256), o.x.H, nb);
        L.name = "upsample2x";
        L.bytes = px_in * o.x.C * 5 * 2;
        L.grid = L.items = static_cast<int>(grid.x * grid.y * grid.z);
        L.fn = [p, grid](cudaStream_t st) { launch_k(upsample2x_kernel, grid, 256, 0, st, p); };
        break;
      }
      case OP_ATTN: {
        AttnParams p{ptr_of(r, o.x), o.x.pitch, ptr_of(r, o.y), o.y.pitch, nb, o.x.H * o.x.W, o.heads,
                     1.0f / sqrtf(static_cast<float>(ATT_KD)), nullptr, nullptr, o.x.W};
        if (o.layer >= 0) { p.pe_w = r->dl[o.layer].w32; p.pe_b = r->dl[o.layer].bias; }   // fused positional encoding
        const size_t smem = static_cast<size_t>(p.N) * (ATT_KSTRIDE + ATT_VSTRIDE) * sizeof(__half);
        XR_CHECK(p.N % 16 == 0 && p.N % ATT_CHUNK == 0 && p.N / 16 <= 26, "attention kernel needs N %% 80 == 0 and N <= 416 (N = %d)", p.N);
        const int threads = 13 * 32;
        dim3 g(nb * o.heads, ceil_div(p.N / 16, 13));
        L.name = o.layer >= 0 ? "c2psa.attention+pe" : "c2psa.attention";
        L.flops = 2.0 * nb * o.heads * static_cast<double>(p.N) * p.N * (ATT_KD + ATT_HD) +
                  (o.layer >= 0 ? 2.0 * px_out * o.y.C * 9 : 0.0);
        L.bytes = px_in * (o.x.C + o.y.C) * 2;
        L.grid = L.items = static_cast<int>(g.x * g.y);
        L.fn = [p, g, smem, threads](cudaStream_t st) { launch_k(attention_kernel, g, threads, smem, st, p); };
        break;
      }
    }
    L.branch = o.branch; L.wait_tag = o.wait_tag; L.signal_tag = o.signal_tag;
    out.push_back(std::move(L));
  }
}

template <typename T>
void fill_scale_src(ScaleSrc<T> (&s)[3], const T* box, const T* cls, const T* coef, const int (&fh)[3],
                    const int (&fw)[3], const long (&bstr)[3][3], const int (&pitch)[3][3], const long (&off)[3][3]) {
  int a_off = 0;
  const float strides[3] = {8.f, 16.f, 32.f};
  for (int i = 0; i < 3; ++i) {
    s[i].box = box + off[i][0]; s[i].box_bstride = bstr[i][0]; s[i].box_pitch = pitch[i][0];
    s[i].cls = cls + off[i][1]; s[i].cls_bstride = bstr[i][1]; s[i].cls_pitch = pitch[i][1];
    s[i].coef = coef + off[i][2]; s[i].coef_bstride = bstr[i][2]; s[i].coef_pitch = pitch[i][2];
    s[i].h = fh[i]; s[i].w = fw[i]; s[i].a_off = a_off; s[i].stride = strides[i];
    a_off += fh[i] * fw[i];
  }
}

void net_scale_src(xrseg_runner* r, ScaleSrc<__half> (&s)[3]) {
  Net& net = *r->net;
  long bstr[3][3], off[3][3];
  int pitch[3][3];
  for (int i = 0; i < 3; ++i) {
    const TV* t[3] = {&net.box[i], &net.cls[i], &net.coef[i]};
    for (int j = 0; j < 3; ++j) {
      bstr[i][j] = static_cast<long>(t[j]->H) * t[j]->W * t[j]->pitch;
      pitch[i][j] = t[j]->pitch;
      off[i][j] = static_cast<long>(t[j]->off);
    }
  }
  fill_scale_src<__half>(s, r->arena, r->arena, r->arena, net.fh, net.fw, bstr, pitch, off);
}

template <typename T>
void dense_scale_src(xrseg_runner* r, ScaleSrc<T> (&s)[3], const T* box, const T* cls, const T* coef) {
  Net& net = *r->net;
  long bstr[3][3], off[3][3];
  int pitch[3][3];
  const int ch[3] = {64, class_pitch(r->nc), NM};   // class rows padded like the network's (the decode reads nc of them)
  long a_off = 0;
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) {
      bstr[i][j] = static_cast<long>(r->A) * ch[j];
      pitch[i][j] = ch[j];
      off[i][j] = a_off * ch[j];
    }
    a_off += net.fh[i] * net.fw[i];
  }
  fill_scale_src<T>(s, box, cls, coef, net.fh, net.fw, bstr, pitch, off);
}

#ifdef XRSEG_DEBUG_API
__global__ void f16_to_f32_kernel(const __half* src, float* dst, long n) {
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long>(gridDim.x) * blockDim.x)
    dst[i] = __half2float(src[i]);
}
__global__ void f32_to_f16_kernel(const float* src, __half* dst, long n) {
  for (long i = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long>(gridDim.x) * blockDim.x)
    dst[i] = __float2half_rn(src[i]);
}
#endif

// ------------------------------------------------------------------------------------------------
// post-processing of frames [b0, b0 + nb): decode -> sort -> bitmask -> reduce -> offsets -> gather -> masks
// ------------------------------------------------------------------------------------------------
template <typename T, bool PLANAR>
void add_post_launches(xrseg_runner* r, int b0, int nb, const ScaleSrc<T> (&src)[3], const T* protos, long proto_bstride,
                       int proto_pitch, bool do_decode, bool corners_given, std::vector<Launch>& out) {
  const int A = r->A;
  if (do_decode) {
    DecodeParams<T> dp{};
    for (int i = 0; i < 3; ++i) dp.s[i] = src[i];
    dp.B = nb; dp.A = A; dp.nc = r->nc; dp.score_thr = r->cfg.score_threshold;
    {
      const double t = r->cfg.score_threshold;
      dp.logit_floor = t <= 0.0 ? -3.0e38f : (t >= 1.0 ? 3.0e38f : static_cast<float>(std::log(t / (1.0 - t)) - 0.01));
    }
    dp.boxes = r->d_boxes + static_cast<long>(b0) * A * 4;
    dp.scores = r->d_scores + static_cast<long>(b0) * A;
    dp.labels = r->d_labels + static_cast<long>(b0) * A;
    dp.keys = r->d_keys + static_cast<long>(b0) * A;
    dp.cand_count = r->d_cand_count + b0;
    dp.filt_count = r->d_cand_count + r->cfg.max_batch + b0;
    dp.filt_list = r->d_filt_list + static_cast<long>(b0) * A;
    Launch L;
    L.name = "post.decode";
    // every anchor's class row (padding included: it shares the rows' sectors); box logits only for candidates
    const int pitch = src[0].cls_pitch;
    L.bytes = static_cast<double>(nb) * A * pitch * sizeof(T);
    constexpr int EPC = 16 / static_cast<int>(sizeof(T));
    for (int i = 0; i < 3; ++i)
      XR_CHECK(src[i].cls_pitch == pitch && pitch % EPC == 0 && pitch >= r->nc && pitch <= NC_MAX, "class tensor pitch %d", src[i].cls_pitch);
    const dim3 grid(ceil_div(A, 256), nb);
    const int variant = decode_variant(r->nc, pitch, EPC);
    if (variant == DECODE_80) {   // the COCO models: the kernel specialised for 80 classes
      L.fn = [dp, grid](cudaStream_t st) { launch_k(decode_filter_kernel<T>, grid, 256, 0, st, dp); };
    } else if (variant == DECODE_TABLE) {
      const size_t smem = static_cast<size_t>(8) * 32 * (pitch / EPC) * sizeof(float);
      L.fn = [dp, grid, smem](cudaStream_t st) { launch_k(decode_filter_nc_kernel<T>, grid, 256, smem, st, dp); };
    } else {
      L.fn = [dp, grid](cudaStream_t st) { launch_k(decode_filter_wide_kernel<T>, grid, 256, 0, st, dp); };
    }
    out.push_back(std::move(L));
    Launch L2;
    L2.name = "post.decode_exact";
    if (r->nc == NC) L2.fn = [dp, nb](cudaStream_t st) { launch_k(decode_exact_kernel<T, NC>, dim3(8, nb), 256, 0, st, dp); };
    else L2.fn = [dp, nb](cudaStream_t st) { launch_k(decode_exact_kernel<T, 0>, dim3(8, nb), 256, 0, st, dp); };
    out.push_back(std::move(L2));
  }
  SortParams sp{};
  sp.keys = r->d_keys + static_cast<long>(b0) * A;
  sp.cand_count = r->d_cand_count + b0;
  sp.boxes = corners_given ? r->dbg_corners + static_cast<long>(b0) * A * 4 : r->d_boxes + static_cast<long>(b0) * A * 4;
  sp.corners_given = corners_given ? 1 : 0;
  sp.A = A; sp.max_cand = r->max_cand;
  sp.sorted_idx = r->d_sorted_idx + static_cast<long>(b0) * r->max_cand;
  sp.sorted_corners = r->d_sorted_corners + static_cast<long>(b0) * r->max_cand;
  sp.n_cand = r->d_n_cand + b0;
  sp.overflow = r->d_overflow;
  MaskBitsParams mp{};
  mp.sorted_corners = sp.sorted_corners; mp.n_cand = sp.n_cand; mp.max_cand = r->max_cand; mp.words = r->words;
  mp.iou_thr = r->cfg.iou_threshold;
  mp.mask = r->d_mask + static_cast<long>(b0) * r->max_cand * r->words;
  ReduceParams rp{};
  rp.mask = mp.mask; rp.n_cand = sp.n_cand; rp.sorted_idx = sp.sorted_idx;
  rp.max_cand = r->max_cand; rp.words = r->words; rp.max_det = r->max_det;
  rp.keep_idx = r->d_keep_idx + static_cast<long>(b0) * r->max_det;
  rp.keep_n = r->d_keep_n + b0;
  rp.overflow = r->d_overflow;
  rp.keep_n_all = r->d_keep_n; rp.offsets = r->d_offsets; rp.done = r->d_done; rp.scan_upto = b0 + nb;
  const int words = r->words;
  {
    Launch L;
    L.name = "post.nms_sort";
    L.fn = [sp, nb](cudaStream_t st) { launch_k(nms_sort_kernel, nb, 1024, 16384 * sizeof(unsigned long long), st, sp); };
    out.push_back(std::move(L));
  }
  {
    Launch L;
    L.name = "post.nms_bitmask";
    L.fn = [mp, words, nb](cudaStream_t st) { launch_k(nms_bitmask_kernel, dim3(words, nb), 256, 0, st, mp); };
    out.push_back(std::move(L));
  }
  {
    Launch L;
    L.name = "post.nms_reduce";
    L.fn = [rp, words, nb](cudaStream_t st) {
      const size_t row_block = static_cast<size_t>(words) * 64 * sizeof(unsigned long long);
      if (words <= 32) launch_k(nms_reduce_kernel<1, 4>, nb, 128, 4 * row_block, st, rp);
      else launch_k(nms_reduce_kernel<5, 2>, nb, 128, 2 * row_block, st, rp);
    };
    out.push_back(std::move(L));
  }
  if (!src[0].coef) return;  // NMS-only debug path
  GatherParams<T> gp{};
  for (int i = 0; i < 3; ++i) gp.s[i] = src[i];
  gp.keep_idx = rp.keep_idx; gp.keep_n = rp.keep_n; gp.offsets = r->d_offsets + b0;
  gp.boxes = r->d_boxes + static_cast<long>(b0) * A * 4;
  gp.scores = r->d_scores + static_cast<long>(b0) * A;
  gp.labels = r->d_labels + static_cast<long>(b0) * A;
  gp.B = nb; gp.A = A; gp.max_det = r->max_det;
  gp.out_boxes = r->o_boxes; gp.out_labels = r->o_labels; gp.out_coefs = r->o_coefs; gp.out_scores = r->o_scores;
  gp.out_anchor = r->o_anchor; gp.out_frame = r->o_frame;
  {
    Launch L;
    L.name = "post.gather";
    L.fn = [gp, nb](cudaStream_t st) { launch_k(gather_kernel<T>, dim3(16, nb), 256, 0, st, gp); };
    out.push_back(std::move(L));
  }
  if (protos) {
    MaskParams<T, PLANAR> kp{};
    kp.protos = protos; kp.proto_bstride = proto_bstride; kp.proto_pitch = proto_pitch;
    kp.coefs = r->o_coefs; kp.keep_n = rp.keep_n; kp.offsets = gp.offsets; kp.max_det = r->max_det;
    kp.probs = r->o_probs;
    Launch L;
    L.name = "post.mask_prob";
    L.bytes = static_cast<double>(nb) * NM * PROTO_PIX * sizeof(T);   // + 102400 B per detection, added by the caller
    if constexpr (!PLANAR && std::is_same<T, __half>::value) {
      // network path: tensor-core variant (XRSEG_MASK_MMA=0 keeps the scalar FMA-chain kernel)
      if (mask_mma_enabled()) {
        L.fn = [kp, nb](cudaStream_t st) { launch_k(mask_prob_mma_kernel, dim3(PROTO_PIX / MASK_MMA_PIX, nb), 256, 0, st, kp); };
      } else {
        L.fn = [kp, nb](cudaStream_t st) { launch_k(mask_prob_kernel<T, PLANAR>, dim3(PROTO_PIX / 256, nb), 256, 0, st, kp); };
      }
    } else {
      L.fn = [kp, nb](cudaStream_t st) { launch_k(mask_prob_kernel<T, PLANAR>, dim3(PROTO_PIX / 256, nb), 256, 0, st, kp); };
    }
    out.push_back(std::move(L));
  }
}

// frame offset fix-up: gather/mask kernels index frames relative to b0 but o_frame must be global
__global__ void add_frame_base_kernel(int* frames, const int* offsets, int b0, int nb) {
  XR_PDL_ENTRY();
  const int b = blockIdx.x;
  if (b >= nb) return;
  const int lo = offsets[b0 + b], hi = offsets[b0 + b + 1];
  for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) frames[i] = b0 + b;
}

void preprocess(xrseg_runner* r, const uint8_t* d_src, int w, int h, int stride_bytes, int fmt, int flip, int nb, cudaStream_t st) {
  PreParams p{};
  p.src = d_src;
  p.dst = ptr_of(r, r->net->input);
  p.B = nb; p.sw = w; p.sh = h; p.stride_bytes = stride_bytes; p.bpp = fmt == XRSEG_FMT_RGBA8 ? 4 : 3;
  p.mode = r->cfg.resize_mode;
  p.flip = flip;
  if (p.mode == XRSEG_RESIZE_LETTERBOX) {
    const double rr = std::min(640.0 / h, 640.0 / w);
    p.nh = static_cast<int>(std::nearbyint(h * rr));   // round half to even, like Python's round() in oracle/preprocess.letterbox
    p.nw = static_cast<int>(std::nearbyint(w * rr));
    p.top = (640 - p.nh) / 2;
    p.left = (640 - p.nw) / 2;
    p.scale_x = static_cast<float>(w) / static_cast<float>(p.nw);
    p.scale_y = static_cast<float>(h) / static_cast<float>(p.nh);
  } else {
    p.scale_x = static_cast<float>(w) / 640.0f;
    p.scale_y = static_cast<float>(h) / 640.0f;
  }
  launch_k(preprocess_kernel, dim3(5, 640, nb), 128, 0, st, p);
  XR_CUDA(cudaGetLastError());
}

void build_chunk_launches(xrseg_runner* r, int b0, int nb, std::vector<Launch>& out) {
  add_network_launches(r, nb, out);
  ScaleSrc<__half> src[3];
  net_scale_src(r, src);
  const TV& pr = r->net->protos;
  add_post_launches<__half, false>(r, b0, nb, src, ptr_of(r, pr), static_cast<long>(pr.H) * pr.W * pr.pitch, pr.pitch,
                                   true, false, out);
  if (b0 == 0) return;   // gather already wrote chunk-relative frame ids, which are global for the first chunk
  Launch L;
  L.name = "post.frame_ids";
  int* frames = r->o_frame;
  const int* offsets = r->d_offsets;
  L.fn = [frames, offsets, b0, nb](cudaStream_t st) { launch_k(add_frame_base_kernel, nb, 64, 0, st, frames, offsets, b0, nb); };
  out.push_back(std::move(L));
}

// part: 0 = everything, 1 = only the first launch (the stem, whose source pointer may change per call),
//       2 = everything after the first launch (what the CUDA graph captures)
int pipeline_chunk(xrseg_runner* r, int b0, int nb, cudaStream_t st, int part = 0) {
  std::vector<Launch>* ls = nullptr;
  for (auto& c : r->launch_cache)
    if (c.b0 == b0 && c.nb == nb) ls = static_cast<std::vector<Launch>*>(c.list);
  if (!ls) {
    ls = new std::vector<Launch>();
    build_chunk_launches(r, b0, nb, *ls);
    r->launch_cache.push_back({b0, nb, ls});
  }
  const size_t lo = part == 2 ? 1 : 0, hi = part == 1 ? 1 : ls->size();
  // Branch concurrency (only while capturing the graph, part == 2): the head / prototype chains run on side streams,
  // forked after the feature map they read (P3 / P4 / P5) and joined before the post-processing.  The small P4 / P5
  // kernels keep only part of the SMs busy; this lets independent ones share the GPU.
  const bool fork = part == 2 && r->side[0] != nullptr && r->cfg.use_cuda_graph && !branches_disabled();
  bool used[5] = {};
  static const bool dbg_sync = getenv("XRSEG_DBG_SYNC") != nullptr;
  for (size_t i = lo; i < hi; ++i) {
    Launch& L = (*ls)[i];
    cudaStream_t s = st;
    if (fork && L.branch > 0) {
      s = r->side[L.branch - 1];
      if (L.wait_tag) XR_CUDA(cudaStreamWaitEvent(s, r->ev_tag[L.wait_tag - 3], 0));
      used[L.branch] = true;
    } else if (fork && L.branch == 0 && (used[1] || used[2] || used[3] || used[4]) && L.name.rfind("post.", 0) == 0) {
      for (int b = 1; b <= 4; ++b)                       // join before the first post-processing kernel
        if (used[b]) {
          XR_CUDA(cudaEventRecord(r->ev_join[b - 1], r->side[b - 1]));
          XR_CUDA(cudaStreamWaitEvent(st, r->ev_join[b - 1], 0));
          used[b] = false;
        }
    }
#ifdef XRSEG_DEBUG_API
    // XRSEG_SKIP=prefix1,prefix2,...: leave out every launch whose name starts with one of the prefixes (timing experiments
    // only: the results are garbage) -- how much of a step a group of launches costs INSIDE the captured graph
    static const std::string skip_env = getenv("XRSEG_SKIP") ? getenv("XRSEG_SKIP") : "";
    bool skipped = false;
    for (size_t a0 = 0; a0 < skip_env.size();) {
      size_t a1 = skip_env.find(',', a0);
      if (a1 == std::string::npos) a1 = skip_env.size();
      if (a1 > a0 && L.name.compare(0, a1 - a0, skip_env, a0, a1 - a0) == 0) skipped = true;
      a0 = a1 + 1;
    }
    if (!skipped)
#endif
    L.fn(s);
    if (dbg_sync && !r->cfg.use_cuda_graph) {            // XRSEG_DBG_SYNC=1 (no graph): name the launch that faults
      const cudaError_t e = cudaStreamSynchronize(s);
      XR_CHECK(e == cudaSuccess, "launch %zu '%s' (frames %d..%d): %s", i, L.name.c_str(), b0, b0 + nb - 1, cudaGetErrorString(e));
    }
    if (fork && L.signal_tag) XR_CUDA(cudaEventRecord(r->ev_tag[L.signal_tag - 3], s));
  }
  XR_CUDA(cudaGetLastError());
  return static_cast<int>(hi - lo);
}

}  // namespace
void free_launch_cache(xrseg_runner* r) {
  for (auto& c : r->launch_cache) delete static_cast<std::vector<Launch>*>(c.list);
  r->launch_cache.clear();
}
namespace {

void* ensure_scratch(xrseg_runner* r, size_t bytes) {
  if (bytes > r->scratch_cap) {
    XR_CUDA(cudaStreamSynchronize(r->stream));
    if (r->scratch) XR_CUDA(cudaFree(r->scratch));
    r->scratch_cap = bytes + bytes / 2 + 4096;
    XR_CUDA(cudaMalloc(&r->scratch, r->scratch_cap));
  }
  return r->scratch;
}

void reset_counters(xrseg_runner* r, int batch, cudaStream_t st) {
  XR_CUDA(cudaMemsetAsync(r->d_cand_count, 0, sizeof(int) * 2 * r->cfg.max_batch, st));   // candidate + filter counters
  XR_CUDA(cudaMemsetAsync(r->d_overflow, 0, sizeof(int), st));
  XR_CUDA(cudaMemsetAsync(r->d_done, 0, sizeof(int), st));                                // nms_reduce's ticket (self-resetting; belt and braces)
}

int do_schedule(xrseg_runner* r, const uint8_t* src, bool src_on_device, int w, int h, int stride_bytes, int fmt_flags,
                int batch) {
  if (!r) return XRSEG_ERR_INVALID;
  const int flip = (fmt_flags & XRSEG_FMT_BOTTOM_UP) ? 1 : 0;
  const int fmt = fmt_flags & ~XRSEG_FMT_BOTTOM_UP;
  try {
    if (!src || batch < 1 || batch > r->cfg.max_batch || w < 1 || h < 1 ||
        stride_bytes < w * (fmt == XRSEG_FMT_RGBA8 ? 4 : 3) || (fmt != XRSEG_FMT_RGB8 && fmt != XRSEG_FMT_RGBA8)) {
      r->err = "xrseg_schedule: invalid arguments";
      return XRSEG_ERR_INVALID;
    }
    XR_CUDA(cudaSetDevice(r->device));
    cudaStream_t st = r->stream;
    const size_t frame_bytes = static_cast<size_t>(h) * stride_bytes;
    const uint8_t* d_src = src;
    const int n_chunks = ceil_div(batch, r->mb);
    if (!src_on_device) {
      if (frame_bytes * batch > r->d_frames_cap) {
        XR_CUDA(cudaStreamSynchronize(st));
        if (r->d_frames) XR_CUDA(cudaFree(r->d_frames));
        r->d_frames_cap = frame_bytes * r->cfg.max_batch;
        XR_CUDA(cudaMalloc(&r->d_frames, r->d_frames_cap));
      }
      while (static_cast<int>(r->ev_copy.size()) < n_chunks + 1) {
        cudaEvent_t e;
        XR_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        r->ev_copy.push_back(e);
      }
      // the staging buffer may still be read by the previous run: order the copies after everything enqueued so far
      XR_CUDA(cudaEventRecord(r->ev_copy[n_chunks], st));
      XR_CUDA(cudaStreamWaitEvent(r->copy_stream, r->ev_copy[n_chunks], 0));
      for (int k = 0; k < n_chunks; ++k) {
        const int b0 = k * r->mb, nb = std::min(r->mb, batch - b0);
        XR_CUDA(cudaMemcpyAsync(r->d_frames + b0 * frame_bytes, src + b0 * frame_bytes, frame_bytes * nb,
                                cudaMemcpyHostToDevice, r->copy_stream));
        XR_CUDA(cudaEventRecord(r->ev_copy[k], r->copy_stream));
      }
      d_src = r->d_frames;
    }
    r->batch = batch;
    const TV& pr = r->net->protos;
    if (batch > r->mb)
      r->mask_protos = {nullptr, 0, 0, "640-px masks need the prototypes of every frame resident: use micro_batch >= batch"};
    else
      r->mask_protos = {ptr_of(r, pr), static_cast<long>(pr.H) * pr.W * pr.pitch, pr.pitch, nullptr};
    r->timed = !r->cfg.use_cuda_graph;
    if (r->timed) XR_CUDA(cudaEventRecord(r->ev[0], st));
    reset_counters(r, batch, st);
    const bool fused = (w == 640 && h == 640);     // no resample needed: the stem reads the uint8 frames directly
    r->fused_stride = stride_bytes;
    r->fused_bpp = fmt == XRSEG_FMT_RGBA8 ? 4 : 3;
    r->fused_flip = flip;
    int launches = 0;
    for (int k = 0; k < n_chunks; ++k) {
      const int b0 = k * r->mb, nb = std::min(r->mb, batch - b0);
      const uint8_t* chunk_src = d_src + static_cast<size_t>(b0) * frame_bytes;
      if (!src_on_device) XR_CUDA(cudaStreamWaitEvent(st, r->ev_copy[k], 0));   // chunk k+1 copies while chunk k computes
      r->fused_src = fused ? chunk_src : nullptr;
      if (!fused) preprocess(r, chunk_src, w, h, stride_bytes, fmt, flip, nb, st);
      if (r->timed && k == 0) XR_CUDA(cudaEventRecord(r->ev[1], st));
      launches += fused ? 0 : 1;
      if (r->cfg.use_cuda_graph) {
        // the stem stays outside the graph (its source pointer varies from call to call); the rest is replayed
        launches += pipeline_chunk(r, b0, nb, st, 1);
        cudaGraphExec_t exec = nullptr;
        for (auto& g : r->graphs)
          if (g.b0 == b0 && g.nb == nb) exec = g.exec;
        if (!exec) {
          cudaGraph_t g = nullptr;
          XR_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
          try {
            r->chunk_launches = pipeline_chunk(r, b0, nb, st, 2);
          } catch (...) {
            cudaStreamEndCapture(st, &g);
            if (g) cudaGraphDestroy(g);
            throw;
          }
          XR_CUDA(cudaStreamEndCapture(st, &g));
          XR_CUDA(cudaGraphInstantiate(&exec, g, 0));
          XR_CUDA(cudaGraphDestroy(g));
          r->graphs.push_back({b0, nb, exec});
        }
        XR_CUDA(cudaGraphLaunch(exec, st));
        launches += r->chunk_launches;
      } else {
        launches += pipeline_chunk(r, b0, nb, st);
      }
    }
    r->launches = launches;
    if (r->timed) XR_CUDA(cudaEventRecord(r->ev[2], st));
    XR_CUDA(cudaMemcpyAsync(r->h_offsets, r->d_offsets, sizeof(int) * (batch + 1), cudaMemcpyDeviceToHost, st));
    XR_CUDA(cudaMemcpyAsync(r->h_counts, r->d_keep_n, sizeof(int) * batch, cudaMemcpyDeviceToHost, st));
    XR_CUDA(cudaMemcpyAsync(r->h_overflow, r->d_overflow, sizeof(int), cudaMemcpyDeviceToHost, st));
    XR_CUDA(cudaEventRecord(r->ev_done, st));
    r->state = 1;
    return XRSEG_OK;
  } catch (const CudaError& e) {
    r->err = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    r->err = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    r->err = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
}

int finish(xrseg_runner* r) {
  if (r->state == 0) { r->err = "no run scheduled"; return XRSEG_ERR_STATE; }
  if (r->state == 1) {
    cudaError_t e = cudaEventSynchronize(r->ev_done);
    if (e != cudaSuccess) { r->err = std::string("run failed: ") + cudaGetErrorString(e); return XRSEG_ERR_CUDA; }
    if (r->timed) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, r->ev[0], r->ev[2]) == cudaSuccess) r->timings[0] = ms;
      if (cudaEventElapsedTime(&ms, r->ev[0], r->ev[1]) == cudaSuccess) r->timings[1] = ms;
      cudaGetLastError();  // an unrecorded event is not an error of the run
    }
    r->state = 2;
    // The reference's NonMaxSuppression is unlimited (maxOutputBoxesPerClass = -1, IEModelEditorConverter.cs:76); this build
    // works inside max_candidates / max_det.  A run that hit either cap is reported ONCE, here: the (truncated) results stay
    // readable, later calls on the finished run return normally, xrseg_overflow() keeps the bits.
    if (*r->h_overflow) {
      char b[200];
      snprintf(b, sizeof(b), "NMS capacity exceeded:%s%s -- results are truncated; recreate the runner with larger caps",
               (*r->h_overflow & 1) ? " more score-filtered candidates than max_candidates" : "",
               (*r->h_overflow & 2) ? " more kept boxes than max_det" : "");
      r->err = b;
      return XRSEG_ERR_CAPACITY;
    }
  }
  return 1;
}

size_t out_row_bytes(int idx) {
  switch (idx) {
    case 0: return 4 * sizeof(float);
    case 1: return sizeof(int);
    case 2: return NM * sizeof(float);
    case 3: return static_cast<size_t>(PROTO_PIX) * sizeof(float);
  }
  return 0;
}
const void* out_ptr(xrseg_runner* r, int idx) {
  switch (idx) {
    case 0: return r->o_boxes;
    case 1: return r->o_labels;
    case 2: return r->o_coefs;
    case 3: return r->o_probs;
  }
  return nullptr;
}

}  // namespace

void free_launch_cache(xrseg_runner* r);

xrseg_runner::~xrseg_runner() {
  cudaSetDevice(device);
  if (stream) cudaStreamSynchronize(stream);
  for (auto& g : graphs) cudaGraphExecDestroy(g.exec);
  free_launch_cache(this);
  if (copy_stream) cudaStreamDestroy(copy_stream);
  for (cudaStream_t s : side) if (s) cudaStreamDestroy(s);
  for (cudaEvent_t e : ev_tag) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : ev_join) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : ev_copy) cudaEventDestroy(e);
  cudaFree(scratch);
  for (DevLayer& d : dl) {
    cudaFree(d.wpack); cudaFree(d.wfrag); cudaFree(d.tail_w); cudaFree(d.tail_bias); cudaFree(d.w16_rows); cudaFree(d.bias); cudaFree(d.w16); cudaFree(d.w32); cudaFree(d.w32_u8);
  }
  void* bufs[] = {arena, d_frames, d_boxes, d_scores, d_labels, d_keys, d_cand_count, d_n_cand, d_sorted_idx, d_filt_list,
                  d_overflow, d_sorted_corners, d_mask, d_keep_idx, d_keep_n, d_offsets, d_done, o_boxes, o_coefs, o_scores,
                  o_probs, o_labels, o_anchor, o_frame, dbg_box, dbg_cls, dbg_coef, dbg_proto, dbg_corners, dbg_h16};
  for (void* b : bufs) cudaFree(b);
  if (h_counts) cudaFreeHost(h_counts);
  if (h_offsets) cudaFreeHost(h_offsets);
  if (h_overflow) cudaFreeHost(h_overflow);
  if (ev_done) cudaEventDestroy(ev_done);
  for (cudaEvent_t e : ev) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : user_ev) if (e) cudaEventDestroy(e);
  if (stream) cudaStreamDestroy(stream);
}

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int xrseg_abi_version(void) { return XRSEG_ABI_VERSION; }

const char* xrseg_last_error(const xrseg_runner* r) { return r ? r->err.c_str() : g_create_error.c_str(); }

void* xrseg_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}
void xrseg_host_free(void* p) {
  if (p) cudaFreeHost(p);
}
int xrseg_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  int ok = 0;
  for (int i = 0; i < n; ++i) {
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, i) == cudaSuccess && prop.major == 10) ++ok;
  }
  return ok;
}

int xrseg_layer_count(int model_scale) { return xrseg_layer_count_nc(model_scale, 80); }

int xrseg_layer_count_nc(int model_scale, int num_classes) {
  try {
    if ((model_scale != 'n' && model_scale != 's') || num_classes < NC_MIN || num_classes > NC_MAX) return XRSEG_ERR_INVALID;
    Net net(model_scale, 1, 640, true, true, num_classes);
    return static_cast<int>(net.layers.size());
  } catch (const CudaError& e) {
    g_create_error = e.msg;
    return XRSEG_ERR_INVALID;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    g_create_error = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_INVALID;
  } catch (...) {
    g_create_error = "unknown exception";
    return XRSEG_ERR_INVALID;
  }
}

int xrseg_layer_info_get(int model_scale, int index, xrseg_layer_info* info) {
  return xrseg_layer_info_get_nc(model_scale, 80, index, info);
}

int xrseg_layer_info_get_nc(int model_scale, int num_classes, int index, xrseg_layer_info* info) {
  try {
    if ((model_scale != 'n' && model_scale != 's') || num_classes < NC_MIN || num_classes > NC_MAX || !info) return XRSEG_ERR_INVALID;
    Net net(model_scale, 1, 640, true, true, num_classes);
    if (index < 0 || index >= static_cast<int>(net.layers.size())) return XRSEG_ERR_INVALID;
    const LayerRec& l = net.layers[index];
    memset(info, 0, sizeof(*info));
    strncpy(info->name, l.name.c_str(), sizeof(info->name) - 1);
    info->cin = l.cin; info->cout = l.cout; info->k = l.k; info->stride = l.stride; info->groups = l.groups;
    info->act = l.act; info->transposed = l.transposed; info->h_in = l.h_in; info->w_in = l.w_in;
    return XRSEG_OK;
  } catch (const CudaError& e) {
    g_create_error = e.msg;
    return XRSEG_ERR_INVALID;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    g_create_error = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_INVALID;
  } catch (...) {
    g_create_error = "unknown exception";
    return XRSEG_ERR_INVALID;
  }
}

int xrseg_sentis_info(const void* data, size_t bytes, int32_t* n_convs, float* iou_threshold, float* score_threshold) {
  if (!data) return XRSEG_ERR_INVALID;
  try {
    if (!looks_like_sentis(data, bytes)) { g_create_error = "not a .sentis container"; return XRSEG_ERR_WEIGHTS; }
    SentisWeights sw = sentis_load(data, bytes);
    if (n_convs) *n_convs = static_cast<int32_t>(sw.convs.size());
    if (iou_threshold) *iou_threshold = sw.has_nms ? sw.iou_threshold : 0.f;
    if (score_threshold) *score_threshold = sw.has_nms ? sw.score_threshold : 0.f;
    return XRSEG_OK;
  } catch (const CudaError& e) {
    g_create_error = e.msg;
    return XRSEG_ERR_WEIGHTS;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    g_create_error = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_WEIGHTS;
  } catch (...) {
    g_create_error = "unknown exception";
    return XRSEG_ERR_WEIGHTS;
  }
}

int xrseg_weights_info(const void* data, size_t bytes, int32_t* model_scale, int32_t* num_classes) {
  if (!data) return XRSEG_ERR_INVALID;
  try {
    int scale = 0, nc = 0;
    weights_info(data, bytes, scale, nc);
    if (model_scale) *model_scale = scale;
    if (num_classes) *num_classes = nc;
    return XRSEG_OK;
  } catch (const CudaError& e) {
    g_create_error = e.msg;
    return XRSEG_ERR_WEIGHTS;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    g_create_error = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_WEIGHTS;
  } catch (...) {
    g_create_error = "unknown exception";
    return XRSEG_ERR_WEIGHTS;
  }
}

int xrseg_num_classes(const xrseg_runner* r) { return r ? r->nc : XRSEG_ERR_INVALID; }

int xrseg_sentis_layer(const void* data, size_t bytes, int index, float* w, size_t w_cap, float* b, size_t b_cap,
                       int32_t* w_shape4, int32_t* transposed) {
  if (!data || index < 0) return XRSEG_ERR_INVALID;
  try {
    if (!looks_like_sentis(data, bytes)) { g_create_error = "not a .sentis container"; return XRSEG_ERR_WEIGHTS; }
    SentisWeights sw = sentis_load(data, bytes);
    if (static_cast<size_t>(index) >= sw.convs.size()) return XRSEG_ERR_INVALID;
    const SentisConv& cv = sw.convs[index];
    if (w_shape4) for (int i = 0; i < 4; ++i) w_shape4[i] = i < static_cast<int>(cv.w_shape.size()) ? cv.w_shape[i] : 1;
    if (transposed) *transposed = cv.transposed ? 1 : 0;
    if ((w && w_cap < cv.w.size()) || (b && b_cap < cv.b.size())) return XRSEG_ERR_CAPACITY;
    if (w) memcpy(w, cv.w.data(), cv.w.size() * sizeof(float));
    if (b) memcpy(b, cv.b.data(), cv.b.size() * sizeof(float));
    return static_cast<int>(cv.w.size());
  } catch (const CudaError& e) {
    g_create_error = e.msg;
    return XRSEG_ERR_WEIGHTS;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    g_create_error = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_WEIGHTS;
  } catch (...) {
    g_create_error = "unknown exception";
    return XRSEG_ERR_WEIGHTS;
  }
}

int xrseg_create(const xrseg_config* cfg_in, xrseg_runner** out) {
  if (!cfg_in || !out || cfg_in->struct_size != sizeof(xrseg_config)) {
    g_create_error = "xrseg_create: bad config (struct_size mismatch?)";
    return XRSEG_ERR_INVALID;
  }
  *out = nullptr;
  std::unique_ptr<xrseg_runner> r(new xrseg_runner());
  r->cfg = *cfg_in;
  xrseg_config& c = r->cfg;
  if (c.iou_threshold == 0.f) c.iou_threshold = 0.43f;
  if (c.score_threshold == 0.f) c.score_threshold = 0.301f;
  if (c.mask_threshold == 0.f) c.mask_threshold = 0.5f;
  if (c.mask_threshold < 0.f) c.mask_threshold = 0.f;   // negative = "exactly 0" (0 itself means default)
  if (c.max_det <= 0) c.max_det = 300;
  if (c.max_candidates <= 0) c.max_candidates = 2048;
  if (c.max_candidates > NUM_ANCHORS_MAX) c.max_candidates = NUM_ANCHORS_MAX;
  if (c.max_batch <= 0) c.max_batch = 1;
  if (c.model_scale != 'n' && c.model_scale != 's') {
    g_create_error = "model_scale must be 'n' or 's'";
    return XRSEG_ERR_INVALID;
  }
  try {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || c.device < 0 || c.device >= ndev) {
      g_create_error = "no CUDA device available (libxrseg has no CPU fallback)";
      return XRSEG_ERR_NO_DEVICE;
    }
    cudaDeviceProp prop{};
    XR_CUDA(cudaGetDeviceProperties(&prop, c.device));
    if (prop.major != 10) {
      g_create_error = std::string("device '") + prop.name + "' is not sm_100 (Blackwell B200); no other code path exists";
      return XRSEG_ERR_NO_DEVICE;
    }
    r->device = c.device;
    r->num_sms = prop.multiProcessorCount;
    XR_CUDA(cudaSetDevice(c.device));
    XR_CUDA(cudaStreamCreateWithFlags(&r->stream, cudaStreamNonBlocking));
    XR_CUDA(cudaStreamCreateWithFlags(&r->copy_stream, cudaStreamNonBlocking));
    for (auto& s : r->side) XR_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    for (auto& e : r->ev_tag) XR_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (auto& e : r->ev_join) XR_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    XR_CUDA(cudaEventCreateWithFlags(&r->ev_done, cudaEventDisableTiming));
    for (auto& e : r->ev) XR_CUDA(cudaEventCreate(&e));
    conv_umma_prepare_device();
    conv_tma_prepare_device();
    bneck_prepare_device();
    XR_CUDA(cudaFuncSetAttribute(attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    XR_CUDA(cudaFuncSetAttribute(nms_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 16384 * 8));
    XR_CUDA(cudaFuncSetAttribute((nms_reduce_kernel<1, 4>), cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * 32 * 64 * 8));
    XR_CUDA(cudaFuncSetAttribute((nms_reduce_kernel<5, 2>), cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 132 * 64 * 8));

    try {   // the class count comes from the weights; a nonzero num_classes only confirms it
      int wscale = 0;
      weights_info(c.weights, c.weights_bytes, wscale, r->nc);
      XR_CHECK(c.num_classes == 0 || c.num_classes == r->nc, "num_classes is %d, the weights have %d classes", c.num_classes, r->nc);
    } catch (const CudaError& e) {
      g_create_error = e.msg;
      return XRSEG_ERR_WEIGHTS;
    } catch (const std::exception& e) {
      g_create_error = std::string("unexpected exception: ") + e.what();
      return XRSEG_ERR_WEIGHTS;
    }
    r->mb = c.micro_batch > 0 ? std::min(c.micro_batch, c.max_batch) : c.max_batch;
    const char* fuse_env = getenv("XRSEG_FUSE");
    const bool fuse = c.conv_impl == XRSEG_CONV_UMMA && !(fuse_env && fuse_env[0] == '0');
    const char* bneck_env = getenv("XRSEG_FUSE_BNECK");
    r->net.reset(new Net(c.model_scale, r->mb, 640, fuse, !(bneck_env && bneck_env[0] == '0'), r->nc, true));
    Net& net = *r->net;
    r->A = net.fh[0] * net.fw[0] + net.fh[1] * net.fw[1] + net.fh[2] * net.fw[2];
    std::vector<HostLayerWeights> hw;
    try {
      if (looks_like_sentis(c.weights, c.weights_bytes)) {
        // the sample's own asset (↔ ModelLoader.Load(_sentisModel), IEE:382): dequantize its convolutions in chain order
        SentisWeights sw = sentis_load(c.weights, c.weights_bytes);
        XR_CHECK(sw.convs.size() == net.layers.size(), "sentis asset has %zu convolutions, the '%c' topology has %zu",
                 sw.convs.size(), static_cast<char>(c.model_scale), net.layers.size());
        hw.resize(sw.convs.size());
        for (size_t i = 0; i < sw.convs.size(); ++i) {
          const LayerRec& l = net.layers[i];
          const SentisConv& cv = sw.convs[i];
          const int cin_g = l.cin / l.groups;
          const int d0 = l.transposed ? l.cin : l.cout, d1 = l.transposed ? l.cout : cin_g;
          XR_CHECK(cv.transposed == (l.transposed != 0) && cv.w_shape.size() == 4 && cv.w_shape[0] == d0 && cv.w_shape[1] == d1 &&
                       cv.w_shape[2] == l.k && cv.w_shape[3] == l.k && cv.b.size() == static_cast<size_t>(l.cout),
                   "sentis convolution %zu does not match topology layer %s", i, l.name.c_str());
          hw[i].w = cv.w;
          hw[i].b = cv.b;
        }
        // thresholds baked into the asset's NonMaxSuppression chain win over the built-in defaults (not over the caller)
        if (sw.has_nms && cfg_in->iou_threshold == 0.f) c.iou_threshold = sw.iou_threshold;
        if (sw.has_nms && cfg_in->score_threshold == 0.f) c.score_threshold = sw.score_threshold;
      } else {
        xrsw_load(c.weights, c.weights_bytes, net.layers, c.model_scale, hw);
      }
    } catch (const CudaError& e) {
      g_create_error = e.msg;
      return XRSEG_ERR_WEIGHTS;
    } catch (const std::exception& e) {   // nothing may unwind across the C boundary
      g_create_error = std::string("unexpected exception: ") + e.what();
      return XRSEG_ERR_WEIGHTS;
    } catch (...) {
      g_create_error = "unknown exception";
      return XRSEG_ERR_WEIGHTS;
    }
    r->arena = dev_alloc<__half>(net.arena_elems);
    XR_CUDA(cudaMemset(r->arena, 0, net.arena_elems * sizeof(__half)));
    upload_layers(r.get(), hw);

    const int B = c.max_batch, A = r->A;
    r->max_cand = c.max_candidates;
    r->max_det = c.max_det;
    r->words = ceil_div(r->max_cand, 64);
    r->d_boxes = dev_alloc<float>(static_cast<size_t>(B) * A * 4);
    r->d_scores = dev_alloc<float>(static_cast<size_t>(B) * A);
    r->d_labels = dev_alloc<int>(static_cast<size_t>(B) * A);
    r->d_keys = dev_alloc<unsigned long long>(static_cast<size_t>(B) * A);
    r->d_cand_count = dev_alloc<int>(2 * B);               // [0,B) candidates per frame, [B,2B) logit-filter survivors
    r->d_filt_list = dev_alloc<int>(static_cast<size_t>(B) * A);
    r->d_n_cand = dev_alloc<int>(B);
    r->d_sorted_idx = dev_alloc<int>(static_cast<size_t>(B) * r->max_cand);
    r->d_sorted_corners = dev_alloc<float4>(static_cast<size_t>(B) * r->max_cand);
    r->d_overflow = dev_alloc<int>(1);
    r->d_mask = dev_alloc<unsigned long long>(static_cast<size_t>(B) * r->max_cand * r->words);
    r->d_keep_idx = dev_alloc<int>(static_cast<size_t>(B) * r->max_det);
    r->d_keep_n = dev_alloc<int>(B);
    r->d_offsets = dev_alloc<int>(B + 1);
    r->d_done = dev_alloc<int>(1);
    XR_CUDA(cudaMemset(r->d_done, 0, sizeof(int)));
    const size_t cap = static_cast<size_t>(B) * r->max_det;
    r->o_boxes = dev_alloc<float>(cap * 4);
    r->o_labels = dev_alloc<int>(cap);
    r->o_coefs = dev_alloc<float>(cap * NM);
    r->o_scores = dev_alloc<float>(cap);
    r->o_anchor = dev_alloc<int>(cap);
    r->o_frame = dev_alloc<int>(cap);
    r->o_probs = dev_alloc<float>(cap * PROTO_PIX);
    XR_CUDA(cudaHostAlloc(&r->h_counts, sizeof(int) * B, cudaHostAllocDefault));
    XR_CUDA(cudaHostAlloc(&r->h_offsets, sizeof(int) * (B + 1), cudaHostAllocDefault));
    memset(r->h_counts, 0, sizeof(int) * B);
    memset(r->h_offsets, 0, sizeof(int) * (B + 1));
    XR_CUDA(cudaHostAlloc(&r->h_overflow, sizeof(int), cudaHostAllocDefault));
    *r->h_overflow = 0;
    XR_CUDA(cudaMemset(r->d_keep_n, 0, sizeof(int) * B));
    XR_CUDA(cudaMemset(r->d_offsets, 0, sizeof(int) * (B + 1)));
    XR_CUDA(cudaDeviceSynchronize());
  } catch (const CudaError& e) {
    g_create_error = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    g_create_error = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    g_create_error = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  *out = r.release();
  return XRSEG_OK;
}

void xrseg_destroy(xrseg_runner* r) { delete r; }

int xrseg_schedule(xrseg_runner* r, const uint8_t* frames, int w, int h, int stride_bytes, int fmt, int batch) {
  return do_schedule(r, frames, false, w, h, stride_bytes, fmt, batch);
}
int xrseg_schedule_device(xrseg_runner* r, const uint8_t* d_frames, int w, int h, int stride_bytes, int fmt, int batch) {
  return do_schedule(r, d_frames, true, w, h, stride_bytes, fmt, batch);
}

int xrseg_poll(xrseg_runner* r) {
  if (!r) return XRSEG_ERR_INVALID;
  if (r->state == 0) { r->err = "no run scheduled"; return XRSEG_ERR_STATE; }
  if (r->state == 2) return 1;
  cudaError_t e = cudaEventQuery(r->ev_done);
  if (e == cudaErrorNotReady) return 0;
  if (e != cudaSuccess) { r->err = std::string("run failed: ") + cudaGetErrorString(e); return XRSEG_ERR_CUDA; }
  return finish(r);
}

int xrseg_wait(xrseg_runner* r) {
  if (!r) return XRSEG_ERR_INVALID;
  return finish(r);
}

int xrseg_counts(xrseg_runner* r, int32_t* counts, int cap) {
  if (!r || !counts) return XRSEG_ERR_INVALID;
  int rc = finish(r);
  if (rc < 0) return rc;
  if (cap < r->batch) { r->err = "counts buffer too small"; return XRSEG_ERR_CAPACITY; }
  for (int i = 0; i < r->batch; ++i) counts[i] = r->h_counts[i];
  return r->batch;
}

int xrseg_overflow(xrseg_runner* r) {
  if (!r) return XRSEG_ERR_INVALID;
  if (r->state != 2) { r->err = "no finished run"; return XRSEG_ERR_STATE; }
  return *r->h_overflow;
}

int xrseg_peek_output(xrseg_runner* r, int idx, xrseg_tensor_view* v) {
  if (!r || !v || idx < 0 || idx > 3) return XRSEG_ERR_INVALID;
  int rc = finish(r);
  if (rc < 0) return rc;
  const int n = r->h_offsets[r->batch];
  memset(v, 0, sizeof(*v));
  v->device_ptr = out_ptr(r, idx);
  v->dtype = idx == 1 ? XRSEG_I32 : XRSEG_F32;
  v->shape[0] = n;
  if (idx == 0) { v->rank = 2; v->shape[1] = 4; }
  if (idx == 1) { v->rank = 1; }
  if (idx == 2) { v->rank = 2; v->shape[1] = NM; }
  if (idx == 3) { v->rank = 3; v->shape[1] = PROTO_HW; v->shape[2] = PROTO_HW; }
  return XRSEG_OK;
}

int xrseg_readback(xrseg_runner* r, int idx, void* dst, size_t cap_bytes, int64_t* shape, int* rank) {
  if (!r || idx < 0 || idx > 3) return XRSEG_ERR_INVALID;
  xrseg_tensor_view v;
  int rc = xrseg_peek_output(r, idx, &v);
  if (rc < 0) return rc;
  if (shape) for (int i = 0; i < v.rank; ++i) shape[i] = v.shape[i];
  if (rank) *rank = v.rank;
  const size_t bytes = static_cast<size_t>(v.shape[0]) * out_row_bytes(idx);
  if (bytes == 0) return XRSEG_OK;
  if (!dst || cap_bytes < bytes) { r->err = "readback buffer too small"; return XRSEG_ERR_CAPACITY; }
  try {
    XR_CUDA(cudaSetDevice(r->device));
    XR_CUDA(cudaMemcpyAsync(dst, v.device_ptr, bytes, cudaMemcpyDeviceToHost, r->stream));
    XR_CUDA(cudaStreamSynchronize(r->stream));
  } catch (const CudaError& e) {
    r->err = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    r->err = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    r->err = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  return XRSEG_OK;
}

int xrseg_keep_indices(xrseg_runner* r, int32_t* idx, float* scores, int cap) {
  if (!r) return XRSEG_ERR_INVALID;
  int rc = finish(r);
  if (rc < 0) return rc;
  const int n = r->h_offsets[r->batch];
  if (cap < n) { r->err = "keep buffer too small"; return XRSEG_ERR_CAPACITY; }
  try {
    XR_CUDA(cudaSetDevice(r->device));
    if (idx && n) XR_CUDA(cudaMemcpyAsync(idx, r->o_anchor, sizeof(int) * n, cudaMemcpyDeviceToHost, r->stream));
    if (scores && n) XR_CUDA(cudaMemcpyAsync(scores, r->o_scores, sizeof(float) * n, cudaMemcpyDeviceToHost, r->stream));
    XR_CUDA(cudaStreamSynchronize(r->stream));
  } catch (const CudaError& e) {
    r->err = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    r->err = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    r->err = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  return n;
}

int xrseg_decode(xrseg_runner* r, float screen_w, float screen_h, int convention, xrseg_box* out, int cap, int* n_out) {
  if (!r || !out || !n_out || convention < 0 || convention > 2) return XRSEG_ERR_INVALID;
  int rc = finish(r);
  if (rc < 0) return rc;
  static_assert(sizeof(xrseg_box) == sizeof(BoxOut), "box layout");
  const int per_frame_cap = convention == XRSEG_BOX_PARSEBOXES ? 50 : (convention == XRSEG_BOX_DRAWBOXES ? 200 : 0);
  int total = 0;
  for (int b = 0; b < r->batch; ++b) total += per_frame_cap ? std::min(r->h_counts[b], per_frame_cap) : r->h_counts[b];
  *n_out = total;
  if (total == 0) return XRSEG_OK;
  if (cap < total) { r->err = "box buffer too small"; return XRSEG_ERR_CAPACITY; }
  try {
    XR_CUDA(cudaSetDevice(r->device));
    BoxOut* d_out = static_cast<BoxOut*>(ensure_scratch(r, sizeof(BoxOut) * total + 16));
    int* d_n = reinterpret_cast<int*>(reinterpret_cast<uint8_t*>(d_out) + sizeof(BoxOut) * total);
    boxes_to_screen_kernel<<<r->batch, 32, 0, r->stream>>>(r->o_boxes, r->o_labels, r->d_keep_n, r->d_offsets, r->batch,
                                                    convention, screen_w, screen_h, per_frame_cap, d_out, d_n);
    XR_CUDA(cudaMemcpyAsync(out, d_out, sizeof(BoxOut) * total, cudaMemcpyDeviceToHost, r->stream));
    XR_CUDA(cudaStreamSynchronize(r->stream));
  } catch (const CudaError& e) {
    r->err = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    r->err = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    r->err = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  return XRSEG_OK;
}

// Enqueues the mask kernels (and the device->host copy when out != NULL) on the runner's stream; sync = false leaves the
// synchronisation to the caller (xrseg_collect puts boxes, labels and masks behind ONE).
static int masks_enqueue(xrseg_runner* r, const xrseg_mask_params* mp, uint8_t* out, size_t cap_bytes, bool sync) {
  if (!r || !mp || mp->struct_size != sizeof(xrseg_mask_params)) return XRSEG_ERR_INVALID;
  int rc = finish(r);
  if (rc < 0) return rc;
  const int total = r->h_offsets[r->batch];
  const int first = mp->first;
  const int count = mp->count > 0 ? mp->count : total - first;
  if (first < 0 || count < 0 || first + count > total) { r->err = "mask range out of bounds"; return XRSEG_ERR_INVALID; }
  if (count == 0) return 0;
  size_t per = 0;
  switch (mp->mode) {
    case XRSEG_MASK_REFERENCE_160:
    case XRSEG_MASK_CROP_160: per = PROTO_PIX; break;
    case XRSEG_MASK_UPSAMPLE_640: per = 640 * 640; break;
    case XRSEG_MASK_BITS_160: per = PROTO_HW * 5 * 4; break;
    default: return XRSEG_ERR_INVALID;
  }
  if (out && cap_bytes < per * count) { r->err = "mask buffer too small"; return XRSEG_ERR_CAPACITY; }
  if (mp->mode == XRSEG_MASK_REFERENCE_160 &&
      (mp->image_w < 1 || mp->image_h < 1 || !(mp->screen_w > 0.f) || !(mp->screen_h > 0.f) ||
       mp->box_convention < 0 || mp->box_convention > 2)) {
    r->err = "xrseg_masks: REFERENCE_160 needs image_w/image_h >= 1, screen_w/screen_h > 0 and a box convention";
    return XRSEG_ERR_INVALID;
  }
  // threshold: 0 -> the runner's mask_threshold (IEE:32 _confidenceThreshold); a negative value asks for exactly 0
  const float thr = mp->threshold == 0.f ? r->cfg.mask_threshold : (mp->threshold < 0.f ? 0.f : mp->threshold);
  try {
    XR_CUDA(cudaSetDevice(r->device));
    uint8_t* d_out = static_cast<uint8_t*>(ensure_scratch(r, per * count));
    if (mp->mode == XRSEG_MASK_UPSAMPLE_640 && !r->mask_protos.ptr) {
      r->err = r->mask_protos.why;
      return XRSEG_ERR_STATE;
    }
    // gridDim.y / .z hold the detection index: at most 65535 per launch (batch 512 x 300 detections = 153600)
    for (int s0 = 0; s0 < count; s0 += 65535) {
      const int n = std::min(65535, count - s0);
      uint8_t* slice_out = d_out + per * s0;
      if (mp->mode == XRSEG_MASK_UPSAMPLE_640) {
        Mask640Params p{r->mask_protos.ptr, r->mask_protos.bstride, r->mask_protos.pitch, r->o_coefs, r->o_boxes,
                        r->o_frame, first + s0, slice_out,
                        thr <= 0.f ? -3.0e38f : (thr >= 1.f ? 3.0e38f : logf(thr / (1.f - thr)))};
        if (thr == 0.5f) p.logit_thr = 0.f;
        mask640_kernel<<<dim3(10, 10, n), 256, 0, r->stream>>>(p);
      } else {
        MaskThrParams p{};
        p.probs = r->o_probs; p.boxes = r->o_boxes; p.n = n; p.first = first + s0;
        p.mode = mp->mode == XRSEG_MASK_REFERENCE_160 ? 0 : 1;
        p.conv = mp->box_convention; p.sw = mp->screen_w; p.sh = mp->screen_h;
        p.image_w = mp->image_w; p.image_h = mp->image_h; p.thr = thr; p.out = slice_out;
        if (mp->mode == XRSEG_MASK_BITS_160)
          mask_bits_kernel<<<dim3(PROTO_HW, n), PROTO_HW, 0, r->stream>>>(p);
        else
          mask_threshold_kernel<<<dim3(PROTO_PIX / 256, n), 256, 0, r->stream>>>(p);
      }
    }
    XR_CUDA(cudaGetLastError());
    if (out) {   // out == NULL: the masks stay in the runner's device scratch (kernel timing, device-side consumers)
      XR_CUDA(cudaMemcpyAsync(out, d_out, per * count, cudaMemcpyDeviceToHost, r->stream));
      if (sync) XR_CUDA(cudaStreamSynchronize(r->stream));
    }
  } catch (const CudaError& e) {
    r->err = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    r->err = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    r->err = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  return count;
}

int xrseg_masks(xrseg_runner* r, const xrseg_mask_params* mp, uint8_t* out, size_t cap_bytes) {
  return masks_enqueue(r, mp, out, cap_bytes, true);
}

int xrseg_collect(xrseg_runner* r, float* boxes, int32_t* labels, int cap_dets, const xrseg_mask_params* mp, uint8_t* masks,
                  size_t masks_cap) {
  if (!r) return XRSEG_ERR_INVALID;
  int rc = finish(r);
  if (rc < 0) return rc;
  const int total = r->h_offsets[r->batch];
  if (total == 0) return 0;
  if ((boxes || labels) && cap_dets < total) { r->err = "xrseg_collect: detection buffers too small"; return XRSEG_ERR_CAPACITY; }
  try {
    XR_CUDA(cudaSetDevice(r->device));
    if (boxes) XR_CUDA(cudaMemcpyAsync(boxes, r->o_boxes, sizeof(float) * 4 * total, cudaMemcpyDeviceToHost, r->stream));
    if (labels) XR_CUDA(cudaMemcpyAsync(labels, r->o_labels, sizeof(int32_t) * total, cudaMemcpyDeviceToHost, r->stream));
  } catch (const CudaError& e) {
    r->err = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (...) {
    r->err = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  if (mp && masks) {
    rc = masks_enqueue(r, mp, masks, masks_cap, false);
    if (rc < 0) return rc;
  }
  if (cudaStreamSynchronize(r->stream) != cudaSuccess) { r->err = "xrseg_collect: synchronisation failed"; return XRSEG_ERR_CUDA; }
  return total;
}

int xrseg_extract_points(xrseg_runner* r, const xrseg_depth_params* dp, const uint16_t* depth_host, float* out_xyzd, int cap,
                         int* n_out) {
  if (!r || !dp || !depth_host || !out_xyzd || !n_out || dp->struct_size != sizeof(xrseg_depth_params)) return XRSEG_ERR_INVALID;
  int rc = finish(r);
  if (rc < 0) return rc;
  const int total = r->h_offsets[r->batch];
  const int step = dp->sampling_step > 0 ? dp->sampling_step : 5;
  const int max_points = dp->max_points > 0 ? dp->max_points : 8000;
  if (dp->detection < 0 || dp->detection >= total || dp->depth_w < 1 || dp->depth_h < 1 || step > PROTO_HW) {
    r->err = "xrseg_extract_points: bad detection index or depth geometry";
    return XRSEG_ERR_INVALID;
  }
  try {
    XR_CUDA(cudaSetDevice(r->device));
    const size_t depth_bytes = static_cast<size_t>(dp->depth_w) * dp->depth_h * sizeof(uint16_t);
    const size_t out_bytes = static_cast<size_t>(max_points) * sizeof(float4);
    uint8_t* base = static_cast<uint8_t*>(ensure_scratch(r, out_bytes + 16 + depth_bytes));
    DepthParams k{};
    k.out = reinterpret_cast<float4*>(base);
    k.out_n = reinterpret_cast<int*>(base + out_bytes);
    uint16_t* d_depth = reinterpret_cast<uint16_t*>(base + out_bytes + 16);
    XR_CUDA(cudaMemcpyAsync(d_depth, depth_host, depth_bytes, cudaMemcpyHostToDevice, r->stream));
    k.probs = r->o_probs + static_cast<size_t>(dp->detection) * PROTO_PIX;
    k.box = r->o_boxes + static_cast<size_t>(dp->detection) * 4;
    k.depth = d_depth;
    k.depth_w = dp->depth_w; k.depth_h = dp->depth_h; k.step = step; k.max_points = max_points;
    k.thr = dp->confidence_threshold > 0.f ? dp->confidence_threshold : r->cfg.mask_threshold;
    k.screen_w = dp->screen_w; k.screen_h = dp->screen_h;
    for (int i = 0; i < 3; ++i) k.pos[i] = dp->camera_position[i];
    for (int i = 0; i < 4; ++i) k.rot[i] = dp->camera_rotation[i];
    for (int i = 0; i < 2; ++i) { k.focal[i] = dp->focal_length[i]; k.principal[i] = dp->principal_point[i]; k.sensor[i] = dp->sensor_resolution[i]; }
    depth_extract_kernel<<<1, 1024, 0, r->stream>>>(k);
    XR_CUDA(cudaGetLastError());
    int n = 0;
    XR_CUDA(cudaMemcpyAsync(&n, k.out_n, sizeof(int), cudaMemcpyDeviceToHost, r->stream));
    XR_CUDA(cudaStreamSynchronize(r->stream));
    *n_out = n;
    if (n > cap) { r->err = "point buffer too small"; return XRSEG_ERR_CAPACITY; }
    if (n) XR_CUDA(cudaMemcpy(out_xyzd, k.out, static_cast<size_t>(n) * sizeof(float4), cudaMemcpyDeviceToHost));
  } catch (const CudaError& e) {
    r->err = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    r->err = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    r->err = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  return XRSEG_OK;
}

int xrseg_associate(xrseg_runner* r, int frame, float lx, float ly, int llabel, float screen_w, float screen_h, float max_dist,
                    int* best_index, float* best_dist) {
  if (!r || !best_index) return XRSEG_ERR_INVALID;
  int rc = finish(r);
  if (rc < 0) return rc;
  if (frame < 0 || frame >= r->batch) return XRSEG_ERR_INVALID;
  try {
    XR_CUDA(cudaSetDevice(r->device));
    uint8_t* base = static_cast<uint8_t*>(ensure_scratch(r, 16));
    int* d_idx = reinterpret_cast<int*>(base);
    float* d_dist = reinterpret_cast<float*>(base + 4);
    associate_kernel<<<1, 32, 0, r->stream>>>(r->o_boxes, r->o_labels, r->h_offsets[frame], r->h_counts[frame], 50, screen_w,
                                              screen_h, lx, ly, llabel, max_dist > 0.f ? max_dist : 300.f, d_idx, d_dist);
    XR_CUDA(cudaGetLastError());
    int idx = -1;
    float dist = 0.f;
    XR_CUDA(cudaMemcpyAsync(&idx, d_idx, sizeof(int), cudaMemcpyDeviceToHost, r->stream));
    XR_CUDA(cudaMemcpyAsync(&dist, d_dist, sizeof(float), cudaMemcpyDeviceToHost, r->stream));
    XR_CUDA(cudaStreamSynchronize(r->stream));
    *best_index = idx;
    if (best_dist) *best_dist = dist;
  } catch (const CudaError& e) {
    r->err = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    r->err = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    r->err = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  return XRSEG_OK;
}

int xrseg_last_timings(xrseg_runner* r, float* ms, int n) {
  if (!r || !ms) return XRSEG_ERR_INVALID;
  int rc = finish(r);
  if (rc < 0) return rc;
  for (int i = 0; i < n && i < 5; ++i) ms[i] = r->timings[i];
  return XRSEG_OK;
}

int xrseg_launch_count(xrseg_runner* r) { return r ? r->launches : XRSEG_ERR_INVALID; }

int xrseg_event_record(xrseg_runner* r, int slot) {
  if (!r || slot < 0 || slot >= 8) return XRSEG_ERR_INVALID;
  try {
    XR_CUDA(cudaSetDevice(r->device));
    if (!r->user_ev[slot]) XR_CUDA(cudaEventCreate(&r->user_ev[slot]));
    XR_CUDA(cudaEventRecord(r->user_ev[slot], r->stream));
  } catch (const CudaError& e) {
    r->err = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    r->err = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    r->err = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  return XRSEG_OK;
}

int xrseg_event_elapsed_ms(xrseg_runner* r, int a, int b, float* ms) {
  if (!r || !ms || a < 0 || a >= 8 || b < 0 || b >= 8 || !r->user_ev[a] || !r->user_ev[b]) return XRSEG_ERR_INVALID;
  try {
    XR_CUDA(cudaEventSynchronize(r->user_ev[b]));
    XR_CUDA(cudaEventElapsedTime(ms, r->user_ev[a], r->user_ev[b]));
  } catch (const CudaError& e) {
    r->err = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    r->err = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    r->err = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  return XRSEG_OK;
}

int xrseg_sync(xrseg_runner* r) {
  if (!r) return XRSEG_ERR_INVALID;
  cudaError_t e = cudaStreamSynchronize(r->stream);
  if (e != cudaSuccess) { r->err = cudaGetErrorString(e); return XRSEG_ERR_CUDA; }
  return XRSEG_OK;
}

int xrseg_profile_ops(xrseg_runner* r, int iters, float* ms, char* names, double* flops, double* bytes, int cap) {
  if (!r || !ms || iters < 1) return XRSEG_ERR_INVALID;
  int rc = finish(r);
  if (rc < 0) return rc;
  try {
    XR_CUDA(cudaSetDevice(r->device));
    const int nb = std::min(r->batch, r->mb);
    std::vector<Launch> ls;
    build_chunk_launches(r, 0, nb, ls);
    if (static_cast<int>(ls.size()) > cap) { r->err = "profile buffers too small"; return XRSEG_ERR_CAPACITY; }
    // One event pair per launch, whole pipeline per pass: every kernel sees exactly the data of a normal run
    // (replaying a single launch in a loop would re-apply the in-place residual convolutions of C2PSA).
    const size_t n = ls.size();
    std::vector<cudaEvent_t> ev(2 * n);
    for (auto& e : ev) XR_CUDA(cudaEventCreate(&e));
    std::vector<double> acc(n, 0.0);
    const int total_det = r->h_offsets[r->batch];
    for (int it = -1; it < iters; ++it) {   // pass -1 warms up
      reset_counters(r, nb, r->stream);
      for (size_t i = 0; i < n; ++i) {
        XR_CUDA(cudaEventRecord(ev[2 * i], r->stream));
        ls[i].fn(r->stream);
        XR_CUDA(cudaEventRecord(ev[2 * i + 1], r->stream));
      }
      XR_CUDA(cudaStreamSynchronize(r->stream));
      if (it < 0) continue;
      for (size_t i = 0; i < n; ++i) {
        float t = 0;
        XR_CUDA(cudaEventElapsedTime(&t, ev[2 * i], ev[2 * i + 1]));
        acc[i] += t;
      }
    }
    for (size_t i = 0; i < n; ++i) {
      ms[i] = static_cast<float>(acc[i] / iters);
      if (names) { memset(names + i * 32, 0, 32); strncpy(names + i * 32, ls[i].name.c_str(), 31); }
      double by = ls[i].bytes;
      if (ls[i].name == "post.mask_prob") by += static_cast<double>(total_det) * PROTO_PIX * 4;
      if (flops) flops[i] = ls[i].flops;
      if (bytes) bytes[i] = by;
    }
    XR_CUDA(cudaGetLastError());
    for (auto& e : ev) cudaEventDestroy(e);
    return static_cast<int>(ls.size());
  } catch (const CudaError& e) {
    r->err = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    r->err = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    r->err = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
}

// ---- debug / parity: exported by libxrseg_debug.so only (include/xrseg_debug.h) -----------------------------------------
#ifdef XRSEG_DEBUG_API
int xrseg_debug_fetch(xrseg_runner* r, const char* name, float* dst, size_t cap_floats, int64_t* shape4) {
  return xrseg_debug_fetch_frames(r, name, 0, -1, dst, cap_floats, shape4);
}

int xrseg_debug_fetch_frames(xrseg_runner* r, const char* name, int first, int count, float* dst, size_t cap_floats,
                             int64_t* shape4) {
  if (!r || !name || !dst || first < 0) return XRSEG_ERR_INVALID;
  int rc = finish(r);
  if (rc < 0) return rc;
  Net& net = *r->net;
  TV t;
  int C;
  std::string nm(name);
  // head tensors are fetched per scale: "box_logits.0" .. ; protos as a whole
  if (nm.rfind("box_logits.", 0) == 0) { t = net.box[nm.back() - '0']; }
  else if (nm.rfind("cls_logits.", 0) == 0) { t = net.cls[nm.back() - '0']; }
  else if (nm.rfind("coefs.", 0) == 0) { t = net.coef[nm.back() - '0']; }
  else if (nm == "protos") { t = net.protos; }
  else {
    auto it = net.named.find(nm);
    if (it == net.named.end()) { r->err = "unknown tensor " + nm; return XRSEG_ERR_INVALID; }
    t = it->second;
  }
  C = t.C;
  // the arena holds the LAST micro-batch of the run: frames (n_chunks - 1) * mb .. batch - 1
  const int resident = r->batch > 0 ? r->batch - (ceil_div(r->batch, r->mb) - 1) * r->mb : 0;
  if (count < 0) count = resident - first;
  if (count <= 0 || first + count > resident) { r->err = "no frames, or frames outside the resident chunk"; return XRSEG_ERR_INVALID; }
  const int nb = count;
  const size_t n = static_cast<size_t>(nb) * C * t.H * t.W;
  if (shape4) { shape4[0] = nb; shape4[1] = C; shape4[2] = t.H; shape4[3] = t.W; }
  if (cap_floats < n) { r->err = "fetch buffer too small"; return XRSEG_ERR_CAPACITY; }
  try {
    XR_CUDA(cudaSetDevice(r->device));
    float* d = dev_alloc<float>(n);
    const __half* src = ptr_of(r, t) + static_cast<size_t>(first) * t.H * t.W * t.pitch;
    nhwc_f16_to_nchw_f32_kernel<<<grid_for(static_cast<long>(n)), 256, 0, r->stream>>>(src, d, nb, C, t.H, t.W, t.pitch);
    XR_CUDA(cudaMemcpyAsync(dst, d, n * sizeof(float), cudaMemcpyDeviceToHost, r->stream));
    XR_CUDA(cudaStreamSynchronize(r->stream));
    cudaFree(d);
  } catch (const CudaError& e) {
    r->err = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    r->err = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    r->err = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  return XRSEG_OK;
}

int xrseg_debug_launches(xrseg_runner* r, int* grid, int* items, int* mode, char* names, int cap) {
  if (!r || !grid || !items || !mode) return XRSEG_ERR_INVALID;
  int rc = finish(r);
  if (rc < 0) return rc;
  if (r->batch < 1) { r->err = "no run"; return XRSEG_ERR_STATE; }
  const int b0 = (ceil_div(r->batch, r->mb) - 1) * r->mb, nb = r->batch - b0;
  const std::vector<Launch>* ls = nullptr;
  for (auto& c : r->launch_cache)
    if (c.b0 == b0 && c.nb == nb) ls = static_cast<const std::vector<Launch>*>(c.list);
  if (!ls) { r->err = "the last chunk ran without a launch list"; return XRSEG_ERR_STATE; }
  if (static_cast<int>(ls->size()) > cap) { r->err = "launch buffers too small"; return XRSEG_ERR_CAPACITY; }
  for (size_t i = 0; i < ls->size(); ++i) {
    const Launch& L = (*ls)[i];
    grid[i] = L.grid; items[i] = L.items; mode[i] = L.mode;
    if (names) { memset(names + i * 32, 0, 32); strncpy(names + i * 32, L.name.c_str(), 31); }
  }
  return static_cast<int>(ls->size());
}

static int debug_post_impl(xrseg_runner* r, const float* box_logits, const float* cls_logits, const float* coefs,
                           const float* protos, int batch, bool as_f16) {
  if (!r || !box_logits || !cls_logits || !coefs || !protos || batch < 1 || batch > r->cfg.max_batch)
    return XRSEG_ERR_INVALID;
  try {
    XR_CUDA(cudaSetDevice(r->device));
    const size_t A = r->A;
    const size_t B = r->cfg.max_batch;
    const size_t nc = r->nc, pitch = class_pitch(r->nc);      // caller rows [A, nc] -> device rows of `pitch` (padding stays 0)
    if (!r->dbg_box) {
      r->dbg_box = dev_alloc<float>(B * A * 64);
      r->dbg_cls = dev_alloc<float>(B * A * pitch);
      XR_CUDA(cudaMemset(r->dbg_cls, 0, sizeof(float) * B * A * pitch));
      r->dbg_coef = dev_alloc<float>(B * A * NM);
      r->dbg_proto = dev_alloc<float>(B * NM * PROTO_PIX);
    }
    cudaStream_t st = r->stream;
    XR_CUDA(cudaMemcpyAsync(r->dbg_box, box_logits, sizeof(float) * batch * A * 64, cudaMemcpyHostToDevice, st));
    XR_CUDA(cudaMemcpy2DAsync(r->dbg_cls, sizeof(float) * pitch, cls_logits, sizeof(float) * nc, sizeof(float) * nc, batch * A,
                              cudaMemcpyHostToDevice, st));
    XR_CUDA(cudaMemcpyAsync(r->dbg_coef, coefs, sizeof(float) * batch * A * NM, cudaMemcpyHostToDevice, st));
    XR_CUDA(cudaMemcpyAsync(r->dbg_proto, protos, sizeof(float) * batch * NM * PROTO_PIX, cudaMemcpyHostToDevice, st));
    r->batch = batch;
    r->timed = false;
    reset_counters(r, batch, st);
    std::vector<Launch> ls;
    if (as_f16) {
      // the product kernels (fp16 head tensors, NHWC prototypes, mma.sync mask assembly) on the caller's tensors
      const size_t nb_ = batch * A * 64, nc_ = batch * A * pitch, nm_ = batch * A * NM, np_ = static_cast<size_t>(batch) * NM * PROTO_PIX;
      if (!r->dbg_h16) r->dbg_h16 = dev_alloc<__half>(B * (A * (64 + pitch + NM) + static_cast<size_t>(NM) * PROTO_PIX));
      __half *hb = r->dbg_h16, *hc = hb + B * A * 64, *hm = hc + B * A * pitch, *hp = hm + B * A * NM;
      f32_to_f16_kernel<<<grid_for(static_cast<long>(nb_)), 256, 0, st>>>(r->dbg_box, hb, static_cast<long>(nb_));
      f32_to_f16_kernel<<<grid_for(static_cast<long>(nc_)), 256, 0, st>>>(r->dbg_cls, hc, static_cast<long>(nc_));
      f32_to_f16_kernel<<<grid_for(static_cast<long>(nm_)), 256, 0, st>>>(r->dbg_coef, hm, static_cast<long>(nm_));
      nchw_f32_to_nhwc_f16_kernel<<<grid_for(static_cast<long>(np_)), 256, 0, st>>>(r->dbg_proto, hp, batch, NM, 160, 160, NM, NM);
      ScaleSrc<__half> src[3];
      dense_scale_src<__half>(r, src, hb, hc, hm);
      add_post_launches<__half, false>(r, 0, batch, src, hp, static_cast<long>(NM) * PROTO_PIX, NM, true, false, ls);
      r->mask_protos = {hp, static_cast<long>(NM) * PROTO_PIX, NM, nullptr};
    } else {
      r->mask_protos = {nullptr, 0, 0, "640-px masks after xrseg_debug_post: its prototypes are fp32 planar, use xrseg_debug_post_f16"};
      ScaleSrc<float> src[3];
      dense_scale_src<float>(r, src, r->dbg_box, r->dbg_cls, r->dbg_coef);
      add_post_launches<float, true>(r, 0, batch, src, r->dbg_proto, static_cast<long>(NM) * PROTO_PIX, 0, true, false, ls);
    }
    if (getenv("XRSEG_DBG_TIME")) {
      // per-launch CUDA-event timing of the post-processing stage on these tensors (tools/bench_post.py): one untimed pass,
      // counters reset, then every launch between two events on the runner's stream
      for (Launch& l : ls) l.fn(st);
      std::vector<cudaEvent_t> ev(ls.size() + 1);
      for (auto& e : ev) XR_CUDA(cudaEventCreate(&e));
      reset_counters(r, batch, st);
      for (size_t i = 0; i < ls.size(); ++i) {
        XR_CUDA(cudaEventRecord(ev[i], st));
        ls[i].fn(st);
      }
      XR_CUDA(cudaEventRecord(ev[ls.size()], st));
      XR_CUDA(cudaStreamSynchronize(st));
      int kept = 0;
      std::vector<int> kn(batch);
      XR_CUDA(cudaMemcpy(kn.data(), r->d_keep_n, sizeof(int) * batch, cudaMemcpyDeviceToHost));
      for (int v : kn) kept += v;
      for (size_t i = 0; i < ls.size(); ++i) {
        float ms = 0;
        cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
        double bytes = ls[i].bytes;
        if (ls[i].name == "post.mask_prob") bytes += static_cast<double>(kept) * PROTO_PIX * sizeof(float);
        fprintf(stderr, "xrseg_debug_post: %-20s %8.1f us  %8.1f MB  %7.1f GB/s\n", ls[i].name.c_str(), ms * 1e3f, bytes / 1e6,
                bytes > 0 ? bytes / (ms * 1e6) : 0.0);
        if (i == 0) r->post_times.clear();
        r->post_times.push_back({ls[i].name, {ms, bytes}});
      }
      fprintf(stderr, "xrseg_debug_post: batch %d, %d detections kept\n", batch, kept);
      for (auto& e : ev) cudaEventDestroy(e);
    } else {
      for (Launch& l : ls) l.fn(st);
    }
    launch_k(add_frame_base_kernel, batch, 64, 0, st, r->o_frame, r->d_offsets, 0, batch);
    XR_CUDA(cudaGetLastError());
    XR_CUDA(cudaMemcpyAsync(r->h_offsets, r->d_offsets, sizeof(int) * (batch + 1), cudaMemcpyDeviceToHost, st));
    XR_CUDA(cudaMemcpyAsync(r->h_counts, r->d_keep_n, sizeof(int) * batch, cudaMemcpyDeviceToHost, st));
    XR_CUDA(cudaMemcpyAsync(r->h_overflow, r->d_overflow, sizeof(int), cudaMemcpyDeviceToHost, st));
    XR_CUDA(cudaEventRecord(r->ev_done, st));
    r->state = 1;
  } catch (const CudaError& e) {
    r->err = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    r->err = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    r->err = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  return XRSEG_OK;
}

// Per-launch CUDA-event times of the last xrseg_debug_post* call made with XRSEG_DBG_TIME set: ms[i], bytes[i]
// (algorithmic), names[i*32].  Returns the number of launches.
int xrseg_debug_post_timings(xrseg_runner* r, float* ms, double* bytes, char* names, int cap) {
  if (!r || !ms || !bytes || !names) return XRSEG_ERR_INVALID;
  const int n = static_cast<int>(r->post_times.size());
  if (n > cap) return XRSEG_ERR_CAPACITY;
  for (int i = 0; i < n; ++i) {
    ms[i] = r->post_times[i].second.first;
    bytes[i] = r->post_times[i].second.second;
    memset(names + i * 32, 0, 32);
    strncpy(names + i * 32, r->post_times[i].first.c_str(), 31);
  }
  return n;
}

int xrseg_debug_post(xrseg_runner* r, const float* box_logits, const float* cls_logits, const float* coefs,
                     const float* protos, int batch) {
  return debug_post_impl(r, box_logits, cls_logits, coefs, protos, batch, false);
}
int xrseg_debug_post_f16(xrseg_runner* r, const float* box_logits, const float* cls_logits, const float* coefs,
                         const float* protos, int batch) {
  return debug_post_impl(r, box_logits, cls_logits, coefs, protos, batch, true);
}

int xrseg_debug_nms(xrseg_runner* r, const float* corners, const float* scores, int batch, int num_anchors) {
  if (!r || !corners || !scores || batch < 1 || batch > r->cfg.max_batch || num_anchors != r->A) return XRSEG_ERR_INVALID;
  try {
    XR_CUDA(cudaSetDevice(r->device));
    const size_t A = r->A, B = r->cfg.max_batch;
    if (!r->dbg_corners) r->dbg_corners = dev_alloc<float>(B * A * 4);
    cudaStream_t st = r->stream;
    XR_CUDA(cudaMemcpyAsync(r->dbg_corners, corners, sizeof(float) * batch * A * 4, cudaMemcpyHostToDevice, st));
    XR_CUDA(cudaMemcpyAsync(r->d_scores, scores, sizeof(float) * batch * A, cudaMemcpyHostToDevice, st));
    XR_CUDA(cudaMemsetAsync(r->d_labels, 0, sizeof(int) * batch * A, st));
    XR_CUDA(cudaMemcpyAsync(r->d_boxes, r->dbg_corners, sizeof(float) * batch * A * 4, cudaMemcpyDeviceToDevice, st));
    r->batch = batch;
    r->timed = false;
    reset_counters(r, batch, st);
    scores_to_keys_kernel<<<dim3(ceil_div(static_cast<int>(A), 128), batch), 128, 0, st>>>(
        r->d_scores, batch, static_cast<int>(A), r->cfg.score_threshold, r->d_keys, r->d_cand_count);
    ScaleSrc<float> src[3] = {};
    std::vector<Launch> ls;
    add_post_launches<float, true>(r, 0, batch, src, nullptr, 0, 0, false, true, ls);
    for (Launch& l : ls) l.fn(st);
    XR_CUDA(cudaGetLastError());
    // anchors / scores of the kept boxes, compacted (no coefficient gather on this path)
    XR_CUDA(cudaMemcpyAsync(r->h_offsets, r->d_offsets, sizeof(int) * (batch + 1), cudaMemcpyDeviceToHost, st));
    XR_CUDA(cudaMemcpyAsync(r->h_counts, r->d_keep_n, sizeof(int) * batch, cudaMemcpyDeviceToHost, st));
    XR_CUDA(cudaMemcpyAsync(r->h_overflow, r->d_overflow, sizeof(int), cudaMemcpyDeviceToHost, st));
    XR_CUDA(cudaStreamSynchronize(st));
    std::vector<int> keep(static_cast<size_t>(batch) * r->max_det);
    XR_CUDA(cudaMemcpy(keep.data(), r->d_keep_idx, sizeof(int) * keep.size(), cudaMemcpyDeviceToHost));
    std::vector<int> flat;
    std::vector<float> fs;
    for (int b = 0; b < batch; ++b)
      for (int i = 0; i < r->h_counts[b]; ++i) {
        const int a = keep[static_cast<size_t>(b) * r->max_det + i];
        flat.push_back(a);
        fs.push_back(scores[static_cast<size_t>(b) * A + a]);
      }
    if (!flat.empty()) {
      XR_CUDA(cudaMemcpy(r->o_anchor, flat.data(), sizeof(int) * flat.size(), cudaMemcpyHostToDevice));
      XR_CUDA(cudaMemcpy(r->o_scores, fs.data(), sizeof(float) * fs.size(), cudaMemcpyHostToDevice));
    }
    XR_CUDA(cudaEventRecord(r->ev_done, st));
    r->state = 1;
  } catch (const CudaError& e) {
    r->err = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    r->err = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    r->err = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  return XRSEG_OK;
}

int xrseg_debug_mask_threshold(xrseg_runner* r, const float* probs, const float* boxes, int n, int image_w, int image_h,
                               float thr, uint8_t* out) {
  if (!r || !probs || !boxes || !out || n < 1) return XRSEG_ERR_INVALID;
  try {
    XR_CUDA(cudaSetDevice(r->device));
    float* d_p = dev_alloc<float>(static_cast<size_t>(n) * PROTO_PIX);
    float* d_b = dev_alloc<float>(static_cast<size_t>(n) * 4);
    uint8_t* d_o = dev_alloc<uint8_t>(static_cast<size_t>(n) * PROTO_PIX);
    XR_CUDA(cudaMemcpy(d_p, probs, sizeof(float) * n * PROTO_PIX, cudaMemcpyHostToDevice));
    XR_CUDA(cudaMemcpy(d_b, boxes, sizeof(float) * n * 4, cudaMemcpyHostToDevice));
    MaskThrParams p{};
    p.probs = d_p; p.boxes = d_b; p.n = n; p.first = 0; p.mode = 0; p.conv = -1;
    p.image_w = image_w; p.image_h = image_h; p.thr = thr; p.out = d_o;
    mask_threshold_kernel<<<dim3(PROTO_PIX / 256, n), 256, 0, r->stream>>>(p);
    XR_CUDA(cudaGetLastError());
    XR_CUDA(cudaStreamSynchronize(r->stream));
    XR_CUDA(cudaMemcpy(out, d_o, static_cast<size_t>(n) * PROTO_PIX, cudaMemcpyDeviceToHost));
    cudaFree(d_p); cudaFree(d_b); cudaFree(d_o);
  } catch (const CudaError& e) {
    r->err = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    r->err = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    r->err = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  return XRSEG_OK;
}

// One convolution through the selected engine (standalone: no runner needed).
int xrseg_debug_conv(int device, int impl, const float* x, int b, int cin, int h, int w, const float* wgt,
                     const float* bias, int cout, int k, int stride, int groups, int act, int transposed,
                     const float* residual, float* y, int variant) {
  if (!x || !wgt || !y || groups != 1) return XRSEG_ERR_INVALID;
  try {
    XR_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop{};
    XR_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) { g_create_error = "not an sm_100 device"; return XRSEG_ERR_NO_DEVICE; }
    conv_umma_prepare_device();
    const int cin_p = round_up(cin, 16), cout_p = round_up(cout, 16);
    const int ho = transposed ? h * 2 : (h + 2 * (k / 2) - k) / stride + 1;
    const int wo = transposed ? w * 2 : (w + 2 * (k / 2) - k) / stride + 1;
    const size_t nx = static_cast<size_t>(b) * cin * h * w, ny = static_cast<size_t>(b) * cout * ho * wo;
    float* d_x32 = dev_alloc<float>(nx);
    float* d_y32 = dev_alloc<float>(ny);
    float* d_r32 = residual ? dev_alloc<float>(ny) : nullptr;
    __half* d_x = dev_alloc<__half>(static_cast<size_t>(b) * h * w * cin_p);
    __half* d_y = dev_alloc<__half>(static_cast<size_t>(b) * ho * wo * cout_p);
    __half* d_r = residual ? dev_alloc<__half>(static_cast<size_t>(b) * ho * wo * cout_p) : nullptr;
    XR_CUDA(cudaMemcpy(d_x32, x, nx * sizeof(float), cudaMemcpyHostToDevice));
    nchw_f32_to_nhwc_f16_kernel<<<grid_for(static_cast<long>(b) * h * w * cin_p), 256>>>(d_x32, d_x, b, cin, h, w, cin_p, cin_p);
    if (residual) {
      XR_CUDA(cudaMemcpy(d_r32, residual, ny * sizeof(float), cudaMemcpyHostToDevice));
      nchw_f32_to_nhwc_f16_kernel<<<grid_for(static_cast<long>(b) * ho * wo * cout_p), 256>>>(d_r32, d_r, b, cout, ho, wo, cout_p, cout_p);
    }
    XR_CUDA(cudaMemset(d_y, 0, static_cast<size_t>(b) * ho * wo * cout_p * sizeof(__half)));
    std::vector<float> zero_bias(cout, 0.f);
    const float* hb = bias ? bias : zero_bias.data();
    __half* d_w = nullptr;
    float* d_b = nullptr;
    if (impl == XRSEG_CONV_UMMA) {
      ConvDesc cd{b, h, w, cin_p, cin_p, cout_p, cout_p, k, stride, act, transposed, residual ? cout_p : 0};
      ConvParams p;
      bool tma = (variant == 0 || variant == 4) && plan_conv_halo_tma(cd, prop.multiProcessorCount, p, variant == 0);
      const bool flat = !tma && variant == 0 && plan_conv_flat_tma(cd, prop.multiProcessorCount, p);
      const bool s2 = !tma && !flat && variant == 0 && plan_conv_s2_tma(cd, prop.multiProcessorCount, p);
      tma = tma || flat || s2;
      if (!tma) p = plan_conv(cd, prop.multiProcessorCount, variant & 1);
      std::vector<__half> wp;
      std::vector<float> bp;
      if (tma && p.sw) pack_conv_weights_sw<__half>(p, wgt, hb, cin, cout, wp, bp);
      else pack_conv_weights<__half>(p, wgt, hb, cin, cout, wp, bp);
      d_w = dev_upload(wp);
      d_b = dev_upload(bp);
      p.in = d_x; p.out = d_y; p.res = d_r; p.wpack = d_w; p.bias = d_b;
      const char* dbg = getenv("XRSEG_DBG_SKIP");
      if (dbg) p.dbg_skip = atoi(dbg);
      long long* d_clk = nullptr;
      if (getenv("XRSEG_DBG_TIME") && tma) {
        d_clk = dev_alloc<long long>(static_cast<size_t>(p.grid) * 12);
        XR_CUDA(cudaMemset(d_clk, 0, sizeof(long long) * p.grid * 12));
        p.dbg_clk = d_clk;
      }
      const int reps = getenv("XRSEG_DBG_TIME") ? 5 : 1;
      cudaEvent_t e0, e1;
      XR_CUDA(cudaEventCreate(&e0));
      XR_CUDA(cudaEventCreate(&e1));
      for (int rep = 0; rep < reps; ++rep) {
        if (rep == reps - 1) XR_CUDA(cudaEventRecord(e0, 0));
        if (tma) {
          conv_tma_prepare_device();
          TmapSet maps{};
          if (s2) maps = make_s2_tensor_maps(d_x, b, h, w, cin_p, cin_p, p);
          else maps.m[0] = flat ? make_flat_tensor_map(d_x, static_cast<long>(b) * h * w, cin_p, cin_p, p)
                                : make_halo_tensor_map(d_x, b, h, w, cin_p, cin_p, p.Wp, p.hbox, p.sw ? p.cb : 8, p.sw);
          launch_conv_halo_tma(p, maps, 0);
        } else {
          launch_conv_umma(p, 0);
        }
      }
      XR_CUDA(cudaEventRecord(e1, 0));
      XR_CUDA(cudaEventSynchronize(e1));
      if (reps > 1) {
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        fprintf(stderr, "xrseg_debug_conv: mode %d sw %d cb %d S %d nks %d nsub %d R %d grid %d smem %d tiles %d skip %d: %.1f us\n", p.mode, p.sw, p.cb,
                p.S, p.nks, p.nsub, p.R, p.grid, p.smem_bytes, p.m_tiles * p.n_tiles, p.dbg_skip, ms * 1e3f);
        if (d_clk) {
          std::vector<long long> h(static_cast<size_t>(p.grid) * 12);
          XR_CUDA(cudaMemcpy(h.data(), d_clk, sizeof(long long) * h.size(), cudaMemcpyDeviceToHost));
          const char* nm[12] = {"prod_wait_empty", "mma_wait_bres", "mma_wait_tempty", "mma_wait_full", "mma_issue", "mma_total",
                                "epi_wait_tfull", "epi_work", "mma_fence", "mma_commit", "mma_total_ns", "-"};
          for (int k = 0; k < 11; ++k) {
            double sum = 0;
            for (int c = 0; c < p.grid; ++c) sum += static_cast<double>(h[c * 12 + k]);
            fprintf(stderr, "   %-16s avg %.0f cycles per CTA (last of %d launches)\n", nm[k], sum / p.grid, reps);
          }
          cudaFree(d_clk);
        }
      }
      cudaEventDestroy(e0);
      cudaEventDestroy(e1);
    } else {
      const int taps = transposed ? 4 : k * k;
      std::vector<__half> wd(static_cast<size_t>(cout_p) * taps * cin_p, __half(0.f));
      std::vector<float> bs(cout_p, 0.f);
      for (int co = 0; co < cout; ++co) {
        bs[co] = hb[co];
        for (int ci = 0; ci < cin; ++ci)
          for (int t = 0; t < taps; ++t)
            if (transposed) wd[(static_cast<size_t>(t) * cout_p + co) * cin_p + ci] = __half(wgt[(static_cast<size_t>(ci) * cout + co) * 4 + t]);
            else wd[(static_cast<size_t>(co) * taps + t) * cin_p + ci] = __half(wgt[(static_cast<size_t>(co) * cin + ci) * taps + t]);
      }
      d_w = dev_upload(wd);
      d_b = dev_upload(bs);
      DirectParams p{};
      p.in = d_x; p.in_pitch = cin_p; p.out = d_y; p.out_pitch = cout_p; p.res = d_r; p.res_pitch = cout_p;
      p.w = d_w; p.bias = d_b; p.B = b; p.H = h; p.W = w; p.Cin = cin_p; p.Ho = ho; p.Wo = wo; p.Cout = cout_p;
      p.k = k; p.stride = stride; p.pad = k / 2; p.act = act; p.transposed = transposed;
      conv_direct_kernel<<<grid_for(static_cast<long>(b) * ho * wo * cout_p, 256, 148 * 32), 256>>>(p);
    }
    XR_CUDA(cudaGetLastError());
    nhwc_f16_to_nchw_f32_kernel<<<grid_for(static_cast<long>(ny)), 256>>>(d_y, d_y32, b, cout, ho, wo, cout_p);
    XR_CUDA(cudaDeviceSynchronize());
    XR_CUDA(cudaMemcpy(y, d_y32, ny * sizeof(float), cudaMemcpyDeviceToHost));
    cudaFree(d_x32); cudaFree(d_y32); cudaFree(d_r32); cudaFree(d_x); cudaFree(d_y); cudaFree(d_r); cudaFree(d_w); cudaFree(d_b);
  } catch (const CudaError& e) {
    g_create_error = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    g_create_error = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    g_create_error = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  return XRSEG_OK;
}

// The fused Bottleneck kernel on caller tensors (test hook): y = silu(conv3x3(silu(conv3x3(x, w1) + b1), w2) + b2) (+ x).
// x [b,c1,h,w], w1 [cm,c1,3,3], w2 [c2,cm,3,3], y [b,c2,h,w], all fp32 NCHW on the host.
int xrseg_debug_bottleneck(int device, const float* x, int b, int c1, int h, int w, const float* w1, const float* b1, int cm,
                           const float* w2, const float* b2, int c2, int residual, float* y) {
  if (!x || !w1 || !b1 || !w2 || !b2 || !y) return XRSEG_ERR_INVALID;
  try {
    XR_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop{};
    XR_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) { g_create_error = "not an sm_100 device"; return XRSEG_ERR_NO_DEVICE; }
    const int c1p = round_up(c1, 16), cmp = round_up(cm, 8), c2p = round_up(c2, 16);
    if (!bneck_supported(c1p, cmp, c2p) || (residual && c1 != c2)) { g_create_error = "unsupported channel triple"; return XRSEG_ERR_INVALID; }
    bneck_prepare_device();
    const size_t nx = static_cast<size_t>(b) * c1 * h * w, ny = static_cast<size_t>(b) * c2 * h * w;
    float* d_x32 = dev_alloc<float>(nx);
    float* d_y32 = dev_alloc<float>(ny);
    __half* d_x = dev_alloc<__half>(static_cast<size_t>(b) * h * w * c1p);
    __half* d_y = dev_alloc<__half>(static_cast<size_t>(b) * h * w * c2p);
    XR_CUDA(cudaMemcpy(d_x32, x, nx * sizeof(float), cudaMemcpyHostToDevice));
    nchw_f32_to_nhwc_f16_kernel<<<grid_for(static_cast<long>(b) * h * w * c1p), 256>>>(d_x32, d_x, b, c1, h, w, c1p, c1p);
    XR_CUDA(cudaMemset(d_y, 0, static_cast<size_t>(b) * h * w * c2p * sizeof(__half)));
    std::vector<uint32_t> f1, f2;
    pack_bneck_weights(w1, c1, cm, c1p, cmp, f1);
    pack_bneck_weights(w2, cm, c2, cmp, c2p, f2);
    std::vector<float> hb1(cmp, 0.f), hb2(c2p, 0.f);
    std::copy(b1, b1 + cm, hb1.begin());
    std::copy(b2, b2 + c2, hb2.begin());
    uint32_t *d_f1 = dev_upload(f1), *d_f2 = dev_upload(f2);
    float *d_b1 = dev_upload(hb1), *d_b2 = dev_upload(hb2);
    BneckParams p{};
    p.in = d_x; p.in_pitch = c1p; p.out = d_y; p.out_pitch = c2p;
    p.w1 = reinterpret_cast<uint2*>(d_f1); p.w2 = reinterpret_cast<uint2*>(d_f2); p.b1 = d_b1; p.b2 = d_b2;
    p.B = b; p.H = h; p.W = w;
    const int reps = getenv("XRSEG_DBG_TIME") ? 5 : 1;
    cudaEvent_t e0, e1;
    XR_CUDA(cudaEventCreate(&e0));
    XR_CUDA(cudaEventCreate(&e1));
    for (int rep = 0; rep < reps; ++rep) {
      if (rep == reps - 1) XR_CUDA(cudaEventRecord(e0, 0));
      launch_bneck(c1p, cmp, c2p, p, residual != 0, 0);
    }
    XR_CUDA(cudaEventRecord(e1, 0));
    XR_CUDA(cudaEventSynchronize(e1));
    XR_CUDA(cudaGetLastError());
    if (reps > 1) {
      float ms = 0;
      cudaEventElapsedTime(&ms, e0, e1);
      fprintf(stderr, "xrseg_debug_bottleneck: %d-%d-%d %dx%d batch %d: %.1f us\n", c1p, cmp, c2p, h, w, b, ms * 1e3f);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    nhwc_f16_to_nchw_f32_kernel<<<grid_for(static_cast<long>(ny)), 256>>>(d_y, d_y32, b, c2, h, w, c2p);
    XR_CUDA(cudaDeviceSynchronize());
    XR_CUDA(cudaMemcpy(y, d_y32, ny * sizeof(float), cudaMemcpyDeviceToHost));
    cudaFree(d_x32); cudaFree(d_y32); cudaFree(d_x); cudaFree(d_y); cudaFree(d_f1); cudaFree(d_f2); cudaFree(d_b1); cudaFree(d_b2);
  } catch (const CudaError& e) {
    g_create_error = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    g_create_error = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    g_create_error = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  return XRSEG_OK;
}

// Host-only: the B-fragment weight packing of the fused Bottleneck kernel (bottleneck.cuh), for CPU tests of the
// layout.  w [cout][cin][taps] fp32; out receives ceil(taps*C/16) * (N/8) * 64 words; returns the word count or < 0.
int xrseg_debug_pack_bneck(const float* w, int cin, int cout, int C, int N, int taps, uint32_t* out, size_t cap_words) {
  if (!w || !out || cin < 1 || cout < 1 || C < cin || C % 8 || N < cout || N % 8 || (taps != 1 && taps != 9)) return XRSEG_ERR_INVALID;
  std::vector<uint32_t> f;
  pack_bneck_weights(w, cin, cout, C, N, f, taps);
  if (f.size() > cap_words) return XRSEG_ERR_INVALID;
  memcpy(out, f.data(), f.size() * sizeof(uint32_t));
  return static_cast<int>(f.size());
}

// Host emulation of the UMMA kernel's data movement (test infrastructure; fp32; no GPU involved).
int xrseg_debug_emulate_conv(const float* x, int b, int cin, int h, int w, const float* wgt, const float* bias, int cout,
                             int k, int stride, int act, int transposed, const float* residual, float* y, int variant) {
  if (!x || !wgt || !y) return XRSEG_ERR_INVALID;
  try {
    const int cin_p = round_up(cin, 16), cout_p = round_up(cout, 16);
    const int ho = transposed ? h * 2 : (h + 2 * (k / 2) - k) / stride + 1;
    const int wo = transposed ? w * 2 : (w + 2 * (k / 2) - k) / stride + 1;
    ConvDesc cd{b, h, w, cin_p, cin_p, cout_p, cout_p, k, stride, act, transposed, residual ? cout_p : 0};
    ConvParams p;
    bool tma = (variant == 0 || variant == 4) && plan_conv_halo_tma(cd, 148, p, variant == 0);
    const bool flat = !tma && variant == 0 && plan_conv_flat_tma(cd, 148, p);
    const bool s2 = !tma && !flat && variant == 0 && plan_conv_s2_tma(cd, 148, p);
    tma = tma || flat || s2;
    if (!tma) p = plan_conv(cd, 148, variant & 1);
    std::vector<float> wp, bp;
    std::vector<float> zero_bias(cout, 0.f);
    if (tma && p.sw) pack_conv_weights_sw<float>(p, wgt, bias ? bias : zero_bias.data(), cin, cout, wp, bp);
    else pack_conv_weights<float>(p, wgt, bias ? bias : zero_bias.data(), cin, cout, wp, bp);
    std::vector<float> xin(static_cast<size_t>(b) * h * w * cin_p, 0.f), yo(static_cast<size_t>(b) * ho * wo * cout_p, 0.f), rr;
    for (int n = 0; n < b; ++n)
      for (int c = 0; c < cin; ++c)
        for (int i = 0; i < h * w; ++i) xin[(static_cast<size_t>(n) * h * w + i) * cin_p + c] = x[(static_cast<size_t>(n) * cin + c) * h * w + i];
    if (residual) {
      rr.assign(yo.size(), 0.f);
      for (int n = 0; n < b; ++n)
        for (int c = 0; c < cout; ++c)
          for (int i = 0; i < ho * wo; ++i) rr[(static_cast<size_t>(n) * ho * wo + i) * cout_p + c] = residual[(static_cast<size_t>(n) * cout + c) * ho * wo + i];
    }
    if (s2) {
      if (!emulate_conv_s2_tma(p, xin.data(), wp.data(), bp.data(), residual ? rr.data() : nullptr, yo.data())) {
        g_create_error = "s2 plan: a valid output reads outside its plane buffer";
        return XRSEG_ERR_INVALID;
      }
    } else if (flat) emulate_conv_flat_tma(p, xin.data(), wp.data(), bp.data(), residual ? rr.data() : nullptr, yo.data());
    else if (tma) emulate_conv_halo_tma(p, xin.data(), wp.data(), bp.data(), residual ? rr.data() : nullptr, yo.data());
    else emulate_conv_umma(p, xin.data(), wp.data(), bp.data(), residual ? rr.data() : nullptr, yo.data());
    for (int n = 0; n < b; ++n)
      for (int c = 0; c < cout; ++c)
        for (int i = 0; i < ho * wo; ++i) y[(static_cast<size_t>(n) * cout + c) * ho * wo + i] = yo[(static_cast<size_t>(n) * ho * wo + i) * cout_p + c];
  } catch (const CudaError& e) {
    g_create_error = e.msg;
    return XRSEG_ERR_INVALID;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    g_create_error = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_INVALID;
  } catch (...) {
    g_create_error = "unknown exception";
    return XRSEG_ERR_INVALID;
  }
  return XRSEG_OK;
}

// The C2PSA attention kernel alone (graph chains 160-168) on caller tensors: qkv f32 [b, n, heads*(32+32+64)] per token
// and head (query | key | value), out f32 [b, n, heads*64].
int xrseg_debug_attention(int device, const float* qkv, int b, int n, int heads, float* out, const float* pe_w, const float* pe_b,
                          int map_w) {
  if (!qkv || !out || b < 1 || heads < 1 || n < 16 || n % 16 || n % ATT_CHUNK || n / 16 > 26) return XRSEG_ERR_INVALID;
  if (pe_w && (!pe_b || map_w < 1 || n % map_w)) return XRSEG_ERR_INVALID;
  try {
    XR_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop{};
    XR_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) { g_create_error = "not an sm_100 device"; return XRSEG_ERR_NO_DEVICE; }
    XR_CUDA(cudaFuncSetAttribute(attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    const int cq = heads * (2 * ATT_KD + ATT_HD), co = heads * ATT_HD;
    const size_t nq = static_cast<size_t>(b) * n * cq, no = static_cast<size_t>(b) * n * co;
    float* d_q32 = dev_alloc<float>(nq);
    float* d_o32 = dev_alloc<float>(no);
    __half* d_q = dev_alloc<__half>(nq);
    __half* d_o = dev_alloc<__half>(no);
    XR_CUDA(cudaMemcpy(d_q32, qkv, nq * sizeof(float), cudaMemcpyHostToDevice));
    f32_to_f16_kernel<<<grid_for(static_cast<long>(nq)), 256>>>(d_q32, d_q, static_cast<long>(nq));
    AttnParams p{d_q, cq, d_o, co, b, n, heads, 1.0f / sqrtf(static_cast<float>(ATT_KD)), nullptr, nullptr, map_w > 0 ? map_w : n};
    float *d_pw = nullptr, *d_pb = nullptr;
    if (pe_w) {                                  // pe_w: [heads*64][3][3] (the depthwise layer's own layout) -> tap-major [9][C]
      std::vector<float> wt(static_cast<size_t>(9) * co), bt(pe_b, pe_b + co);
      for (int c = 0; c < co; ++c)
        for (int t = 0; t < 9; ++t) wt[static_cast<size_t>(t) * co + c] = pe_w[static_cast<size_t>(c) * 9 + t];
      d_pw = dev_upload(wt);
      d_pb = dev_upload(bt);
      p.pe_w = d_pw; p.pe_b = d_pb;
    }
    const size_t smem = static_cast<size_t>(n) * (ATT_KSTRIDE + ATT_VSTRIDE) * sizeof(__half);
    launch_k(attention_kernel, dim3(b * heads, ceil_div(n / 16, 13)), 13 * 32, smem, 0, p);
    XR_CUDA(cudaGetLastError());
    f16_to_f32_kernel<<<grid_for(static_cast<long>(no)), 256>>>(d_o, d_o32, static_cast<long>(no));
    XR_CUDA(cudaDeviceSynchronize());
    XR_CUDA(cudaMemcpy(out, d_o32, no * sizeof(float), cudaMemcpyDeviceToHost));
    cudaFree(d_q32); cudaFree(d_o32); cudaFree(d_q); cudaFree(d_o); cudaFree(d_pw); cudaFree(d_pb);
  } catch (const CudaError& e) {
    g_create_error = e.msg;
    return XRSEG_ERR_CUDA;
  } catch (const std::exception& e) {   // nothing may unwind across the C boundary
    g_create_error = std::string("unexpected exception: ") + e.what();
    return XRSEG_ERR_CUDA;
  } catch (...) {
    g_create_error = "unknown exception";
    return XRSEG_ERR_CUDA;
  }
  return XRSEG_OK;
}
#endif  // XRSEG_DEBUG_API

}  // extern "C"
