// model.cuh -- YOLO11-seg topology builder (n / s widths, any batch) and XRSW weight-pack reader.
//
// Restates the layer graph the reference runs (SURVEY.md Appendix A: the 499 chains of
// Assets/Resources/Model/yolo11n-seg-sentis.sentis, executed through IEExecutor.cs:371,397) as a list of kernel
// launches over NHWC fp16 buffers.  Concat / Split are channel-slice views of a shared buffer (no copies), residual
// Adds ride in the convolution epilogue, Swish is fused into every producing kernel.  Convolutions are emitted in
// the asset's chain order, which is the canonical layer order of the XRSW weight pack.
#pragma once

#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "common.cuh"
#include "conv_tma.cuh"
#include "conv_umma.cuh"

namespace xrseg {

struct TV {           // tensor view inside the activation arena (element offsets, resolved at launch)
  size_t off = 0;
  int B = 0, H = 0, W = 0, C = 0, Cp = 0, pitch = 0;
};

struct LayerRec {
  std::string name;
  int cin, cout, k, stride, groups, act, transposed, h_in, w_in;
};

enum OpKind { OP_STEM, OP_CONV, OP_DW, OP_SPPF, OP_UP, OP_ATTN, OP_BNECK };

struct Op {
  OpKind kind;
  int layer = -1;
  TV x, y, res;
  bool has_res = false;
  int k = 1, stride = 1, act = 0, transposed = 0, heads = 0;
  int in_grp = 0, in_grp_stride = 0, in_grp_off = 0;   // OP_DW channel remap (see DwParams)
  // Branch concurrency inside the captured graph: ops of branch > 0 (the head / proto chains) run on side streams.  The
  // first op of a branch segment waits for the event `wait_tag` (3/4/5 = P3/P4/P5 ready); the op producing that feature
  // map carries `signal_tag`.
  int branch = 0, wait_tag = 0, signal_tag = 0;
  // sibling fusion: a second convolution of the same input / kernel / stride / activation computed by the same launch
  // (OP_BNECK: the second 3x3 convolution of the fused Bottleneck, whose output is y)
  int layer2 = -1;
  TV y2;
  // fused trailing 1x1 convolution (conv_tma.cuh "tail"): the 1x1 layer `tail_layer` consumes this op's 64-channel output inside
  // the kernel; ytail is its destination (y stays the never-materialised intermediate)
  int tail_layer = -1, tail_act = 0;
  TV ytail;
  // merged leading ConvTranspose 2x2 / stride 2 (fuse_up_conv): x is that layer's input, the 3x3 `layer` runs on the
  // upsampled map without it ever existing
  int up_layer = -1;
};

// Channel triples (input, middle, output; as laid out in shared memory) the fused Bottleneck kernel is built for
// (bottleneck.cuh).  Anything else keeps its two tcgen05 launches.
static inline bool bneck_supported(int c1, int cm, int c2) {
  return (c1 == 16 && cm == 8 && c2 == 16) || (c1 == 32 && cm == 16 && c2 == 32);
}

// XRSEG_FLAT_TMA=0: keep the 1x1 convolutions on the thread-gather kernel (A/B measurements only)
static inline bool flat_tma_disabled() {
  const char* e = getenv("XRSEG_FLAT_TMA");
  return e && e[0] == '0';
}

struct Spec {
  int ch[5];
  int mid0, mid1;     // C3k2 output widths of layers 2 / 4 (n: 64 / 128)
  int cls_mid, box_mid, coef_mid, proto_mid, heads;
  int nc;             // classes: outputs of the three cls.2 convolutions
};

constexpr int NC_MIN = 1, NC_MAX = 1024;   // supported class counts (csrc/post.cuh sizes its decode paths for them)

// Channel pitch of the class-logit tensors: whole N tiles of the 1x1 convolution's TMA plan (conv_tma.cuh tma_n_split), so
// that every class count gets one.  round_up(nc, 16) up to 256 classes (one tile; 80 stays 80), else two or four equal
// tiles of a multiple of 16 channels (365 -> 2 x 192, 601 -> 4 x 160, 1024 -> 4 x 256).  The extra channels get zero
// weights and bias; the decode never reads past nc.
static inline int class_pitch(int nc) {
  int nt = 1;
  while (round_up(ceil_div(nc, nt), 16) > 256) nt *= 2;
  return nt * round_up(ceil_div(nc, nt), 16);
}

// The post-processing decode filter of a class tensor (xrseg_api.cu add_post_launches, tools/plan_dump sig): the kernel
// specialised for 80 classes (post.cuh NC), the segment-table kernel while a class row is at most 32 chunks of epc elements
// (16 bytes each), else the wide kernel.
enum { DECODE_80, DECODE_TABLE, DECODE_WIDE };
static inline int decode_variant(int nc, int pitch, int epc) {
  return nc == 80 ? DECODE_80 : (pitch / epc <= 32 ? DECODE_TABLE : DECODE_WIDE);
}

static inline Spec make_spec(int scale, int nc = 80) {
  const int wnum = (scale == 's') ? 2 : 1;  // width = wnum / 4
  Spec s;
  const int base[5] = {64, 128, 256, 512, 1024};
  for (int i = 0; i < 5; ++i) s.ch[i] = base[i] * wnum / 4;
  s.mid0 = 256 * wnum / 4;
  s.mid1 = 512 * wnum / 4;
  s.nc = nc;
  const int cls_floor = nc < 100 ? nc : 100;    // Ultralytics: c3 = max(ch[0], min(nc, 100))
  s.cls_mid = s.ch[2] > cls_floor ? s.ch[2] : cls_floor;
  s.box_mid = 64;
  if (s.ch[2] / 4 > s.box_mid) s.box_mid = s.ch[2] / 4;
  s.coef_mid = s.ch[2] / 4 > 32 ? s.ch[2] / 4 : 32;
  s.proto_mid = 256 * wnum / 4;
  s.heads = (s.ch[4] / 2) / 64;
  return s;
}

class Net {
 public:
  int B;
  Spec sp;
  std::vector<LayerRec> layers;
  std::vector<Op> ops;
  std::map<std::string, TV> named;
  size_t arena_elems = 0;
  int cur_branch = 0, pending_wait = 0;   // see Op::branch
  bool fuse_enabled = true;               // sibling fusion (fuse_siblings); off for the direct-convolution cross-check
  bool fuse_bneck = true;                 // Bottleneck fusion (fuse_bottlenecks)
  bool fuse_pe = true;                    // C2PSA positional encoding inside the attention kernel (fuse_attention_pe)
  bool fuse_tail = true;                  // proto.cv3 (1x1, 64 -> 32) inside proto.cv2's launch (fuse_tail_1x1)
  bool fuse_up = false;                   // proto.up inside that launch too (fuse_up_conv): requested by the caller, decided in build()
  TV input;                 // [B,640,640,4] fp16
  TV box[3], cls[3], coef[3], protos;
  int fh[3], fw[3];

  // up: merge proto.up into proto.cv2's launch where that is supported (fuse_up_conv).  The runner asks for it; the default is the
  // layer-per-launch list with only the sibling / Bottleneck / attention / tail fusions.
  Net(int scale, int batch, int in_hw = 640, bool fuse = true, bool bneck = true, int nc = 80, bool up = false)
      : B(batch), sp(make_spec(scale, nc)), fuse_enabled(fuse), fuse_bneck(fuse && bneck), fuse_tail(fuse), fuse_up(fuse && up) {
    XR_CHECK(nc >= NC_MIN && nc <= NC_MAX, "%d classes: supported are %d..%d", nc, NC_MIN, NC_MAX);
    build(in_hw);
  }

  TV alloc(int H, int W, int C, int pitch_override = 0) {
    TV t;
    t.B = B; t.H = H; t.W = W; t.C = C;
    t.Cp = pitch_override ? pitch_override : round_up(C, 16);
    t.pitch = t.Cp;
    t.off = arena_elems;
    arena_elems += static_cast<size_t>(B) * H * W * t.pitch;
    arena_elems = (arena_elems + 127) / 128 * 128;
    return t;
  }
  // A view that no launch reads or writes (an intermediate a fusion pass removes): shape only, an offset far outside the arena.
  static constexpr size_t NO_STORAGE = static_cast<size_t>(1) << 60;
  TV unallocated(int H, int W, int C, int id) const {
    TV t;
    t.B = B; t.H = H; t.W = W; t.C = C;
    t.Cp = t.pitch = round_up(C, 16);
    t.off = NO_STORAGE + static_cast<size_t>(id) * 128;
    return t;
  }
  int ops_reading_unallocated() const {
    int n = 0;
    for (const Op& o : ops) {
      const bool tail = o.tail_layer >= 0;    // a fused tail's y is its never-materialised intermediate
      n += o.x.off >= NO_STORAGE || (!tail && o.y.off >= NO_STORAGE) || (o.has_res && o.res.off >= NO_STORAGE) ||
           (o.layer2 >= 0 && o.y2.off >= NO_STORAGE) || (tail && o.ytail.off >= NO_STORAGE);
    }
    return n;
  }
  static TV slice(const TV& t, int c0, int c) {
    XR_CHECK(c0 % 16 == 0 && c % 16 == 0 && c0 + c <= t.Cp, "bad slice %d+%d of %d", c0, c, t.Cp);
    TV s = t;
    s.off = t.off + c0;
    s.C = c;
    s.Cp = c;
    return s;
  }

  TV conv(const TV& x, int cout, int k, int s, bool act, const std::string& name, const TV* dst = nullptr,
          const TV* res = nullptr, bool transposed = false) {
    LayerRec l{name, x.C, cout, k, s, 1, act ? 1 : 0, transposed ? 1 : 0, x.H, x.W};
    layers.push_back(l);
    const int Ho = transposed ? x.H * 2 : (x.H + 2 * (k / 2) - k) / s + 1;
    const int Wo = transposed ? x.W * 2 : (x.W + 2 * (k / 2) - k) / s + 1;
    TV y = dst ? *dst : alloc(Ho, Wo, cout);
    XR_CHECK(y.H == Ho && y.W == Wo && y.C == cout, "conv %s: destination mismatch", name.c_str());
    Op o;
    o.kind = layers.size() == 1 ? OP_STEM : OP_CONV;
    o.layer = static_cast<int>(layers.size()) - 1;
    o.x = x; o.y = y; o.k = k; o.stride = s; o.act = act; o.transposed = transposed;
    if (res) { o.res = *res; o.has_res = true; }
    o.branch = cur_branch; o.wait_tag = pending_wait; pending_wait = 0;
    ops.push_back(o);
    named[name] = y;
    return y;
  }
  // grp > 0: the conv's C = n_grp * grp input channels are read from x at (c / grp) * grp_stride + grp_off + c % grp
  TV dw(const TV& x, bool act, const std::string& name, const TV* res = nullptr, int grp = 0, int grp_stride = 0,
        int grp_off = 0, int n_grp = 0) {
    const int C = grp > 0 ? grp * n_grp : x.C;
    LayerRec l{name, C, C, 3, 1, C, act ? 1 : 0, 0, x.H, x.W};
    layers.push_back(l);
    TV y = alloc(x.H, x.W, C);
    Op o;
    o.kind = OP_DW;
    o.layer = static_cast<int>(layers.size()) - 1;
    o.x = x; o.y = y; o.k = 3; o.act = act;
    o.in_grp = grp; o.in_grp_stride = grp_stride; o.in_grp_off = grp_off;
    if (res) { o.res = *res; o.has_res = true; }
    o.branch = cur_branch; o.wait_tag = pending_wait; pending_wait = 0;
    ops.push_back(o);
    named[name] = y;
    return y;
  }

  TV c3k2(const TV& x, int c_out, int c, bool c3k, const std::string& n, const TV* dst = nullptr) {
    TV cat = alloc(x.H, x.W, 3 * c);
    TV ab = slice(cat, 0, 2 * c);
    conv(x, 2 * c, 1, 1, true, n + ".cv1", &ab);
    TV b = slice(cat, c, c);
    TV m = slice(cat, 2 * c, c);
    if (!c3k) {
      TV t = conv(b, c / 2, 3, 1, true, n + ".m0.cv1");
      conv(t, c, 3, 1, true, n + ".m0.cv2", &m, &b);
    } else {
      const int c_ = c / 2;
      TV cat2 = alloc(x.H, x.W, 2 * c_);
      TV t0 = conv(b, c_, 1, 1, true, n + ".m0.cv1");
      TV h = conv(t0, c_, 3, 1, true, n + ".m0.m0.cv1");
      TV t1 = conv(h, c_, 3, 1, true, n + ".m0.m0.cv2", nullptr, &t0);
      h = conv(t1, c_, 3, 1, true, n + ".m0.m1.cv1");
      TV t2 = slice(cat2, 0, c_);
      conv(h, c_, 3, 1, true, n + ".m0.m1.cv2", &t2, &t1);
      TV u = slice(cat2, c_, c_);
      conv(b, c_, 1, 1, true, n + ".m0.cv2", &u);
      conv(cat2, c, 1, 1, true, n + ".m0.cv3", &m);
    }
    return conv(cat, c_out, 1, 1, true, n + ".cv2", dst);
  }

  void head_box_cls(const TV& p, int i, const std::string& n) {
    cur_branch = 1; pending_wait = 3 + i;            // box chain: side stream 1, after P(3+i)
    TV t = conv(p, sp.box_mid, 3, 1, true, n + ".box.0");
    t = conv(t, sp.box_mid, 3, 1, true, n + ".box.1");
    box[i] = conv(t, 64, 1, 1, false, n + ".box.2");
    cur_branch = 2; pending_wait = 3 + i;            // class chain: side stream 2
    t = dw(p, true, n + ".cls.0dw");
    t = conv(t, sp.cls_mid, 1, 1, true, n + ".cls.0pw");
    t = dw(t, true, n + ".cls.1dw");
    t = conv(t, sp.cls_mid, 1, 1, true, n + ".cls.1pw");
    TV logits = alloc(t.H, t.W, sp.nc, class_pitch(sp.nc));
    cls[i] = conv(t, sp.nc, 1, 1, false, n + ".cls.2", &logits);
    cur_branch = 0;
  }
  void head_coef(const TV& p, int i, const std::string& n) {
    cur_branch = 3; pending_wait = 3 + i;            // coefficient chain: side stream 3
    TV t = conv(p, sp.coef_mid, 3, 1, true, n + ".coef.0");
    t = conv(t, sp.coef_mid, 3, 1, true, n + ".coef.1");
    coef[i] = conv(t, 32, 1, 1, false, n + ".coef.2");
    cur_branch = 0;
  }

  // Two convolutions that read the same tensor with the same kernel / stride / activation and no residual become one
  // launch with N = Cout_a + Cout_b (the input is read once, one launch less): the two 1x1 convs at the head of every
  // C3k block (m0.cv1 | m0.cv2) and the first 3x3 of the box and coefficient branches of every scale (box.0 | coef.0).
  // The second op disappears from `ops`; its consumers wait for the fused launch through event tag 6 + pair index.
  void fuse_siblings() {
    if (!fuse_enabled) return;
    auto find = [&](const std::string& nm) {
      for (size_t i = 0; i < ops.size(); ++i)
        if (ops[i].layer >= 0 && layers[ops[i].layer].name == nm) return static_cast<int>(i);
      return -1;
    };
    std::vector<std::pair<std::string, std::string>> pairs;
    for (const char* blk : {"b6", "b8", "n22"}) pairs.push_back({std::string(blk) + ".m0.cv1", std::string(blk) + ".m0.cv2"});
    for (const char* h : {"h3", "h4", "h5"}) pairs.push_back({std::string(h) + ".box.0", std::string(h) + ".coef.0"});
    int tag = 6;
    for (const auto& pr : pairs) {
      const int ia = find(pr.first), ib = find(pr.second);
      if (ia < 0 || ib < 0) continue;
      // a fused pair needs a TMA plan (xrseg_api.cu upload_layers): with the flat TMA planner off, 1x1 pairs keep two launches
      if (ops[ia].k == 1 && flat_tma_disabled()) continue;
      Op& a = ops[ia];
      const Op b = ops[ib];
      const bool same = a.kind == OP_CONV && b.kind == OP_CONV && a.x.off == b.x.off && a.x.C == b.x.C && a.x.pitch == b.x.pitch &&
                        a.k == b.k && a.stride == b.stride && a.act == b.act && !a.has_res && !b.has_res && !a.transposed &&
                        !b.transposed && a.layer2 < 0 && a.y.Cp + b.y.Cp <= 256;
      if (!same) continue;
      a.layer2 = b.layer;
      a.y2 = b.y;
      if (a.branch != b.branch) {
        // the consumer chain of b runs on another stream: it must wait for the fused launch (which runs on a's stream)
        a.signal_tag = tag;
        for (size_t j = ib + 1; j < ops.size(); ++j)
          if (ops[j].branch == b.branch) {           // first later op of b's branch = b's consumer
            if (ops[j].wait_tag == 0) ops[j].wait_tag = tag;
            break;
          }
        ++tag;
      }
      ops.erase(ops.begin() + ib);
    }
  }

  // A 3x3 convolution whose ONLY consumer is a 1x1 convolution (rows are independent for a 1x1) runs that 1x1 inside its own
  // launch as a second set of MMAs on the epilogue's fp16 tile kept in tensor memory (ConvParams::tail_n, conv_tma.cuh): the
  // intermediate tensor is never written to HBM or read back.  The one pair is proto.cv2 (64) -> proto.cv3 (32), in place (512
  // accumulator columns are all in use).  The stride-2 stage pairs b1 -> b2.cv1 and b3 -> b4.cv1 were measured too: 76 + 43 ->
  // 113 us and 66 + 27 -> 88 us, frames/s unchanged -- these layers are bound by their epilogue, and two epilogue passes in one
  // launch cost what the second launch did.  Anything else keeps its two launches.
  static bool tail_env_on() {
    static const bool on = [] { const char* e = getenv("XRSEG_FUSE_TAIL"); return !(e && e[0] == '0'); }();
    return on;
  }
  void fuse_tail_1x1() {
    if (!fuse_tail || !tail_env_on()) return;
    for (size_t i = 0; i + 1 < ops.size(); ++i) {
      Op& a = ops[i];
      const Op b = ops[i + 1];
      if (a.kind != OP_CONV || b.kind != OP_CONV || a.layer2 >= 0 || b.layer2 >= 0 || a.tail_layer >= 0) continue;
      const std::string &na = layers[a.layer].name, &nb = layers[b.layer].name;
      const bool proto = na == "proto.cv2" && nb == "proto.cv3" && a.stride == 1 && a.y.Cp == 64 && b.y.Cp == 32;
      if (!proto) continue;
      const bool ok = a.k == 3 && !a.transposed && a.act && !a.has_res && b.k == 1 && b.stride == 1 && !b.transposed && !b.has_res &&
                      b.x.off == a.y.off && b.x.pitch == a.y.pitch && b.x.Cp == a.y.Cp && a.branch == b.branch && b.wait_tag == 0 &&
                      a.signal_tag == 0;
      if (!ok) continue;
      a.tail_layer = b.layer;
      a.tail_act = b.act;
      a.ytail = b.y;
      a.signal_tag = b.signal_tag;
      ops.erase(ops.begin() + i + 1);
    }
  }

  // proto.up (ConvTranspose 2x2 / stride 2, bias, no activation) -> proto.cv2 (3x3, SiLU) is exact linear algebra before the
  // SiLU: for each output parity (dy, dx) it is a 2x2-tap convolution of the 80x80 map with merged weights (K per output
  // pixel 256 instead of 576), plus a bias that depends on which of cv2's taps fall inside the 160x160 map (conv_tma.cuh
  // merge_upconv_weights).  The pair becomes one OP_CONV on the 80x80 map: layer = cv2, up_layer = up, x = up's input.  Only
  // with the fused proto.cv3 tail (the kernel's parity-scatter epilogue is the tail's) and only for 64 channels (the n scale;
  // the s scale's 128 would need four N tiles).  build() decides it up front (fuse_up) so that neither 160x160x64 map is
  // allocated; XRSEG_FUSE_UP=0 (or XRSEG_FUSE_TAIL=0) keeps the three launches.
  void fuse_up_conv() {
    if (!fuse_up) return;
    bool done = false;
    for (size_t i = 0; i + 1 < ops.size(); ++i) {
      Op& a = ops[i];
      const Op b = ops[i + 1];
      if (a.kind != OP_CONV || b.kind != OP_CONV || layers[a.layer].name != "proto.up" || layers[b.layer].name != "proto.cv2") continue;
      const bool ok = a.transposed && a.k == 2 && a.stride == 2 && !a.act && !a.has_res && a.layer2 < 0 && a.tail_layer < 0 &&
                      b.k == 3 && b.stride == 1 && !b.transposed && !b.has_res && b.layer2 < 0 && b.x.off == a.y.off &&
                      a.x.Cp == 64 && b.y.Cp == 64 && a.y.Cp == 64 && a.branch == b.branch && b.wait_tag == 0 && a.signal_tag == 0;
      XR_CHECK(ok, "proto.up -> proto.cv2 cannot be merged");
      for (size_t j = 0; j < ops.size(); ++j)   // up's only consumer is cv2
        XR_CHECK(j == i || j == i + 1 || (ops[j].x.off != a.y.off && !(ops[j].has_res && ops[j].res.off == a.y.off)),
                 "proto.up has a second consumer");
      const int wait = a.wait_tag;
      ops[i + 1].up_layer = a.layer;
      ops[i + 1].x = a.x;
      ops[i + 1].wait_tag = wait;
      ops.erase(ops.begin() + i);
      done = true;
      break;
    }
    XR_CHECK(done, "proto.up / proto.cv2 not found for the merge");
    named.erase("proto.up");                  // never materialised
    named.erase("proto.cv2");
  }

  // C2PSA: x = attention(q, k, v) + pe(v).  The depthwise 3x3 `attn.pe` reads V in place from the qkv tensor and adds the
  // attention output as its residual; the attention kernel already holds the head's V map in shared memory, so the pair
  // becomes one OP_ATTN launch: layer = the pe layer (its weights), y = the pe op's destination.
  void fuse_attention_pe() {
    static const bool env_on = [] { const char* e = getenv("XRSEG_FUSE_PE"); return !(e && e[0] == '0'); }();
    if (!fuse_pe || !env_on) return;
    for (size_t i = 0; i + 1 < ops.size(); ++i) {
      Op& a = ops[i];
      const Op b = ops[i + 1];
      if (a.kind != OP_ATTN || b.kind != OP_DW || a.layer >= 0) continue;
      const bool ok = b.in_grp > 0 && b.x.off == a.x.off && b.has_res && b.res.off == a.y.off && !b.act && a.branch == b.branch &&
                      b.wait_tag == 0 && a.signal_tag == 0;
      if (!ok) continue;
      a.layer = b.layer;
      a.y = b.y;
      a.signal_tag = b.signal_tag;
      ops.erase(ops.begin() + i + 1);
    }
  }

  // The Bottleneck of a C3k2 block without C3k (X.m0.cv1 -> X.m0.cv2 (+ x)): two dependent 3x3 convolutions over 8..32
  // channels become one launch whose intermediate stays in shared memory (bottleneck.cuh).  The pair collapses into one
  // OP_BNECK op: layer = cv1, layer2 = cv2, x = the block input (also the residual), y = cv2's destination.
  void fuse_bottlenecks() {
    if (!fuse_bneck) return;
    for (size_t i = 0; i + 1 < ops.size(); ++i) {
      Op& a = ops[i];
      const Op b = ops[i + 1];
      if (a.kind != OP_CONV || b.kind != OP_CONV || a.layer2 >= 0 || b.layer2 >= 0) continue;
      const std::string &na = layers[a.layer].name, &nb = layers[b.layer].name;
      const bool names = na.size() > 7 && na.compare(na.size() - 7, 7, ".m0.cv1") == 0 && nb == na.substr(0, na.size() - 1) + "2";
      if (!names) continue;
      const bool chain = a.k == 3 && b.k == 3 && a.stride == 1 && b.stride == 1 && a.act && b.act && !a.has_res &&
                         !a.transposed && !b.transposed && b.x.off == a.y.off && a.branch == b.branch && b.wait_tag == 0 &&
                         a.signal_tag == 0 && (!b.has_res || (b.res.off == a.x.off && b.res.pitch == a.x.pitch));
      const int cm = round_up(layers[a.layer].cout, 8);
      if (!chain || !bneck_supported(a.x.Cp, cm, b.y.Cp) || (b.has_res && a.x.Cp != b.y.Cp)) continue;
      a.kind = OP_BNECK;
      a.layer2 = b.layer;
      a.y = b.y;
      a.has_res = b.has_res;
      a.res = b.res;
      a.signal_tag = b.signal_tag;
      ops.erase(ops.begin() + i + 1);
    }
  }

  void build(int hw) {
    const int c1 = sp.ch[0], c2 = sp.ch[1], c5 = sp.ch[4];
    input = alloc(hw, hw, 3, 4);
    named["input"] = input;
    const int h8 = hw / 8, h16 = hw / 16, h32 = hw / 32;
    // concat buffers of the neck, allocated first so that backbone outputs land directly in their slices
    TV cat13 = alloc(h16, h16, c5 + sp.mid1);        // [up(f10) | f6]
    TV cat16 = alloc(h8, h8, sp.mid1 + sp.mid1);     // [up(f13) | f4]
    TV cat19 = alloc(h16, h16, sp.mid0 + sp.mid1);   // [n17 | f13]
    TV cat22 = alloc(h32, h32, sp.mid1 + c5);        // [n20 | f10]

    TV t = conv(input, c1, 3, 2, true, "b0");
    t = conv(t, c2, 3, 2, true, "b1");
    t = c3k2(t, sp.mid0, sp.mid0 / 4, false, "b2");
    t = conv(t, sp.mid0, 3, 2, true, "b3");
    TV f4 = slice(cat16, sp.mid1, sp.mid1);
    c3k2(t, sp.mid1, sp.mid1 / 4, false, "b4", &f4);
    t = conv(f4, sp.mid1, 3, 2, true, "b5");
    TV f6 = slice(cat13, c5, sp.mid1);
    c3k2(t, sp.mid1, sp.mid1 / 2, true, "b6", &f6);
    t = conv(f6, c5, 3, 2, true, "b7");
    t = c3k2(t, c5, c5 / 2, true, "b8");
    {  // SPPF (chains 140-151)
      const int c_ = c5 / 2;
      TV cat = alloc(h32, h32, 4 * c_);
      TV y0 = slice(cat, 0, c_);
      conv(t, c_, 1, 1, true, "b9.cv1", &y0);
      named["b9.pool"] = slice(cat, c_, 3 * c_);   // fetch-only name: the three max-pool outputs
      Op o;
      o.kind = OP_SPPF;
      o.x = cat; o.y = cat;
      ops.push_back(o);
      t = conv(cat, c5, 1, 1, true, "b9.cv2");
    }
    TV f10 = slice(cat22, sp.mid1, c5);
    {  // C2PSA (chains 152-190)
      const int c = c5 / 2;
      const int kd = 32, hd = 64;
      XR_CHECK(c / sp.heads == hd, "attention head dim must be 64");
      TV cat = alloc(h32, h32, 2 * c);
      conv(t, 2 * c, 1, 1, true, "b10.cv1", &cat);
      TV b = slice(cat, c, c);
      TV qkv = conv(b, c + 2 * sp.heads * kd, 1, 1, false, "b10.attn.qkv");
      TV ao = alloc(h32, h32, c);
      Op oa;
      oa.kind = OP_ATTN; oa.x = qkv; oa.y = ao; oa.heads = sp.heads;
      ops.push_back(oa);
      // pe(v) + attention output; V is read in place from qkv (per head: kd query, kd key, hd value channels)
      TV s = dw(qkv, false, "b10.attn.pe", &ao, hd, 2 * kd + hd, 2 * kd, sp.heads);
      conv(s, c, 1, 1, false, "b10.attn.proj", &b, &b);              // b += proj(...)
      TV f = conv(b, 2 * c, 1, 1, true, "b10.ffn.0");
      conv(f, c, 1, 1, false, "b10.ffn.1", &b, &b);                  // b += ffn(b)
      conv(cat, c5, 1, 1, true, "b10.cv2", &f10);
    }
    auto upsample = [&](const TV& src, const TV& dst, const char* name) {
      Op o;
      o.kind = OP_UP; o.x = src; o.y = dst;
      ops.push_back(o);
      named[name] = dst;                        // fetch-only name of the concat slice it fills
    };
    upsample(f10, slice(cat13, 0, c5), "up.13");
    TV f13 = slice(cat19, sp.mid0, sp.mid1);
    c3k2(cat13, sp.mid1, sp.mid1 / 2, false, "n13", &f13);
    upsample(f13, slice(cat16, 0, sp.mid1), "up.16");
    TV p3 = c3k2(cat16, sp.mid0, sp.mid0 / 2, false, "n16");
    ops.back().signal_tag = 3;
    head_box_cls(p3, 0, "h3");
    TV n17 = slice(cat19, 0, sp.mid0);
    conv(p3, sp.mid0, 3, 2, true, "n17", &n17);
    TV p4 = c3k2(cat19, sp.mid1, sp.mid1 / 2, false, "n19");
    ops.back().signal_tag = 4;
    head_box_cls(p4, 1, "h4");
    TV n20 = slice(cat22, 0, sp.mid1);
    conv(p4, sp.mid1, 3, 2, true, "n20", &n20);
    TV p5 = c3k2(cat22, c5, c5 / 2, true, "n22");
    ops.back().signal_tag = 5;
    head_box_cls(p5, 2, "h5");
    head_coef(p3, 0, "h3");
    head_coef(p4, 1, "h4");
    head_coef(p5, 2, "h5");
    cur_branch = 4; pending_wait = 3;                // prototype chain: side stream 4, after P3
    t = conv(p3, sp.proto_mid, 3, 1, true, "proto.cv1");
    {
      // proto.up + proto.cv2 (+ cv3) as one launch (fuse_up_conv): the two 160x160 maps get no storage
      const char* e = getenv("XRSEG_FUSE_UP");
      fuse_up = fuse_up && fuse_tail && tail_env_on() && !(e && e[0] == '0') && sp.proto_mid == 64 && t.W + 2 <= 256;
      TV up_y = unallocated(2 * t.H, 2 * t.W, sp.proto_mid, 0), cv2_y = unallocated(2 * t.H, 2 * t.W, sp.proto_mid, 1);
      t = conv(t, sp.proto_mid, 2, 2, false, "proto.up", fuse_up ? &up_y : nullptr, nullptr, true);
      t = conv(t, sp.proto_mid, 3, 1, true, "proto.cv2", fuse_up ? &cv2_y : nullptr);
    }
    protos = conv(t, 32, 1, 1, true, "proto.cv3");
    cur_branch = 0;
    named["p3"] = p3; named["p4"] = p4; named["p5"] = p5;
    fuse_siblings();
    fuse_bottlenecks();
    fuse_attention_pe();
    fuse_up_conv();
    fuse_tail_1x1();
    XR_CHECK(!fuse_up || ops_reading_unallocated() == 0, "a launch touches a tensor without storage");
    fh[0] = p3.H; fw[0] = p3.W; fh[1] = p4.H; fw[1] = p4.W; fh[2] = p5.H; fw[2] = p5.W;
  }
};

// ---------------------------------------------------------------------------------------------------------------
// A convolution launch's parameters.  The runner (xrseg_api.cu) and tools/plan_dump both derive them here, so that a
// listing of the plans cannot drift from what the runner launches.
// ---------------------------------------------------------------------------------------------------------------
// XRSEG_S2_TMA=0: keep the stride-2 3x3 convolutions on the thread-gather kernel (A/B measurements only)
static inline bool s2_tma_disabled() {
  const char* e = getenv("XRSEG_S2_TMA");
  return e && e[0] == '0';
}

// The plan of conv op `o` for micro-batch mb on the tcgen05 engine: the halo TMA planner (which also takes the merged
// ConvTranspose), else the flat one (1x1 and ConvTranspose 2x2), else the stride-2 one, else the thread-gather kernel.
// Returns true for a TMA plan.
static inline bool plan_conv_op(const Op& o, int mb, int num_sms, ConvParams& p) {
  ConvDesc cd{};
  cd.B = mb; cd.H = o.x.H; cd.W = o.x.W; cd.Cin = o.x.Cp; cd.in_pitch = o.x.pitch;
  cd.Cout = o.y.Cp + (o.layer2 >= 0 ? o.y2.Cp : 0); cd.out_pitch = o.y.pitch;
  cd.k = o.k; cd.stride = o.stride; cd.act = o.act; cd.transposed = o.transposed;
  cd.res_pitch = o.has_res ? o.res.pitch : 0;
  cd.upm = o.up_layer >= 0 ? 1 : 0;
  if (plan_conv_halo_tma(cd, num_sms, p)) return true;
  if (!flat_tma_disabled() && plan_conv_flat_tma(cd, num_sms, p)) return true;
  if (!s2_tma_disabled() && plan_conv_s2_tma(cd, num_sms, p)) return true;
  p = plan_conv(cd, num_sms, 0);
  return false;
}

// The parameters one launch of a layer planned by plan_conv_op runs with, for a chunk of nb frames: a partial last chunk
// keeps the plan's layout with fewer frames (replan_for_batch), then a small TMA launch gets at most half the SMs.
static inline ConvParams conv_launch_params(const ConvParams& plan, bool tma, int nb, int num_sms) {
  ConvParams p = plan;
  if (nb != p.B) p = replan_for_batch(plan, nb, num_sms);
  // Small launches use at most HALF the SMs (XRSEG_TINY_GRID=0 turns it off): 3x3 layers with at most two work items
  // per SM (296: every 20x20 layer, the 3x3 convs of the 40x40 stage) and 1x1 layers with at most 800 items (the 40x40
  // stage).  These kernels are latency-bound -- most of their ~10 us is fill
  // and drain -- and a throughput caller keeps several runners in flight: with half-width grids the small kernels of
  // two steps sit side by side on disjoint SMs instead of taking turns on all of them.  Measured (B200, batch 64, four
  // runners, profiles/r2_experiments.md): 34.5k -> 36.7k frames/s, e2e 32.4k -> 34.0k; one runner alone 30.2k -> 29.9k;
  // batch-1 latency unchanged (its grids are smaller than the cap anyway).
  // Tensor-heavy layers stay at half width too: keeping them on all SMs (b7: 256 items of 72 N = 256 MMAs each, 21 us of
  // tensor time on half the SMs against 10.5 us on all of them; h5.box.0, n20, h4.box.1, n13.cv1, b9.cv2 likewise) made
  // those launches alone 43 -> 28, 30 -> 21, 27 -> 21, 27 -> 19, 37 -> 28, 24 -> 21 us and one runner alone 32.0k -> 32.5k
  // frames/s, but four runners 39.1k -> 38.2k and e2e 35.9k -> 35.6k: side by side on disjoint SMs beats taking turns.
  static const bool tiny_on = [] { const char* e = getenv("XRSEG_TINY_GRID"); return !(e && e[0] == '0'); }();
  const int cap = num_sms / 2;
  const int work = p.m_tiles * p.n_tiles;
  if (tiny_on && tma && p.grid > cap && work <= (p.mode == MODE_FLAT_TMA ? 800 : 296)) p.grid = cap;
  return p;
}

// ---------------------------------------------------------------------------------------------------------------
// XRSW weight pack (written by xr_image_segmentation_b200/weights.py)
// ---------------------------------------------------------------------------------------------------------------
#pragma pack(push, 1)
struct XrswHeader {
  char magic[4];
  uint32_t version, n_layers, scale;
  uint64_t payload_offset;
  uint8_t reserved[8];
};
struct XrswLayer {
  char name[32];
  uint32_t cout, cin_g, k, stride, groups, act, transposed, dtype;
  float w_scale; int32_t w_zp; float b_scale; int32_t b_zp;
  uint64_t w_off, b_off;
};
#pragma pack(pop)
static_assert(sizeof(XrswHeader) == 32, "header size");
static_assert(sizeof(XrswLayer) == 96, "record size");

struct HostLayerWeights {
  std::vector<float> w, b;
};

// Dequantize exactly like the reference graph's DequantizeUint8 layers: (q - zp) * scale per tensor.
static inline void xrsw_load(const void* data, size_t bytes, const std::vector<LayerRec>& layers, int scale,
                             std::vector<HostLayerWeights>& out) {
  XR_CHECK(bytes >= sizeof(XrswHeader), "weight pack too small");
  const uint8_t* p = static_cast<const uint8_t*>(data);
  XrswHeader h;
  memcpy(&h, p, sizeof(h));
  XR_CHECK(memcmp(h.magic, "XRSW", 4) == 0 && h.version == 1, "not an XRSW v1 pack");
  XR_CHECK(h.n_layers == layers.size(), "pack has %u layers, topology has %zu", h.n_layers, layers.size());
  XR_CHECK(static_cast<int>(h.scale) == scale, "pack is for scale '%c'", static_cast<char>(h.scale));
  XR_CHECK(bytes >= sizeof(XrswHeader) + h.n_layers * sizeof(XrswLayer) && h.payload_offset <= bytes, "truncated pack");
  out.resize(h.n_layers);
  for (uint32_t i = 0; i < h.n_layers; ++i) {
    XrswLayer r;
    memcpy(&r, p + sizeof(XrswHeader) + i * sizeof(XrswLayer), sizeof(r));
    const LayerRec& l = layers[i];
    const int cin_g = l.cin / l.groups;
    XR_CHECK(static_cast<int>(r.cout) == l.cout && static_cast<int>(r.cin_g) == cin_g && static_cast<int>(r.k) == l.k &&
                 static_cast<int>(r.stride) == l.stride && static_cast<int>(r.groups) == l.groups &&
                 static_cast<int>(r.transposed) == l.transposed && static_cast<int>(r.act) == l.act,
             "layer %u (%.32s) does not match topology layer %s", i, r.name, l.name.c_str());
    const size_t nw = static_cast<size_t>(l.cout) * cin_g * l.k * l.k;
    const size_t nb = l.cout;
    const size_t esz = r.dtype == 0 ? 4 : 1;
    XR_CHECK(r.dtype == 0 || r.dtype == 3, "unsupported dtype %u", r.dtype);
    XR_CHECK(h.payload_offset + r.w_off + nw * esz <= bytes && h.payload_offset + r.b_off + nb * esz <= bytes,
             "layer %u payload out of range", i);
    const uint8_t* wp = p + h.payload_offset + r.w_off;
    const uint8_t* bp = p + h.payload_offset + r.b_off;
    out[i].w.resize(nw);
    out[i].b.resize(nb);
    if (r.dtype == 0) {
      memcpy(out[i].w.data(), wp, nw * 4);
      memcpy(out[i].b.data(), bp, nb * 4);
    } else {
      for (size_t j = 0; j < nw; ++j) out[i].w[j] = (static_cast<float>(wp[j]) - static_cast<float>(r.w_zp)) * r.w_scale;
      for (size_t j = 0; j < nb; ++j) out[i].b[j] = (static_cast<float>(bp[j]) - static_cast<float>(r.b_zp)) * r.b_scale;
    }
  }
}

}  // namespace xrseg
