// conv_tma.cuh -- the TMA-fed tcgen05 convolution kernel: every convolution of the network except the K = 27 stem.
//
// Same GEMM view as conv_umma.cuh (D[M = output positions, N = Cout] = A[M, K] * W[N, K]^T, fp16 operands, fp32 accumulators
// in TMEM), but nothing except ONE thread ever touches an address: the A operand is fetched by cp.async.bulk.tensor into
// hardware-swizzled shared memory (row = one K-block of 16 / 32 / 64 channels = 32 / 64 / 128 bytes) and a tap is a pure
// ROW SHIFT of the operand descriptor.  Three modes share the kernel:
//   * halo  (3x3 stride 1): a work item is R full rows of one image; per K-block one 4-D box (channels, x = -1..W,
//     y = y0-1..y0+R, image) lands the whole halo, out-of-bounds coordinates are zero-filled by the TMA unit -- which IS the
//     convolution's padding.  Tap (kh,kw) of position j is row j + kh*(W+2) + kw - 1: nine MMAs per 16 channels whose
//     descriptors merely start at different rows.  The input is read ~(R+2)/R times instead of 9x (im2col).
//   * s2    (3x3 stride 2): the input is read as four parity planes X[2ys+py][2xs+px] (four tensor maps), so taps are row
//     shifts again: tap (kh,kw) = plane (kh != 1, kw != 1) at row j + (kh == 2)(Wo+1) - (kw == 0).
//   * flat  (1x1 and the 2x2 stride-2 ConvTranspose): plain GEMM over the flattened [B*H*W, C] matrix, the whole K of a
//     thin layer in one stage; ConvTranspose = N = 4 positions x Cout, scattered by the epilogue.
// Warp roles (416 threads): warp 0 = TMA producer (one lane), warps 1-4 = MMA issuers, ONE PER 128-ROW SUB-TILE (a single
// thread cannot issue tcgen05.mma faster than one per ~50-65 cycles, which bounded every thin layer), warps 5-12 = epilogue
// (tcgen05.ld -> +bias -> SiLU -> +residual -> one 256-bit store per 16 channels into the concat slice).  Accumulators are
// double-buffered in TMEM; weights stay resident in shared memory when they fit, else stream per stage by bulk copy.
// Every launch uses programmatic dependent launch: weights are fetched and TMEM allocated before griddepcontrol.wait.
#pragma once

#include <cuda.h>

#include "conv_umma.cuh"

namespace xrseg {

enum { MODE_HALO_TMA = 2, MODE_FLAT_TMA = 3, MODE_S2_TMA = 4 };

// Up to four tensor maps per launch (MODE_S2_TMA reads four parity planes of the input; the other modes use m[0]).
struct TmapSet {
  CUtensorMap m[4];
};
// warp 0: TMA producer; warps 1-4: MMA issuers (one per 128-row sub-tile: a single thread cannot issue tcgen05.mma faster
// than one per ~50-65 cycles, which bounded every thin layer); warps 5 .. 5 + TMA_EPI_WARPS - 1: epilogue.  The epilogue
// warps form TMA_EPI_WARPS / 4 groups of four (one warp per TMEM lane quadrant); the 16-column units of an item are dealt
// round-robin to the groups.  16 epilogue warps (four per scheduler) is the measured optimum: the epilogue is bound by
// dependency stalls, not by issue slots or the MUFU (tools/probe_mufu.cu: 15.4 SiLU / clk / SM with eight warps), so more
// warps per scheduler hide more of them -- 8 / 12 / 16 / 20 / 24 warps: 31.7k / 32.6k / 33.4k / 32.2k / 29.5k frames/s
// (past 16 the register cap of a 1-CTA-per-SM launch, 65536 / threads, forces spills).
enum { TMA_EPI_WARPS = 16, TMA_EPI_GROUPS = TMA_EPI_WARPS / 4, TMA_THREADS = 32 * (5 + TMA_EPI_WARPS), TMA_TAIL_PAD = 4096,
       TMA_FIRST_EPI_WARP = 5 };

struct TmaPlanExtra {
  int R, nsub, tpi, hbox, slots_box;
};

// ---- tensor map (driver entry point fetched through the runtime: no link dependency on libcuda) ----------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    XR_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
    XR_CHECK(p != nullptr && q == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available");
    fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

// 4-D view (C, W, H, B) of an NHWC fp16 tensor slice; box = (8 channels, W+2, R+2, 1).
static inline CUtensorMap make_halo_tensor_map(const __half* base, int B, int H, int W, int C, int pitch, int box_w,
                                               int box_h, int box_c = 8, int sw = 0) {
  CUtensorMap m;
  cuuint64_t dims[4] = {static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H),
                        static_cast<cuuint64_t>(B)};
  cuuint64_t strides[3] = {static_cast<cuuint64_t>(pitch) * 2, static_cast<cuuint64_t>(W) * pitch * 2,
                           static_cast<cuuint64_t>(H) * W * pitch * 2};
  cuuint32_t box[4] = {static_cast<cuuint32_t>(box_c), static_cast<cuuint32_t>(box_w), static_cast<cuuint32_t>(box_h), 1};
  const CUtensorMapSwizzle swz = sw == 3 ? CU_TENSOR_MAP_SWIZZLE_128B : sw == 2 ? CU_TENSOR_MAP_SWIZZLE_64B
                                 : sw == 1 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = get_encode_tiled()(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<__half*>(base), dims, strides, box,
                                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  XR_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d) for [%d,%d,%d,%d] pitch %d box %dx%d", (int)r, B, H, W,
           C, pitch, box_w, box_h);
  return m;
}

// ---- planning --------------------------------------------------------------------------------------------------
// Few work items (batch-1 streaming: a 20x20 layer is one or two items): a layer with >= 128 output channels whose items would
// keep at most half the SMs busy is planned as TWO N tiles -- twice the CTAs, half the MMAs (and half the streamed weights) on
// each one's critical path.  Set by the plan_conv_*_tma wrappers for a second planning pass; XRSEG_SPLIT_SMALL=0 turns it off.
static inline int& tma_force_split_ref() {
  static thread_local int f = 0;
  return f;
}
static inline void tma_apply_split(ConvParams& p, int ncols) {
  const int f = tma_force_split_ref();          // 0, 2 or 4 N tiles
  if (f && p.n_tiles == 1 && p.Ntile >= 64 * f && (p.Ntile / f) % 16 == 0 && ncols == p.Ntile) {
    p.Ntile /= f;
    p.n_tiles = f;
  }
}
// 0: no split; 2 / 4: N tiles for the second planning pass (four only for 256 output channels on at most a quarter of the SMs)
static inline int tma_wants_split(const ConvParams& p, int num_sms) {
  static const bool on = [] { const char* e = getenv("XRSEG_SPLIT_SMALL"); return !(e && e[0] == '0'); }();
  if (!on || p.n_tiles != 1 || p.Ntile < 128 || p.transposed || 2 * p.m_tiles > num_sms) return 0;
  if (p.Ntile == 256 && 4 * p.m_tiles <= num_sms) return 4;
  return (p.Ntile / 2) % 16 == 0 ? 2 : 0;
}

// A CTA never has more than ceil(work / grid) * nks stages to fetch: a deeper ring only costs shared memory, and a small
// footprint is what lets the next kernel's CTAs become co-resident early (programmatic dependent launch) so that their
// prologue -- barrier init, TMEM allocation, weight fetch -- overlaps this kernel's tail.
// Accumulator sets in TMEM: every plan takes two.  Measured on B200 (YOLO11n-seg, batch 64): ringing four sets for thin
// layers changes no layer by more than noise -- the MMA -> epilogue round trip is not what bounds them.
static inline int clamp_stages(int S, int work, int num_sms, int nks) {
  const int grid = work < num_sms ? work : num_sms;
  int need = ceil_div(work, grid) * nks;
  if (need < 2) need = 2;
  return S < need ? S : need;
}

// Returns false when the layer does not fit this kernel (caller falls back to the thread-gather kernel).
static inline bool plan_conv_halo_tma_impl(const ConvDesc& d, int num_sms, ConvParams& p, bool swizzled = true) {
  if (!(d.k == 3 && d.stride == 1 && !d.transposed)) return false;
  p = ConvParams{};
  p.B = d.B; p.H = d.H; p.W = d.W; p.Cin = d.Cin; p.in_pitch = d.in_pitch;
  p.Cout = d.Cout; p.out_pitch = d.out_pitch; p.res_pitch = d.res_pitch;
  p.k = 3; p.stride = 1; p.pad = 1; p.act = d.act; p.transposed = 0;
  p.Ho = d.H; p.Wo = d.W;
  p.Ntile = d.Cout <= 256 ? d.Cout : 256;
  if (d.Cout % p.Ntile) return false;
  p.n_tiles = d.Cout / p.Ntile;
  // Wide maps with 128 output channels (the s scale's proto.cv2, 160 x 160): two sub-tiles of 128 columns fill the accumulator set,
  // and 256 positions hold ONE 162-position row -- 63 % of every MMA's rows valid, the halo read three times.  Two N tiles of 64
  // channels give four sub-tiles = three rows per item (95 % valid) for the same TMEM columns; the input is read once per N tile.
  // XRSEG_HALO_SPLIT_N=0 turns it off.
  static const bool split_n_on = [] { const char* e = getenv("XRSEG_HALO_SPLIT_N"); return !(e && e[0] == '0'); }();
  if (split_n_on && p.n_tiles == 1 && p.Ntile == 128 && 256 / (d.W + 2) < 2 && 512 / (d.W + 2) >= 2) {
    p.Ntile = 64;
    p.n_tiles = 2;
  }
  tma_apply_split(p, d.Cout);
  p.idesc = umma_idesc_f16(p.Ntile, 0);
  p.mode = MODE_HALO_TMA;
  p.Wp = d.W + 2;
  p.Hp1 = d.H + 1;
  int nsub_max = 256 / p.Ntile;
  if (nsub_max > 4) nsub_max = 4;
  if (nsub_max < 1 || p.Wp > 256) return false;
  int R = (128 * nsub_max) / p.Wp;
  if (R > d.H) R = d.H;
  if (R < 1 || R + 2 > 256) return false;
  {
    // rows per item: the tallest tile that fits unless a shorter one fills the SMs better (20x20 maps: R = 20 would keep
    // 64 CTAs busy with four sub-tiles each, R = 10 keeps 128 busy with two).  Cost = rounds of the busiest CTA x
    // (sub-tiles + fixed item overhead), weighted by the halo re-read (R + 2) / R.
    int best_R = R;
    double best_c = 1e30;
    const bool few_rounds = ceil_div(d.B * ceil_div(d.H, R) * p.n_tiles, num_sms) <= 2;   // only then quantization matters
    for (int r = R; r >= (few_rounds ? 1 : R); --r) {
      const int nsub = ceil_div(r * p.Wp, 128);
      const int items = d.B * ceil_div(d.H, r) * p.n_tiles;
      const double c = ceil_div(items, num_sms) * (nsub + 0.35) * (1.0 + 0.5 / r);
      if (c < best_c - 1e-9) { best_c = c; best_R = r; }
    }
    R = best_R;
  }
  p.R = R;
  p.nsub = ceil_div(R * p.Wp, 128);
  p.tpi = ceil_div(d.H, R);
  p.hbox = R + 2;
  p.slots = p.hbox * p.Wp;
  p.lbo_a = round_up(p.slots * 16, 128);
  if (swizzled) {
    // Swizzled operands: one smem row = one K-block of cb = min(Cin, 64) channels (32 / 64 / 128 bytes), stored with the
    // TMA / UMMA hardware swizzle of that width.  A whole K-block of the halo is ONE TMA box; a tap is still a row shift.
    int best_cb = 0, best_S = 0;
    for (int cb = 64; cb >= 16; cb >>= 1) {
      if (cb > d.Cin || d.Cin % cb) continue;
      const int rb = cb * 2;
      const int a_stage = round_up(p.slots * rb, 1024);
      const int b_stage = 9 * p.Ntile * rb;
      const long total_b = static_cast<long>(d.Cin / cb) * b_stage;
      const bool res = (p.n_tiles == 1 && total_b <= 114688);
      const int fixed = round_up(CONV_HDR_BYTES, 1024) + 1024 + 128 * rb + 1024 +
                        (res ? round_up(static_cast<int>(total_b), 1024) : 0);
      int S = (CONV_SMEM_MAX - fixed) / (a_stage + (res ? 0 : round_up(b_stage, 1024)));
      if (S > CONV_MAX_STAGES) S = CONV_MAX_STAGES;
      if (S > 2 * (d.Cin / cb) + 2) S = 2 * (d.Cin / cb) + 2;
      // The TMA unit delivers one box ROW per ~1.5 cycles whatever its width (tools/probe_tma_rate.cu: 21 / 42 / 85 B/clk per SM
      // for 32 / 64 / 128-byte rows), so a layer that splits its channels into narrow K-blocks pays the row cost Cin / cb
      // times.  Taking the WIDEST K-block that still leaves a two-stage ring was measured on the network (proto.cv2 148 -> 154
      // us, h4.box.0 33 -> 35 us, n13/n19.m0.cv1 equal): the deeper three-stage ring with narrower blocks is the better trade.
      if (S >= 3 || (S == 2 && best_S < 2)) {
        best_cb = cb;
        best_S = S;
        if (S >= 3) break;
      }
    }
    if (best_S < 2) return false;
    const int cb = best_cb;
    p.sw = cb == 64 ? 3 : (cb == 32 ? 2 : 1);
    const int rb = cb * 2;
    p.cb = cb; p.cps = cb / 8; p.nks = d.Cin / cb;
    p.taps = 9; p.K_total = 9 * d.Cin;
    p.nbuf = 2;
    p.tmem_cols = pow2_ceil(p.nbuf * p.nsub * p.Ntile);
    p.a_stage_bytes = round_up(p.slots * rb, 1024);
    p.b_stage_bytes = 9 * p.Ntile * rb;
    const long total_b = static_cast<long>(p.nks) * p.b_stage_bytes;
    p.b_resident = (p.n_tiles == 1 && total_b <= 114688) ? 1 : 0;
    const int resident = p.b_resident ? static_cast<int>(total_b) : 0;
    const int S = clamp_stages(best_S, d.B * p.tpi * p.n_tiles, num_sms, p.nks);
    p.S = S;
    p.M_total = d.B * p.tpi;
    p.m_tiles = p.M_total;
    p.smem_off_b = round_up(CONV_HDR_BYTES, 1024);
    const int b_region = p.b_resident ? resident : S * round_up(p.b_stage_bytes, 1024);
    // one tail pad BEFORE the A stages too: tap (0,0) of position 0 reads the row before the stage
    p.smem_off_a = p.smem_off_b + round_up(b_region, 1024) + 1024;
    p.smem_bytes = p.smem_off_a + S * p.a_stage_bytes + 128 * rb + 1024;
    if (p.smem_bytes > CONV_SMEM_MAX) return false;
    const int work = p.m_tiles * p.n_tiles;
    p.grid = work < num_sms ? work : num_sms;
    p.fd_wp = make_fastdiv(p.Wp);
    p.fd_hp1 = make_fastdiv(p.tpi);
    p.fd_hw = make_fastdiv(1);
    p.fd_wo = make_fastdiv(1);
    p.fd_cin = make_fastdiv(d.Cin);
    p.fd_cout = make_fastdiv(d.Cout);
    return true;
  }
  p.taps = 9;
  p.K_total = 9 * d.Cin;
  p.nbuf = 2;
  p.tmem_cols = pow2_ceil(2 * p.nsub * p.Ntile);
  const int budget = CONV_SMEM_MAX - CONV_HDR_BYTES - TMA_TAIL_PAD;
  const long total_b = 9L * d.Cin * p.Ntile * 2;
  p.b_resident = (p.n_tiles == 1 && total_b <= 114688) ? 1 : 0;
  int best_cb = 0, best_S = 0;
  for (int cb = 64; cb >= 16; cb >>= 1) {
    if (d.Cin % cb) continue;
    const int a_stage = (cb / 8) * p.lbo_a;
    const int b_stage = 9 * cb * p.Ntile * 2;
    const int resident = p.b_resident ? static_cast<int>(total_b) : 0;
    int S = (budget - resident) / (a_stage + (p.b_resident ? 0 : b_stage));
    const int nks = d.Cin / cb;
    if (S > CONV_MAX_STAGES) S = CONV_MAX_STAGES;
    if (S >= 3 || (S == 2 && best_S < 2)) {
      if (S > 2 * nks + 2) S = 2 * nks + 2;
      best_cb = cb;
      best_S = S;
      if (S >= 3) break;
    }
  }
  if (best_S < 2) return false;
  p.cb = best_cb;
  p.cps = best_cb / 8;
  p.nks = d.Cin / best_cb;
  p.S = best_S;
  p.a_stage_bytes = p.cps * p.lbo_a;
  p.b_stage_bytes = 9 * best_cb * p.Ntile * 2;
  p.M_total = d.B * p.tpi;                      // number of (image, row-block) tiles
  p.m_tiles = p.M_total;
  p.smem_off_b = CONV_HDR_BYTES;
  const int b_region = p.b_resident ? p.nks * p.b_stage_bytes : p.S * p.b_stage_bytes;
  p.smem_off_a = CONV_HDR_BYTES + round_up(b_region, 128);
  p.smem_bytes = p.smem_off_a + p.S * p.a_stage_bytes + TMA_TAIL_PAD;
  if (p.smem_bytes > CONV_SMEM_MAX) return false;
  const int work = p.m_tiles * p.n_tiles;
  p.grid = work < num_sms ? work : num_sms;
  p.fd_wp = make_fastdiv(p.Wp);
  p.fd_hp1 = make_fastdiv(p.tpi);               // reused: tile -> (image, row block)
  p.fd_hw = make_fastdiv(1);
  p.fd_wo = make_fastdiv(1);
  p.fd_cin = make_fastdiv(d.Cin);
  p.fd_cout = make_fastdiv(d.Cout);
  return true;
}


// General 4-D tiled map over fp16 data: dims / strides (bytes, dims 1..3) / box given explicitly.
static inline CUtensorMap make_tensor_map_4d(const __half* base, const cuuint64_t (&dims)[4], const cuuint64_t (&strides)[3],
                                             const cuuint32_t (&box)[4], int sw) {
  CUtensorMap m;
  const CUtensorMapSwizzle swz = sw == 3 ? CU_TENSOR_MAP_SWIZZLE_128B : sw == 2 ? CU_TENSOR_MAP_SWIZZLE_64B
                                 : sw == 1 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = get_encode_tiled()(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<__half*>(base), dims, strides, box, estr,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  XR_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return m;
}

// 3x3 STRIDE-2 convolution on the same kernel ("s2" mode).  The input is read as four parity planes
//     plane(py,px)[ys][xs] = X[2 ys + py][2 xs + px]          (four tensor maps: same dims, base shifted by (py W + px) pixels,
//                                                               x / y strides doubled)
// so that every tap is again a pure row shift of a plane buffer in position-linear order (position j = yy*(Wo+1) + cc,
// cc = ox + 1): tap (kh,kw) reads plane (kh != 1, kw != 1) at row j + (kh == 2 ? Wo+1 : 0) - (kw == 0 ? 1 : 0).
// Per K-block the producer issues four TMA boxes (cb channels, Wo+1 columns from xs = -1, R+1 rows from ys = oy0 - py);
// out-of-bounds coordinates are the convolution's zero padding.  The input is read ~(R+1)/R times instead of 2.25x by
// the im2col gather, and nothing but one thread touches addresses.
// NOTE: p.H / p.W / p.Wp hold the OUTPUT geometry (Ho, Wo, Wo+1) in this mode -- that is what the epilogue indexes.
static inline bool plan_conv_s2_tma_impl(const ConvDesc& d, int num_sms, ConvParams& p, bool allow_pair = true) {
  if (!(d.k == 3 && d.stride == 2 && !d.transposed) || (d.H & 1) || (d.W & 1)) return false;
  p = ConvParams{};
  const int Ho = d.H / 2, Wo = d.W / 2;
  p.B = d.B; p.H = Ho; p.W = Wo; p.Cin = d.Cin; p.in_pitch = d.in_pitch;
  p.Cout = d.Cout; p.out_pitch = d.out_pitch; p.res_pitch = d.res_pitch;
  p.k = 3; p.stride = 2; p.pad = 1; p.act = d.act; p.transposed = 0;
  p.Ho = Ho; p.Wo = Wo;
  p.Ntile = d.Cout <= 256 ? d.Cout : 256;
  if (d.Cout % p.Ntile) return false;
  p.n_tiles = d.Cout / p.Ntile;
  tma_apply_split(p, d.Cout);
  p.idesc = umma_idesc_f16(p.Ntile, 0);
  p.mode = MODE_S2_TMA;
  p.taps = 9;
  p.K_total = 9 * d.Cin;
  p.Wp = Wo + 1;
  p.Hp1 = Ho + 1;
  int nsub_max = 256 / p.Ntile;
  if (nsub_max > 4) nsub_max = 4;
  if (nsub_max < 1 || p.Wp > 255) return false;
  const long total_w = 9L * d.Cin * p.Ntile * 2;
  p.b_resident = (p.n_tiles == 1 && total_w <= 98304) ? 1 : 0;
  const int resident = p.b_resident ? static_cast<int>(total_w) : 0;
  // search (cb, R) for the lowest estimated cycles per output position.  Measured constants (tools/probe_tma.py): one
  // tcgen05.mma costs the issuing thread ~50 cycles (or its tensor time 128*N/256 if larger), one stage hand-over ~600,
  // one epilogue pass over 128 rows x 32 columns ~650; a 2-stage ring stalls more than a 3-stage one.
  int best_cb = 0, best_R = 0, best_S = 0;
  double best_cost = 1e30;
  for (int cb = 64; cb >= 16; cb >>= 1) {
    if (cb > d.Cin || d.Cin % cb) continue;
    const int rb = cb * 2;
    for (int R = (128 * nsub_max) / p.Wp; R >= 1; --R) {
      if (R > Ho) continue;
      const int plane = round_up((R + 1) * p.Wp * rb, 1024);
      const int b_stage = 9 * p.Ntile * rb;
      const int fixed = round_up(CONV_HDR_BYTES, 1024) + 1024 + 128 * rb + 1024 + p.Wp * rb + round_up(resident, 1024);
      int S = (CONV_SMEM_MAX - fixed) / (4 * plane + (p.b_resident ? 0 : round_up(b_stage, 1024)));
      if (S > CONV_MAX_STAGES) S = CONV_MAX_STAGES;
      if (S > 2 * (d.Cin / cb) + 2) S = 2 * (d.Cin / cb) + 2;
      if (S < 2) continue;
      const int nks = d.Cin / cb, nsub = ceil_div(R * p.Wp, 128);
      // operand fetch at ~40 bytes per clock.  A row-cost model (~1.5 cycles per TMA box row whatever its width, MMA issue
      // parallel over the sub-tile warps) was measured on the network: n17 (80 -> 40) alone 40.7 -> 27.4 us, b5 51 -> 50 us,
      // b3 (160 -> 80) 64 -> 69 us; restricted to output maps up to 40 x 40 one runner alone gains 1 %, but four runners LOSE
      // 2 % (38.1k -> 37.3k frames/s, three A/B pairs): n17's plan then has 512 items and leaves the half-width rule of the small
      // launches (xrseg_api.cu), and side by side beats faster.
      const double t_mma = nks * 600.0 + 9.0 * (d.Cin / 16) * nsub * (p.Ntile / 2.0 > 50.0 ? p.Ntile / 2.0 : 50.0);
      const double t_epi = nsub * ceil_div(p.Ntile, 32) * 650.0;
      const double t_mem = 4.0 * (R + 1) * p.Wp * d.Cin * 2 / 40.0;
      double t = t_mma > t_epi ? t_mma : t_epi;
      if (t_mem > t) t = t_mem;
      t = (t + 800.0) * (S >= 3 ? 1.0 : 1.15);
      const int items = d.B * ceil_div(Ho, R) * p.n_tiles;
      const double cost = t * ceil_div(items, num_sms);                       // the busiest CTA's time (wave quantization)
      if (cost < best_cost) { best_cost = cost; best_cb = cb; best_R = R; best_S = S; }
    }
  }
  if (best_S < 2) return false;
  const int cb = best_cb, rb = cb * 2;
  p.cb = cb; p.cps = cb / 8; p.nks = d.Cin / cb; p.kps = 1;
  p.sw = cb == 64 ? 3 : (cb == 32 ? 2 : 1);
  p.R = best_R;
  p.nsub = ceil_div(p.R * p.Wp, 128);
  p.tpi = ceil_div(Ho, p.R);
  p.S = clamp_stages(best_S, d.B * p.tpi * p.n_tiles, num_sms, p.nks);
  p.hbox = p.R + 1;
  p.slots = p.hbox * p.Wp;                         // rows of ONE plane box
  p.lbo_a = round_up(p.slots * rb, 1024);          // bytes of one plane buffer
  p.a_stage_bytes = 4 * p.lbo_a;
  p.b_stage_bytes = 9 * p.Ntile * rb;
  p.nbuf = 2;
  p.tmem_cols = pow2_ceil(p.nbuf * p.nsub * p.Ntile);
  p.M_total = d.B * p.tpi;
  p.m_tiles = p.M_total;
  p.smem_off_b = round_up(CONV_HDR_BYTES, 1024);
  const int b_region = p.b_resident ? resident : p.S * round_up(p.b_stage_bytes, 1024);
  p.smem_off_a = p.smem_off_b + round_up(b_region, 1024) + 1024;        // one pad row block before the stages (offset -1)
  p.smem_bytes = p.smem_off_a + p.S * p.a_stage_bytes + 128 * rb + p.Wp * rb + 1024;   // tail: rows read past the last plane
  if (p.smem_bytes > CONV_SMEM_MAX) return false;
  // PIXEL-PAIR rows: when a K-block is the whole pixel (cb == Cin == pixel pitch, <= 32 channels) the even and the odd pixel of
  // a column pair are 2 * rb contiguous bytes in global memory, so the two x-parity planes of a row parity become ONE plane whose
  // rows are [even pixel | odd pixel]: two TMA boxes per K-block with rows twice as wide instead of four -- the TMA unit
  // delivers ~1.5 cycles per box row whatever its width (tools/probe_tma_rate.cu), and b1 (16 channels = 32-byte rows) was bound
  // by exactly that.  The x parity of a tap becomes a +rb offset inside the row (like a k16 step), the operand swizzle is the
  // one of the 2 * rb row; weights are unchanged.  XRSEG_S2_PAIR=0 turns it off.
  static const bool pair_on = [] { const char* e = getenv("XRSEG_S2_PAIR"); return !(e && e[0] == '0'); }();
  if (allow_pair && pair_on && p.nks == 1 && cb == d.Cin && d.in_pitch == d.Cin && cb <= 32) {
    const int rba = 2 * rb;
    const int lbo = round_up(p.slots * rba, 1024);
    const int bytes = p.smem_off_a + p.S * 2 * lbo + 128 * rba + p.Wp * rba + 1024;
    if (bytes <= CONV_SMEM_MAX) {
      p.pair = 1;
      p.lbo_a = lbo;
      p.a_stage_bytes = 2 * lbo;
      p.smem_bytes = bytes;
    }
  }
  const int work = p.m_tiles * p.n_tiles;
  p.grid = work < num_sms ? work : num_sms;
  p.fd_wp = make_fastdiv(p.Wp);
  p.fd_hp1 = make_fastdiv(p.tpi);
  p.fd_hw = make_fastdiv(1);
  p.fd_wo = make_fastdiv(1);
  p.fd_cin = make_fastdiv(d.Cin);
  p.fd_cout = make_fastdiv(d.Cout);
  return true;
}

// The four parity-plane maps of an NHWC input [B,H,W,C] (pixel pitch `pitch`): index py*2 + px.
static inline TmapSet make_s2_tensor_maps(const __half* base, int B, int H, int W, int C, int pitch, const ConvParams& p) {
  TmapSet t{};
  if (p.pair) {   // index py: rows of 2 C channels = the pixel pair (2 xs, 2 xs + 1) of row 2 ys + py
    const cuuint64_t pdims[4] = {static_cast<cuuint64_t>(2 * C), static_cast<cuuint64_t>(W / 2), static_cast<cuuint64_t>(H / 2),
                                 static_cast<cuuint64_t>(B)};
    const cuuint64_t pstrides[3] = {static_cast<cuuint64_t>(pitch) * 4, static_cast<cuuint64_t>(W) * pitch * 4,
                                    static_cast<cuuint64_t>(H) * W * pitch * 2};
    const cuuint32_t pbox[4] = {static_cast<cuuint32_t>(2 * p.cb), static_cast<cuuint32_t>(p.Wp), static_cast<cuuint32_t>(p.hbox), 1};
    for (int py = 0; py < 2; ++py)
      t.m[py] = make_tensor_map_4d(base + static_cast<size_t>(py) * W * pitch, pdims, pstrides, pbox, p.sw + 1);
    return t;
  }
  const cuuint64_t dims[4] = {static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(W / 2), static_cast<cuuint64_t>(H / 2),
                              static_cast<cuuint64_t>(B)};
  const cuuint64_t strides[3] = {static_cast<cuuint64_t>(pitch) * 4, static_cast<cuuint64_t>(W) * pitch * 4,
                                 static_cast<cuuint64_t>(H) * W * pitch * 2};
  const cuuint32_t box[4] = {static_cast<cuuint32_t>(p.cb), static_cast<cuuint32_t>(p.Wp), static_cast<cuuint32_t>(p.hbox), 1};
  for (int py = 0; py < 2; ++py)
    for (int px = 0; px < 2; ++px)
      t.m[py * 2 + px] = make_tensor_map_4d(base + (static_cast<size_t>(py) * W + px) * pitch, dims, strides, box, p.sw);
  return t;
}

// N tiles of a flat-mode plan: one tile up to 256 columns, else two or four equal tiles of a multiple of 16 columns (the kernel
// decodes work items for 1, 2 or 4 N tiles).  The class convolution's output pitch is padded to such a width (model.cuh
// class_pitch) so that every class count gets a plan; every other layer is <= 256, 512 or 1024 columns wide.
static inline bool tma_n_split(int ncols, int& Ntile, int& n_tiles) {
  for (n_tiles = 1; n_tiles <= 4; n_tiles *= 2) {
    Ntile = ncols / n_tiles;
    if (ncols % n_tiles == 0 && Ntile <= 256 && (n_tiles == 1 || Ntile % 16 == 0)) return true;
  }
  return false;
}

// 1x1 stride-1 convolution = plain GEMM over the flattened [B*H*W, C] activation matrix ("flat" mode of the same
// kernel): a work item is 128*nsub consecutive pixels, its A operand ONE (or two) 2-D TMA boxes of cb channels x <= 256
// rows per K-block, swizzled like the halo boxes; taps = 1.  One mbarrier arrival per stage instead of one per producer
// thread is what makes the thin layers (K <= 128, N <= 64) run at memory speed: the thread-gather kernel spends most of
// its time in its own arrive/wait traffic there (tools/probe_umma.py).  Channels beyond Cin inside the last K-block are
// out of bounds for the tensor map and arrive as zeros, so Cin only has to be a multiple of 16 (e.g. the 48-channel
// C3k2 concat).
static inline bool plan_conv_flat_tma_impl(const ConvDesc& d, int num_sms, ConvParams& p) {
  // also the 2x2 stride-2 ConvTranspose: the same GEMM with N = 4 positions x Cout, scattered by the epilogue
  const bool convt = d.transposed && d.k == 2 && d.stride == 2 && d.res_pitch == 0;
  if (!((d.k == 1 && d.stride == 1 && !d.transposed) || convt)) return false;
  p = ConvParams{};
  p.B = d.B; p.H = d.H; p.W = d.W; p.Cin = d.Cin; p.in_pitch = d.in_pitch;
  p.Cout = d.Cout; p.out_pitch = d.out_pitch; p.res_pitch = d.res_pitch;
  p.k = d.k; p.stride = d.stride; p.pad = 0; p.act = d.act; p.transposed = convt ? 1 : 0;
  p.Ho = convt ? 2 * d.H : d.H; p.Wo = convt ? 2 * d.W : d.W;
  const int ncols = convt ? 4 * d.Cout : d.Cout;
  if (!tma_n_split(ncols, p.Ntile, p.n_tiles)) return false;
  if (!convt) tma_apply_split(p, ncols);
  p.idesc = umma_idesc_f16(p.Ntile, 0);
  p.mode = MODE_FLAT_TMA;
  p.taps = 1;
  const long rows = static_cast<long>(d.B) * d.H * d.W;
  if (rows >= (1L << 31)) return false;
  p.flat_rows = static_cast<int>(rows);
  const int cb = d.Cin > 32 ? 64 : d.Cin;          // 16, 32 or 64 channels per K-block (row = 32 / 64 / 128 bytes)
  p.cb = cb; p.cps = cb / 8;
  p.sw = cb == 64 ? 3 : (cb == 32 ? 2 : 1);
  const int nkb = ceil_div(d.Cin, cb);             // K-blocks
  p.K_total = nkb * cb;
  const int rb = cb * 2;
  const int b_block = p.Ntile * rb;
  const long total_b = static_cast<long>(nkb) * b_block;
  p.b_resident = (p.n_tiles == 1 && total_b <= 98304) ? 1 : 0;
  const int resident = p.b_resident ? static_cast<int>(total_b) : 0;
  const int tiles128 = ceil_div(p.flat_rows, 128);
  // the kernel keeps the bias of all N tiles at [256, 256 + 4 * ncols) of the header: more than the standard header's 512
  // entries only for the class convolution of a model with more than 512 classes
  const int hdr = round_up(256 + 4 * ncols > CONV_HDR_BYTES ? 256 + 4 * ncols : static_cast<int>(CONV_HDR_BYTES), 1024);
  int nsub = 256 / p.Ntile;
  if (nsub > 4) nsub = 4;
  if (nsub == 3) nsub = 2;                         // an item is one or two FULL boxes of <= 256 rows: power-of-two sub-tiles only
  if (nsub < 1) nsub = 1;                          // (N = 80 at more than 64 frames picked 3: two 256-row boxes into 384 slots)
  while (nsub > 1 && ceil_div(tiles128, nsub) < 8 * num_sms) nsub >>= 1;  // keep >= 8 items per CTA for balance
  for (;; nsub >>= 1) {
    p.nsub = nsub;
    p.slots = 128 * nsub;
    p.hbox = p.slots < 256 ? p.slots : 256;          // rows per TMA box
    // A stage holds kps K-blocks (each slots x rb bytes, its own swizzled sub-buffer): the MMA warp pays a fixed
    // ~500 cycles per stage hand-over (tools/probe_tma.py), so thin layers put their whole K into one stage.
    int kps = nkb, S = 0;
    for (; kps >= 1; --kps) {
      if (nkb % kps != 0 || (kps > 1 && kps * p.slots * rb > 49152)) continue;
      p.kps = kps;
      p.nks = nkb / kps;
      p.a_stage_bytes = kps * p.slots * rb;          // multiple of 1024 for every cb
      p.b_stage_bytes = kps * b_block;
      const int fixed = hdr + (p.b_resident ? round_up(resident, 1024) : 0);
      S = (CONV_SMEM_MAX - fixed) / (p.a_stage_bytes + (p.b_resident ? 0 : round_up(p.b_stage_bytes, 1024)));
      if (S > CONV_MAX_STAGES) S = CONV_MAX_STAGES;
      if (S >= 2) break;                             // streamed weights of a wide layer: fewer K-blocks per stage
    }
    if (S >= 3 || nsub == 1) {
      if (S < 2) return false;
      p.S = clamp_stages(S, ceil_div(p.flat_rows, p.slots) * p.n_tiles, num_sms, p.nks);
      break;
    }
  }
  p.nbuf = 2;
  p.tmem_cols = pow2_ceil(p.nbuf * p.nsub * p.Ntile);
  p.lbo_a = p.a_stage_bytes;
  p.M_total = ceil_div(p.flat_rows, p.slots);
  p.m_tiles = p.M_total;
  p.smem_off_b = hdr;
  const int b_region = p.b_resident ? resident : p.S * round_up(p.b_stage_bytes, 1024);
  p.smem_off_a = p.smem_off_b + round_up(b_region, 1024);
  p.smem_bytes = p.smem_off_a + p.S * p.a_stage_bytes;
  if (p.smem_bytes > CONV_SMEM_MAX) return false;
  const int work = p.m_tiles * p.n_tiles;
  p.grid = work < num_sms ? work : num_sms;
  p.Wp = 1; p.Hp1 = 1; p.R = 0; p.tpi = 1;
  p.fd_wp = make_fastdiv(1);
  p.fd_hp1 = make_fastdiv(1);
  p.fd_hw = make_fastdiv(d.H * d.W);           // ConvTranspose epilogue: row -> (image, h, w)
  p.fd_wo = make_fastdiv(d.W);
  p.fd_cin = make_fastdiv(d.Cin);
  p.fd_cout = make_fastdiv(d.Cout);
  return true;
}

// Planning with the few-work-items split (tma_wants_split): a second pass of the same planner with the N tiles forced.
template <typename Plan>
static inline bool plan_with_split(ConvParams& p, int num_sms, Plan plan) {
  if (!plan(p)) return false;
  if (const int f = tma_wants_split(p, num_sms)) {
    ConvParams q;
    tma_force_split_ref() = f;
    if (plan(q)) p = q;
    tma_force_split_ref() = 0;
  }
  return true;
}
// ConvTranspose 2x2 / stride 2 + 3x3 stride 1 as ONE halo convolution over the map before the upsampling (ConvDesc::upm; the
// n scale's proto.up -> proto.cv2, 64 -> 64 -> 64 channels, 80x80 -> 160x160).  Output pixel (2y + dy, 2x + dx) is a 2x2-tap
// convolution of input rows y + dy - 1 .. y + dy and columns x + dx - 1 .. x + dx: in the 3x3 halo these are taps
// (dy + {0,1}, dx + {0,1}).  Layout of a work item (R = 3 input rows of one image, one row parity dy = item & 1):
//   * two 128-row sub-tiles of halo positions; each holds BOTH column parities: 2 x 64 accumulator columns, so that the
//     accumulator set has 256 columns and the virtual sub-tile v = 2 u + dx is what the rest of the kernel calls a sub-tile
//     (nsub = 4, Ntile = 64: TMEM, the four MMA warps, the fused-tail epilogue); 246 of 256 rows valid;
//   * MMA warp v issues its parity's four taps x 4 k16 steps against resident weights [dx][tap][64][64] of its CTA's dy:
//     a CTA only ever sees one row parity (the grid is even, items alternate dy), so it keeps 64 KB of the 128 KB resident;
//   * the epilogue scatters halo position (y, x) of virtual sub-tile v to output pixel (2y + dy, 2x + dx); pixels on the
//     border of the 160x160 map add a correction to the bias (cv2's zero padding drops the ConvTranspose bias there).
// The K per output pixel falls from 576 to 256.  One K-block of 64 channels (Cin = 64), two stages (the 410-row halo box is
// 52 KB), two accumulator sets = 512 TMEM columns.
static inline bool plan_conv_upmerge_tma(const ConvDesc& d, int num_sms, ConvParams& p) {
  if (!(d.upm && d.k == 3 && d.stride == 1 && !d.transposed && d.Cin == 64 && d.Cout == 64 && d.res_pitch == 0 && d.H >= 2)) return false;
  p = ConvParams{};
  p.B = d.B; p.H = d.H; p.W = d.W; p.Cin = d.Cin; p.in_pitch = d.in_pitch;
  p.Cout = d.Cout; p.out_pitch = d.out_pitch; p.res_pitch = 0;
  p.k = 3; p.stride = 1; p.pad = 1; p.act = d.act; p.transposed = 0; p.upm = 1;
  p.Ho = 2 * d.H; p.Wo = 2 * d.W;
  p.Ntile = 64; p.n_tiles = 1;
  p.idesc = umma_idesc_f16(p.Ntile, 0);
  p.mode = MODE_HALO_TMA;
  p.Wp = d.W + 2;
  p.Hp1 = d.H + 1;
  if (p.Wp > 256) return false;
  p.R = 256 / p.Wp < d.H ? 256 / p.Wp : d.H;    // the rows two 128-row sub-tiles hold
  const int real_sub = ceil_div(p.R * p.Wp, 128);
  p.nsub = 2 * real_sub;                          // virtual sub-tiles (sub-tile, column parity)
  p.tpi = ceil_div(d.H, p.R);
  p.hbox = p.R + 2;
  p.slots = p.hbox * p.Wp;
  p.cb = 64; p.cps = 8; p.nks = 1; p.kps = 1; p.sw = 3;
  p.taps = 8;                                     // per row parity: 2 column parities x 4 taps
  p.K_total = 4 * d.Cin;
  p.nbuf = 2;
  p.tmem_cols = pow2_ceil(p.nbuf * p.nsub * p.Ntile);
  const int rb = p.cb * 2;
  p.lbo_a = round_up(p.slots * 16, 128);
  p.a_stage_bytes = round_up(p.slots * rb, 1024);
  p.b_stage_bytes = p.taps * p.Ntile * rb;        // one row parity's weights; the image holds both
  p.b_resident = 1;
  p.M_total = 2 * d.B * p.tpi;                    // (row tile, row parity), parity fastest
  p.m_tiles = p.M_total;
  p.smem_off_b = round_up(CONV_HDR_BYTES, 1024);
  p.smem_off_a = p.smem_off_b + round_up(p.b_stage_bytes, 1024) + 1024;   // one pad row block before the stages (row -1)
  // rows read past the last stage: the second sub-tile's last position + the farthest tap (2 Wp + 1)
  const int tail_rows = real_sub * 128 + 2 * p.Wp + 1 - p.slots;
  const int tail = round_up((tail_rows > 0 ? tail_rows : 0) * rb, 1024);
  const int corr = 9 * p.Ntile * 4;
  const int fixed = p.smem_off_a + tail + corr + p.Ntile * 32 * 2 + 1024;   // + the fused tail's W2 (xrseg_api.cu) and its alignment
  int S = (CONV_SMEM_MAX - fixed) / p.a_stage_bytes;
  if (S > CONV_MAX_STAGES) S = CONV_MAX_STAGES;
  if (S < 2) return false;
  p.S = clamp_stages(S, p.m_tiles, num_sms, p.nks);
  p.smem_off_corr = p.smem_off_a + p.S * p.a_stage_bytes + tail;
  p.smem_bytes = p.smem_off_corr + corr;
  if (p.smem_bytes > CONV_SMEM_MAX) return false;
  const int grid = (p.m_tiles < num_sms ? p.m_tiles : num_sms) & ~1;   // even: a CTA's items all have one row parity
  if (grid < 2) return false;
  p.grid = grid;
  p.fd_wp = make_fastdiv(p.Wp);
  p.fd_hp1 = make_fastdiv(p.tpi);
  p.fd_hw = make_fastdiv(1);
  p.fd_wo = make_fastdiv(1);
  p.fd_cin = make_fastdiv(d.Cin);
  p.fd_cout = make_fastdiv(d.Cout);
  return true;
}

static inline bool plan_conv_halo_tma(const ConvDesc& d, int num_sms, ConvParams& p, bool swizzled = true) {
  if (d.upm) return swizzled && plan_conv_upmerge_tma(d, num_sms, p);
  if (!swizzled) return plan_conv_halo_tma_impl(d, num_sms, p, false);
  return plan_with_split(p, num_sms, [&](ConvParams& q) { return plan_conv_halo_tma_impl(d, num_sms, q); });
}
static inline bool plan_conv_s2_tma(const ConvDesc& d, int num_sms, ConvParams& p) {
  return plan_with_split(p, num_sms, [&](ConvParams& q) { return plan_conv_s2_tma_impl(d, num_sms, q); });
}
static inline bool plan_conv_flat_tma(const ConvDesc& d, int num_sms, ConvParams& p) {
  return plan_with_split(p, num_sms, [&](ConvParams& q) { return plan_conv_flat_tma_impl(d, num_sms, q); });
}

// Tensor map of the flat mode: the activation matrix [rows, C] (pixel pitch `pitch`) as (C, rows, 1, 1).
static inline CUtensorMap make_flat_tensor_map(const __half* base, long rows, int C, int pitch, const ConvParams& p) {
  return make_halo_tensor_map(base, 1, 1, static_cast<int>(rows), C, pitch, p.hbox, 1, p.cb, p.sw);
}

// Same layer, fewer frames (the last chunk of a batch): keep every layout-determining choice of the full plan (K-block,
// rows per item, sub-tiles, stages -- the weight image and the tensor-map boxes were built for them) and shrink only the
// batch-dependent extents.
static inline ConvParams replan_for_batch(const ConvParams& full, int nb, int num_sms) {
  ConvParams p = full;
  p.B = nb;
  if (p.mode == MODE_FLAT_TMA) {
    p.flat_rows = nb * p.H * p.W;
    p.M_total = ceil_div(p.flat_rows, p.slots);
  } else if (p.mode == MODE_HALO_TMA || p.mode == MODE_S2_TMA) {
    p.M_total = (nb * p.tpi) << (p.upm ? 1 : 0);     // merged ConvTranspose: (row tile, row parity) items
  } else if (p.mode == MODE_HALO) {
    p.M_total = nb * p.Hp1 * p.Wp;
  } else {
    p.M_total = p.transposed ? nb * p.H * p.W : nb * p.Ho * p.Wo;
  }
  p.m_tiles = (p.mode == MODE_GATHER || p.mode == MODE_HALO) ? ceil_div(p.M_total, 128) : p.M_total;
  const int work = p.m_tiles * p.n_tiles;
  p.grid = work < num_sms ? work : num_sms;
  if (p.upm) p.grid &= ~1;
  return p;
}

// Physical byte offset of logical offset `off` inside a pattern-aligned swizzled buffer (Swizzle<sw,4,3>): the 16-byte
// chunk index (address bits 4..6) is XORed with address bits 7..9, masked to the swizzle width.
static inline size_t sw_phys(size_t off, int sw) {
  const size_t mask = (static_cast<size_t>(1) << sw) - 1;
  return off ^ (((off >> 7) & mask) << 4);
}

// Swizzled weight image: [n_tile][K-block ks][tap][n][cb channels], each (tap) tile swizzled like the A rows.
template <typename HalfT>
static inline void pack_conv_weights_sw(const ConvParams& p, const float* w, const float* bias, int cin_real, int cout_real,
                                        std::vector<HalfT>& wp, std::vector<float>& bp) {
  const int kps = p.kps > 1 ? p.kps : 1;
  const int nkb = p.nks * kps;                                      // K-blocks; a stage holds kps consecutive ones
  const size_t stage_elems = static_cast<size_t>(p.b_stage_bytes) / 2 / kps;
  wp.assign(static_cast<size_t>(p.n_tiles) * nkb * stage_elems, HalfT(0.0f));
  bp.assign(static_cast<size_t>(p.n_tiles) * p.Ntile, 0.0f);
  const int rb = p.cb * 2;
  for (int nt = 0; nt < p.n_tiles; ++nt)
    for (int ks = 0; ks < nkb; ++ks)
      for (int t = 0; t < p.taps; ++t)
        for (int n = 0; n < p.Ntile; ++n)
          for (int c = 0; c < p.cb; ++c) {
            const int ng = nt * p.Ntile + n, ci = ks * p.cb + c;
            if (ci >= cin_real) continue;
            float v;
            if (p.transposed) {                    // column = position (kh,kw) x output channel; weights [cin][cout][2][2]
              const int pos = ng / p.Cout, co = ng - pos * p.Cout;
              if (co >= cout_real) continue;
              v = w[((static_cast<size_t>(ci) * cout_real + co) * 2 + (pos >> 1)) * 2 + (pos & 1)];
            } else {
              if (ng >= cout_real) continue;
              v = w[(static_cast<size_t>(ng) * cin_real + ci) * p.taps + t];   // [cout][cin][kh][kw], t = kh*3+kw
            }
            const size_t off = (static_cast<size_t>(t) * p.Ntile + n) * rb + static_cast<size_t>(c) * 2;
            wp[(static_cast<size_t>(nt) * nkb + ks) * stage_elems + sw_phys(off, p.sw) / 2] = HalfT(v);
          }
  for (int ng = 0; ng < p.n_tiles * p.Ntile; ++ng) {
    const int co = p.transposed ? ng % p.Cout : ng;
    if (co < cout_real && bias) bp[ng] = bias[co];
  }
}

// ConvTranspose 2x2 / stride 2 (wt [ci][cm][2][2], bias bt [cm], no activation) followed by a 3x3 stride-1 convolution (w2
// [co][cm][3][3], bias b2 [co]) on the 2H x 2W map, as the parity convolutions of plan_conv_upmerge_tma; fp64 throughout.
// Tap (kh, kw) of output row 2y + dy reads upsampled row 2y + r, r = dy + kh - 1, i.e. input row y + floor(r / 2) at kernel
// row a = r mod 2 of the ConvTranspose (the same for columns), so
//   wm[dy][dx][th][tw][o][i] = sum over (kh, kw) landing on input tap (dy + th - 1, dx + tw - 1) of sum_c w2[o][c][kh][kw] wt[i][c][a][b].
// cv2 zero-pads the UPSAMPLED map, so bt contributes only through cv2's taps inside it: bm[0, co) is the interior bias
// b2 + sum_{kh,kw} w2[:, :, kh, kw] bt, bm[co (1 + cls) + o] the correction of border class cls = 3 rowc + colc (rowc: 0 inner
// row, 1 first, 2 last; colc likewise; cls 0 = interior, zero) -- minus the terms of the taps that fall outside.  Out-of-range
// taps of the INPUT need nothing: they are zeros (the TMA zero fill).
static inline void merge_upconv_weights(const float* wt, const float* bt, const float* w2, const float* b2, int ci, int cm, int co,
                                        std::vector<double>& wm, std::vector<double>& bm) {
  wm.assign(static_cast<size_t>(16) * co * ci, 0.0);
  bm.assign(static_cast<size_t>(10) * co, 0.0);
  for (int dy = 0; dy < 2; ++dy)
    for (int dx = 0; dx < 2; ++dx)
      for (int kh = 0; kh < 3; ++kh)
        for (int kw = 0; kw < 3; ++kw) {
          const int r = dy + kh - 1, s = dx + kw - 1;
          const int di = r < 0 ? -1 : r / 2, dj = s < 0 ? -1 : s / 2;
          const int a = r - 2 * di, b = s - 2 * dj;
          const int th = di - dy + 1, tw = dj - dx + 1;
          double* dst = wm.data() + static_cast<size_t>(((dy * 2 + dx) * 2 + th) * 2 + tw) * co * ci;
          for (int o = 0; o < co; ++o)
            for (int c = 0; c < cm; ++c) {
              const double w2v = w2[(static_cast<size_t>(o) * cm + c) * 9 + kh * 3 + kw];
              for (int i = 0; i < ci; ++i) dst[static_cast<size_t>(o) * ci + i] += w2v * wt[((static_cast<size_t>(i) * cm + c) * 2 + a) * 2 + b];
            }
        }
  std::vector<double> t(static_cast<size_t>(9) * co, 0.0);          // t[kh][kw][o] = sum_c w2[o][c][kh][kw] bt[c]
  for (int o = 0; o < co; ++o)
    for (int k = 0; k < 9; ++k)
      for (int c = 0; c < cm; ++c) t[static_cast<size_t>(k) * co + o] += static_cast<double>(w2[(static_cast<size_t>(o) * cm + c) * 9 + k]) * bt[c];
  for (int o = 0; o < co; ++o) {
    double s = b2 ? b2[o] : 0.0;
    for (int k = 0; k < 9; ++k) s += t[static_cast<size_t>(k) * co + o];
    bm[o] = s;
  }
  for (int cls = 1; cls < 9; ++cls) {
    const int rowc = cls / 3, colc = cls % 3;
    const int bad_kh = rowc == 1 ? 0 : (rowc == 2 ? 2 : -1), bad_kw = colc == 1 ? 0 : (colc == 2 ? 2 : -1);
    for (int o = 0; o < co; ++o) {
      double s = 0.0;
      for (int k = 0; k < 9; ++k)
        if (k / 3 == bad_kh || k % 3 == bad_kw) s -= t[static_cast<size_t>(k) * co + o];
      bm[static_cast<size_t>(co) * (1 + cls) + o] = s;
    }
  }
}

// Swizzled weight image of a merged plan: [dy][dx][tap = th * 2 + tw][n][64 channels], one row parity = one resident stage;
// each fp64 weight is rounded to fp16 once.
static inline void pack_upmerge_weights_sw(const ConvParams& p, const std::vector<double>& wm, int ci, int co, std::vector<__half>& wp) {
  const size_t stage_elems = static_cast<size_t>(p.b_stage_bytes) / 2;
  wp.assign(2 * stage_elems, __float2half(0.0f));
  const int rb = p.cb * 2;
  for (int dy = 0; dy < 2; ++dy)
    for (int dx = 0; dx < 2; ++dx)
      for (int tap = 0; tap < 4; ++tap)
        for (int n = 0; n < co; ++n)
          for (int c = 0; c < ci; ++c) {
            const double v = wm[((static_cast<size_t>((dy * 2 + dx) * 4 + tap)) * co + n) * ci + c];
            const size_t off = (static_cast<size_t>(dx * 4 + tap) * p.Ntile + n) * rb + static_cast<size_t>(c) * 2;
            wp[dy * stage_elems + sw_phys(off, p.sw) / 2] = __double2half(v);
          }
}

#ifdef __CUDACC__
// ---- PTX: TMA + bulk copy ----------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst_smem, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst_smem), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// MMAs of one pipeline stage for ONE 128-row sub-tile, issued by one thread.  MODE: 0 halo (3x3 s1), 1 parity planes
// (3x3 s2), 2 flat (1x1 / ConvT, kps K-blocks of one tap).  KJ = k16 steps per K-block.  a_sub / b_lo: low descriptor
// words (start address >> 4 | LBO field) of the sub-tile's first row and of the stage's first weight tile.
template <int MODE, int KJ>
__device__ __forceinline__ void issue_taps(uint32_t d_tmem, uint32_t a_sub, uint32_t b_lo, uint64_t hi_sw,
                                           uint32_t idesc, uint32_t acc0, uint32_t row16, uint32_t tap16, uint32_t wp16,
                                           uint32_t plane16, uint32_t blk16, int kps, uint64_t hi_a, uint32_t planex16) {
  uint32_t acc = acc0;
  if (MODE == 2) {
    for (int kb = 0; kb < kps; ++kb) {
#pragma unroll
      for (int j = 0; j < KJ; ++j) {
        umma_f16(d_tmem, hi_a | (a_sub + 2u * j), hi_sw | (b_lo + 2u * j), idesc, acc);
        acc = 1;
      }
      a_sub += blk16;
      b_lo += tap16;
      asm volatile("" : "+r"(a_sub), "+r"(b_lo));   // the next K-block's descriptors are computed after these MMAs were issued
    }
    return;
  }
  if (MODE == 3) {   // merged ConvTranspose (plan_conv_upmerge_tma): a_sub is this parity's tap (0, 0); tap (th, tw) = th Wp + tw rows on
#pragma unroll
    for (int th = 0; th < 2; ++th) {
#pragma unroll
      for (int tw = 0; tw < 2; ++tw) {
        const uint32_t a_tap = a_sub + th * wp16 + tw * row16;
#pragma unroll
        for (int j = 0; j < KJ; ++j) {
          umma_f16(d_tmem, hi_a | (a_tap + 2u * j), hi_sw | (b_lo + 2u * j), idesc, acc);
          acc = 1;
        }
        b_lo += tap16;
        asm volatile("" : "+r"(a_sub), "+r"(b_lo));
      }
    }
    return;
  }
#pragma unroll
  for (int kh = 0; kh < 3; ++kh) {
#pragma unroll
    for (int kw = 0; kw < 3; ++kw) {
      uint32_t a_tap;
      if (MODE == 0) a_tap = a_sub + kh * wp16 + (kw - 1) * row16;                       // row shift kh*Wp + kw - 1
      else a_tap = a_sub + (kh != 1 ? plane16 : 0u) + (kw != 1 ? planex16 : 0u) +        // plane (kh != 1, kw != 1): plane16 = two plane
                   (kh == 2 ? wp16 : 0u) - (kw == 0 ? row16 : 0u);                        // buffers, planex16 = one (pixel-pair rows: one
                                                                                          // buffer / the odd pixel's offset in the row);
                                                                                          // row shift (kh == 2) Wp - (kw == 0)
#pragma unroll
      for (int j = 0; j < KJ; ++j) {
        umma_f16(d_tmem, hi_a | (a_tap + 2u * j), hi_sw | (b_lo + 2u * j), idesc, acc);
        acc = 1;
      }
      b_lo += tap16;
      asm volatile("" : "+r"(a_sub), "+r"(b_lo));     // the next tap's descriptors are computed after this tap's MMAs were issued
    }
  }
}

// ---- epilogue ---------------------------------------------------------------------------------------------------
// One 16-channel unit of one pixel, specialised at compile time: accumulator -> (+ bias, SiLU) -> (+ residual) -> fp16 -> one
// 256-bit store.  hb16 (shared memory) holds 0.5 * bias when ACT (h = 0.5 acc + 0.5 bias is ONE FFMA).
template <bool ACT, bool RES>
__device__ __forceinline__ void tma_epilogue_unit(const uint32_t (&v)[16], const float (&hbr)[16], const __half* res, __half* out,
                                                  int probe, bool valid = true) {
  uint32_t o[8];
  if (probe & 2) {                         // PROBE builds only: store the raw accumulators
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      __half2 h = __floats2half2_rn(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1]));
      o[i] = *reinterpret_cast<uint32_t*>(&h);
    }
    st_global_256(out, o);
    return;
  }
  uint32_t rr[8];
  if (RES) ld_global_256(res, rr);         // issued first: in flight under the math
  if (ACT && (probe & 4)) {                // PROBE builds only: the same FP32-pipe work without the MUFU
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float ha = fmaf(__uint_as_float(v[2 * i]), 0.5f, hbr[2 * i]), hb = fmaf(__uint_as_float(v[2 * i + 1]), 0.5f, hbr[2 * i + 1]);
      __half2 h = __floats2half2_rn(fmaf(ha, ha, ha), fmaf(hb, hb, hb));
      o[i] = *reinterpret_cast<uint32_t*>(&h);
    }
  } else if (ACT) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 b4 = make_float4(hbr[4 * i], hbr[4 * i + 1], hbr[4 * i + 2], hbr[4 * i + 3]);
      o[2 * i] = silu_pack_from_half_arg(fmaf(__uint_as_float(v[4 * i]), 0.5f, b4.x), fmaf(__uint_as_float(v[4 * i + 1]), 0.5f, b4.y));
      o[2 * i + 1] = silu_pack_from_half_arg(fmaf(__uint_as_float(v[4 * i + 2]), 0.5f, b4.z), fmaf(__uint_as_float(v[4 * i + 3]), 0.5f, b4.w));
    }
    if (RES) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        __half2 s2 = __hadd2(*reinterpret_cast<__half2*>(&o[i]), *reinterpret_cast<const __half2*>(&rr[i]));
        o[i] = *reinterpret_cast<uint32_t*>(&s2);
      }
    }
  } else {
    float y[16];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 b4 = make_float4(hbr[4 * i], hbr[4 * i + 1], hbr[4 * i + 2], hbr[4 * i + 3]);
      y[4 * i] = __uint_as_float(v[4 * i]) + b4.x;
      y[4 * i + 1] = __uint_as_float(v[4 * i + 1]) + b4.y;
      y[4 * i + 2] = __uint_as_float(v[4 * i + 2]) + b4.z;
      y[4 * i + 3] = __uint_as_float(v[4 * i + 3]) + b4.w;
    }
    if (RES) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&rr[i]));
        y[2 * i] += f.x;
        y[2 * i + 1] += f.y;
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      __half2 h = __floats2half2_rn(y[2 * i], y[2 * i + 1]);
      o[i] = *reinterpret_cast<uint32_t*>(&h);
    }
  }
  if (probe & 1) {                         // PROBE builds only: keep the math alive without the store
    if ((o[0] ^ o[1] ^ o[2] ^ o[3] ^ o[4] ^ o[5] ^ o[6] ^ o[7]) == 0x12345678u) st_global_256(out, o);
    return;
  }
  if (valid) st_global_256(out, o);
}

// The epilogue warps' whole item loop, specialised on the destination kind (0: one tensor, 1: two tensors split at
// split_n -- fused siblings, 2: ConvTranspose scatter), the activation and the residual.  The per-unit code of the generic
// version was a long serial chain on the uniform datapath (kernel parameters re-read through LDCU, uniform compares and
// branches on act / res / transposed / split_n per 16-channel unit): the epilogue, not the tensor pipe or HBM, bounded every
// large layer at ~5 outputs per clock and SM.  Here everything that does not depend on the unit is resolved at compile time or
// hoisted out of the unit loop: a unit is one TMEM load, the math, one address and one store.
template <bool PROBE, int KIND, bool ACT, bool RES, bool BREG>
__device__ __forceinline__ void tma_epilogue_loop(const ConvParams& p, uint32_t tmem_base, uint64_t* tfull, uint64_t* tempty,
                                                  const float* bias_s, int nbuf, int warp, int lane, int total_work) {
  constexpr int G = TMA_EPI_GROUPS;
  const int ew = warp - TMA_FIRST_EPI_WARP;
  const int q = warp & 3;              // TMEM lane quadrant this warp may access
  const int grp = ew >> 2;             // unit k of an item (sub-tile u, 16-column chunk c; k = u * nch + c) goes to group k % G
  const int nsub = p.nsub, Ntile = p.Ntile, nch = Ntile >> 4, n_units = nsub * nch;
  const bool flat = p.mode == MODE_FLAT_TMA;
  const int Wp = p.Wp, Rr = p.R, Hh = p.H, Ww = p.W, slots = p.slots, flat_rows = p.flat_rows, tpi = p.tpi;
  const int Wo = p.Wo, Cout = p.Cout, n_tiles = p.n_tiles;
  const int out_pitch = p.out_pitch, out2_pitch = p.out2_pitch, res_pitch = p.res_pitch, split_n = p.split_n;
  __half* const outp = p.out;
  __half* const out2p = p.out2;
  const __half* const resp = p.res;
  const FastDiv fd_wp = p.fd_wp, fd_tpi = p.fd_hp1, fd_hw = p.fd_hw, fd_wo = p.fd_wo, fd_cout = p.fd_cout;
  const uint32_t lane_taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
  const bool no_store = PROBE && (p.dbg_skip & 2);
  const bool pipelined = !(PROBE && (p.dbg_skip & 8));   // probe switch 8: wait for every TMEM load right after issuing it
  const int probe_epi = PROBE ? (p.dbg_skip >> 4) & 15 : 0;  // probe switches 16 (no store) / 32 (no math) / 64 (no MUFU) / 128 (no TMEM loads)
  const bool ld_on = !(PROBE && (p.dbg_skip & 128));
  int gu0 = 0, gc0 = grp;              // first unit of this group
  while (gc0 >= nch) { gc0 -= nch; ++gu0; }
  // BREG: the number of chunks divides the number of groups, so this group only ever sees chunk grp % nch -- its 16 bias
  // values live in registers for the whole launch.  (Under load the tensor core's operand reads keep the shared-memory pipe
  // busy: the four LDS.128 of a unit were the longest single stall of the epilogue.)
  float hbr[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) hbr[i] = BREG ? bias_s[gc0 * 16 + i] : 0.f;
  // Accumulator set / use count of the current item, kept incrementally: `tcount % nbuf` and `tcount / nbuf` are integer
  // divisions by a kernel parameter (I2F + MUFU.RCP + fix-up, ~30 dependent instructions each) and were, together with the
  // per-item `G / nch`, a fifth of the stall samples of the thin layers' epilogue (ncu source page of b2.cv1).
  int buf_c = 0, use_c = 0;
  // BREG invariants (fixed chunk per group: nch divides G, n_tiles == 1): destination base, pitch, accumulator column
  const int breg_ustep = BREG ? (nch == 1 ? G : (nch == 2 ? G / 2 : (nch == 4 ? G / 4 : 1))) : 1;
  const int breg_n = gc0 * 16;
  __half* breg_gbase = outp + breg_n;
  int breg_gpitch = out_pitch;
  if (BREG) {
    if (KIND == 2) {
      const int pos = fd_div(fd_cout, breg_n);
      breg_gbase = outp + static_cast<size_t>((pos >> 1) * Wo + (pos & 1)) * out_pitch + (breg_n - pos * Cout);
    } else if (KIND == 1 && breg_n >= split_n) {
      breg_gbase = out2p + (breg_n - split_n);
      breg_gpitch = out2_pitch;
    }
  }
  long long e_wait = 0, e_work = 0, t0 = 0;
  pdl_wait();   // before the first residual read / output store
  for (int w = blockIdx.x; w < total_work; w += gridDim.x) {
    const int tile = w >> (n_tiles == 4 ? 2 : (n_tiles == 2 ? 1 : 0));   // n_tiles is 1, 2 or 4: work item = (row tile, N tile), N tile fastest
    const int n_tile = w & (n_tiles - 1);
    const int b = fd_div(fd_tpi, tile);
    const int y0 = (tile - b * tpi) * Rr;
    const int buf = buf_c;
    const int use = use_c;
    if (++buf_c == nbuf) { buf_c = 0; ++use_c; }
    // this lane's output pixel in each sub-tile (-1: padding column / row past the image / row past the matrix);
    // ConvTranspose: the top-left pixel of the 2x2 output block of input pixel (image, h, w)
    int pix[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      pix[u] = -1;
      if (u < nsub) {
        const int j = 128 * u + q * 32 + lane;
        if (flat) {
          const int m = tile * slots + j;
          if (m < flat_rows) pix[u] = m;
        } else {
          const int yy = fd_div(fd_wp, j);
          const int cc = j - yy * Wp;
          const int y = y0 + yy;
          if (yy < Rr && y < Hh && cc >= 1 && cc <= Ww) pix[u] = (b * Hh + y) * Ww + (cc - 1);
        }
        if (KIND == 2 && pix[u] >= 0) {
          const int m = pix[u];
          const int tb = fd_div(fd_hw, m);
          const int rem = m - tb * fd_hw.d;
          const int th = fd_div(fd_wo, rem);
          const int tw = rem - th * fd_wo.d;
          pix[u] = (tb * p.Ho + 2 * th) * Wo + 2 * tw;
        }
        if (no_store) pix[u] = -1;
      }
    }
    const int n_base = n_tile * Ntile;
    if (PROBE) t0 = clock64();
    mbar_wait(&tfull[buf], static_cast<uint32_t>(use) & 1u);
    if (PROBE) { e_wait += clock64() - t0; t0 = clock64(); }
    tc_fence_after();
    const uint32_t acc = lane_taddr + static_cast<uint32_t>(buf * nsub * Ntile);
    if constexpr (BREG) {
      // Fixed chunk per group (nch divides G): this group's units are chunk gc0 of sub-tiles gu0, gu0 + G / nch, ...  The
      // destination (tensor, channel offset, ConvTranspose position) is the same for all of them: one base pointer per
      // launch, one pixel offset per sub-tile, no per-unit control flow; lanes without a pixel run the math and skip the store.
      const int ustep = breg_ustep;
      const int n = breg_n;                                              // n_tiles == 1
      __half* const gbase = breg_gbase;
      const int gpitch = breg_gpitch;
      const uint32_t acc_g = acc + static_cast<uint32_t>(gc0 * 16);
      uint32_t va[16], vb[16];
      if (!ld_on) {
#pragma unroll
        for (int i = 0; i < 16; ++i) va[i] = vb[i] = 0x3f000000u + i + lane;
      }
      if (gu0 < nsub && ld_on) tmem_ld16(acc_g + static_cast<uint32_t>(gu0 * Ntile), va);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int u = gu0 + j * ustep;
        if (u >= nsub) break;
        if (ld_on) tmem_ld_wait();
        const int un = u + ustep;
        if (un < nsub && ld_on) tmem_ld16(acc_g + static_cast<uint32_t>(un * Ntile), (j & 1) ? va : vb);
        if (!pipelined) tmem_ld_wait();
        const int px = u == 0 ? pix[0] : (u == 1 ? pix[1] : (u == 2 ? pix[2] : pix[3]));
        const size_t pxs = static_cast<size_t>(px < 0 ? 0 : px);
        tma_epilogue_unit<ACT, RES>((j & 1) ? vb : va, hbr, RES ? resp + pxs * res_pitch + n : nullptr, gbase + pxs * gpitch, probe_epi,
                                    px >= 0);
      }
      tc_fence_before();
      __syncwarp();
      if (elect_one()) mbar_arrive(&tempty[buf]);
      if (PROBE) e_work += clock64() - t0;
      continue;
    }
    // generic path (chunks not fixed per group): the bias of a unit is read from shared memory at the point of use -- fetching
    // it one unit ahead needs 16 more registers and spills at the 80-register cap of a 21-warp CTA (measured slower)
    auto finish_unit = [&](const uint32_t (&v)[16], int u, int c) {
      const int px = u == 0 ? pix[0] : (u == 1 ? pix[1] : (u == 2 ? pix[2] : pix[3]));
      if (px < 0) return;
      const int n = n_base + c * 16;
      float hb[16];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 b4 = reinterpret_cast<const float4*>(bias_s + n)[i];
        hb[4 * i] = b4.x; hb[4 * i + 1] = b4.y; hb[4 * i + 2] = b4.z; hb[4 * i + 3] = b4.w;
      }
      __half* dst;
      if (KIND == 2) {                               // column chunk -> output position (pos >> 1, pos & 1) and channel
        const int pos = fd_div(fd_cout, n);
        const int co = n - pos * Cout;
        dst = outp + static_cast<size_t>(px + (pos >> 1) * Wo + (pos & 1)) * out_pitch + co;
      } else if (KIND == 1 && n >= split_n) {
        dst = out2p + static_cast<size_t>(px) * out2_pitch + (n - split_n);
      } else {
        dst = outp + static_cast<size_t>(px) * out_pitch + n;
      }
      tma_epilogue_unit<ACT, RES>(v, hb, RES ? resp + static_cast<size_t>(px) * res_pitch + n : nullptr, dst, probe_epi);
    };
    // software pipeline over this group's units (unit k = u * nch + c lives at accumulator column 16 k): the TMEM load of
    // the next unit is in flight while the current one is converted and stored
    int u = gu0, c = gc0, k = grp;
    uint32_t va[16], vb[16];
    if (!ld_on) {
#pragma unroll
      for (int i = 0; i < 16; ++i) va[i] = vb[i] = 0x3f000000u + i + lane;
    }
    if (k < n_units && ld_on) tmem_ld16(acc + static_cast<uint32_t>(16 * k), va);
    while (k < n_units) {
      int u2 = u, c2 = c + G;
      while (c2 >= nch) { c2 -= nch; ++u2; }
      if (ld_on) tmem_ld_wait();
      if (k + G < n_units && ld_on) tmem_ld16(acc + static_cast<uint32_t>(16 * (k + G)), vb);
      if (!pipelined) tmem_ld_wait();
      finish_unit(va, u, c);
      k += G;
      if (k >= n_units) break;
      u = u2; c = c2;
      c2 = c + G;
      while (c2 >= nch) { c2 -= nch; ++u2; }
      if (ld_on) tmem_ld_wait();
      if (k + G < n_units && ld_on) tmem_ld16(acc + static_cast<uint32_t>(16 * (k + G)), va);
      if (!pipelined) tmem_ld_wait();
      finish_unit(vb, u, c);
      k += G;
      u = u2; c = c2;
    }
    tc_fence_before();
    __syncwarp();
    if (elect_one()) mbar_arrive(&tempty[buf]);
    if (PROBE) e_work += clock64() - t0;
  }
  if (PROBE && p.dbg_clk && warp == TMA_FIRST_EPI_WARP && lane == 0) {
    p.dbg_clk[blockIdx.x * 12 + 6] = e_wait;
    p.dbg_clk[blockIdx.x * 12 + 7] = e_work;
  }
}

// Epilogue of a launch with a fused trailing 1x1 convolution (ConvParams::tail_n; main layer 3x3 stride 1 with Ntile = N1 = 64,
// the 1x1 with N2 = tail_n = 32).  Group g owns chunk g % (N1/16) of the sub-tiles g / (N1/16), + 4/(N1/16), ...:
//   pass 1: 16 accumulator columns -> + bias, SiLU -> 16 fp16 values = 8 packed columns, written BACK into tensor memory inside
//           the group's own, already consumed, 16-column range -> tready;
//   the sub-tile's MMA warp then runs D2 = A[TMEM] x W2^T (issue_tail in the kernel);
//   pass 2 (after t2full): 16 channels of the 1x1 per unit -> + bias2, (SiLU) -> one 32-byte store -> tempty.
// In place (proto.cv2 -> cv3, TMEM full): packed columns 64u + {0, 24, 32, 56}, D2 as two N = 16 halves in the freed runs
// [8, 24) and [40, 56) of the same 64 columns.  The intermediate never reaches shared or global memory.
__device__ __forceinline__ uint32_t tail_pack_col(int c) { return c == 0 ? 0u : (c == 1 ? 24u : (c == 2 ? 32u : 56u)); }
// UPM (merged ConvTranspose, plan_conv_upmerge_tma): virtual sub-tile u = 2 (128-row sub-tile) + column parity, row parity dy =
// item & 1; a lane's halo position (y, x) goes to output pixel (2y + dy, 2x + dx), and the 16 accumulators of a pixel on the
// border of the output map get its class's correction (corr_s [9][64]) added before the bias -- only those lanes do it.
template <bool PROBE, bool UPM>
__device__ __forceinline__ void tma_epilogue_loop_tail(const ConvParams& p, uint32_t tmem_base, uint64_t* tfull, uint64_t* tempty,
                                                       uint64_t* tready, uint64_t* t2full, const float* bias_s, int warp, int lane,
                                                       int total_work) {
  constexpr int G = TMA_EPI_GROUPS;
  const int ew = warp - TMA_FIRST_EPI_WARP;
  const int q = warp & 3;
  const int g = ew >> 2;
  const int nsub = p.nsub, N1 = p.Ntile, N2 = p.tail_n;
  const int nch1 = N1 >> 4, nch2 = N2 >> 4;
  const int c1 = g % nch1, u1 = g / nch1, step1 = G / nch1;     // pass 1: chunk c1 of sub-tiles u1, u1 + step1, ...
  const int c2 = g % nch2, u2 = g / nch2, step2 = G / nch2;     // pass 2: chunk c2 of the 1x1's channels, sub-tiles u2, ...
  const int Wp = p.Wp, Rr = p.R, Hh = p.H, Ww = p.W, tpi = p.tpi;
  const int out_pitch = p.out_pitch;
  __half* const outp = p.out;
  const FastDiv fd_wp = p.fd_wp, fd_tpi = p.fd_hp1;
  const uint32_t lane_taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
  const uint32_t pk_col = tail_pack_col(c1);
  const float* corr_s = reinterpret_cast<const float*>(reinterpret_cast<const uint8_t*>(bias_s) - 256 + p.smem_off_corr);   // UPM only
  float hbr[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) hbr[i] = bias_s[c1 * 16 + i];
  int tcount = 0;
  long long e_wait = 0, e_work = 0, t0 = 0;
  pdl_wait();
  for (int w = blockIdx.x; w < total_work; w += gridDim.x, ++tcount) {
    const int tile = UPM ? w >> 1 : w;
    const int b = fd_div(fd_tpi, tile);
    const int y0 = (tile - b * tpi) * Rr;
    const int buf = tcount & 1;
    const uint32_t use = static_cast<uint32_t>(tcount >> 1);
    int pix[4];
    uint32_t cls4 = 0;                 // UPM: border class of each virtual sub-tile's pixel, 4 bits each
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      pix[u] = -1;
      if (u < nsub) {
        const int j = 128 * (UPM ? u >> 1 : u) + q * 32 + lane;
        const int yy = fd_div(fd_wp, j);
        const int cc = j - yy * Wp;
        const int y = y0 + yy;
        if (yy < Rr && y < Hh && cc >= 1 && cc <= Ww) {
          if (UPM) {
            const int oy = 2 * y + (w & 1), ox = 2 * (cc - 1) + (u & 1), Ho = 2 * Hh, Wo = 2 * Ww;
            pix[u] = (b * Ho + oy) * Wo + ox;
            const uint32_t cls = 3u * (oy == 0 ? 1u : (oy == Ho - 1 ? 2u : 0u)) + (ox == 0 ? 1u : (ox == Wo - 1 ? 2u : 0u));
            cls4 |= cls << (4 * u);
          } else {
            pix[u] = (b * Hh + y) * Ww + (cc - 1);
          }
        }
      }
    }
    if (PROBE) t0 = clock64();
    mbar_wait(&tfull[buf], use & 1u);
    if (PROBE) { e_wait += clock64() - t0; t0 = clock64(); }
    tc_fence_after();
    const uint32_t acc = lane_taddr + static_cast<uint32_t>(buf * nsub * N1);
    // ---- pass 1: accumulators -> packed fp16 in tensor memory.  One 16-register buffer: the next unit's TMEM load is issued as
    // soon as the current values are packed (the double-buffered form spilled at the 80-register cap and the spill reloads
    // -- local memory behind an L1 the TMA traffic keeps busy -- were the longest stalls of this loop).
    {
      uint32_t v[16];
      if (u1 < nsub) tmem_ld16(acc + static_cast<uint32_t>(u1 * N1 + 16 * c1), v);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int u = u1 + k * step1;
        if (u >= nsub) break;
        tmem_ld_wait();
        if (UPM) {
          const uint32_t cls = (cls4 >> (4 * u)) & 15u;
          if (cls) {
            const float* cv = corr_s + cls * 64u + c1 * 16;
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) + cv[i]);
          }
        }
        uint32_t o[8];
#pragma unroll
        for (int i = 0; i < 8; ++i)
          o[i] = silu_pack_from_half_arg(fmaf(__uint_as_float(v[2 * i]), 0.5f, hbr[2 * i]), fmaf(__uint_as_float(v[2 * i + 1]), 0.5f, hbr[2 * i + 1]));
        if (u + step1 < nsub) tmem_ld16(acc + static_cast<uint32_t>((u + step1) * N1 + 16 * c1), v);
        tmem_st8(acc + static_cast<uint32_t>(u * N1) + pk_col, o);
      }
      tmem_st_wait();
    }
    tc_fence_before();
    __syncwarp();
    if (elect_one()) mbar_arrive(&tready[buf]);
    // ---- pass 2: the 1x1's channels
    float hb2[16];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 b4 = reinterpret_cast<const float4*>(bias_s + 256 + 16 * c2)[i];
      hb2[4 * i] = b4.x; hb2[4 * i + 1] = b4.y; hb2[4 * i + 2] = b4.z; hb2[4 * i + 3] = b4.w;
    }
    mbar_wait(&t2full[buf], use & 1u);
    tc_fence_after();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int u = u2 + k * step2;
      if (u >= nsub) break;
      const uint32_t d2 = acc + static_cast<uint32_t>(u * N1) + (c2 ? 40u : 8u);
      uint32_t v[16];
      tmem_ld16(d2, v);
      tmem_ld_wait();
      const int px = u == 0 ? pix[0] : (u == 1 ? pix[1] : (u == 2 ? pix[2] : pix[3]));
      const size_t pxs = static_cast<size_t>(px < 0 ? 0 : px);
      __half* dst = outp + pxs * out_pitch + 16 * c2;
      if (p.tail_act) tma_epilogue_unit<true, false>(v, hb2, nullptr, dst, 0, px >= 0);
      else tma_epilogue_unit<false, false>(v, hb2, nullptr, dst, 0, px >= 0);
    }
    tc_fence_before();
    __syncwarp();
    if (elect_one()) mbar_arrive(&tempty[buf]);
    if (PROBE) e_work += clock64() - t0;
  }
  if (PROBE && p.dbg_clk && warp == TMA_FIRST_EPI_WARP && lane == 0) {
    p.dbg_clk[blockIdx.x * 12 + 6] = e_wait;
    p.dbg_clk[blockIdx.x * 12 + 7] = e_work;
  }
}

// ---- the kernel --------------------------------------------------------------------------------------------------
// PROBE = true (libxrseg_debug.so only, tools/probe_tma.py): per-role clock64() counters (p.dbg_clk) and the p.dbg_skip
// switches (1 = no MMAs, 2 = no stores, 4 = no TMA loads, 8 = software-pipelined epilogue).  The product instantiation
// contains none of it.
template <bool PROBE>
__global__ void __launch_bounds__(TMA_THREADS, 1)
conv_halo_tma_kernel(const __grid_constant__ ConvParams p, const __grid_constant__ TmapSet tmaps) {
  const CUtensorMap& tmap = tmaps.m[0];
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);       // [8]
  uint64_t* empty = full + 8;                               // [8]
  uint64_t* tfull = empty + 8;                              // [2]
  uint64_t* tempty = tfull + 4;                             // [4]
  uint64_t* bres = tempty + 4;                              // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bres + 1);
  uint64_t* tready = reinterpret_cast<uint64_t*>(smem + 208);   // [2] tail: packed intermediate of an item is in tensor memory
  uint64_t* t2full = tready + 2;                                // [2] tail: the 1x1 layer's accumulators are complete
  float* bias_s = reinterpret_cast<float*>(smem + 256);     // [<=512]; the tail's bias lives at [256, 256 + tail_n)
  uint8_t* smem_b = smem + p.smem_off_b;
  uint8_t* smem_a = smem + p.smem_off_a;

  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // provably warp-uniform: role code uses the uniform datapath
  const int lane = tid & 31;
  const int total_work = p.total_work;        // = m_tiles * n_tiles (launch_conv_halo_tma)

  const int n_issuers = p.sw ? p.nsub : 1;    // MMA-issuing warps (swizzled path: one per sub-tile)
  const int nbuf = p.nbuf;                    // TMEM accumulator sets in flight (>= 2: launch_conv_halo_tma)
  if (tid == 0) {
    for (int i = 0; i < CONV_MAX_STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], n_issuers);       // every issuer commits the stage it has consumed
    }
    for (int i = 0; i < 4; ++i) {
      mbar_init(&tfull[i], n_issuers);       // ... and the accumulators it has finished
      mbar_init(&tempty[i], TMA_EPI_WARPS);  // one arrival per epilogue warp
    }
    mbar_init(bres, 1);
    if (p.tail_n) {
      for (int i = 0; i < 2; ++i) {
        mbar_init(&tready[i], TMA_EPI_WARPS);
        mbar_init(&t2full[i], n_issuers);
      }
    }
    mbar_fence_init();
    prefetch_tensormap(&tmap);
    if (p.mode == MODE_S2_TMA)
      for (int i = 1; i < (p.pair ? 2 : 4); ++i) prefetch_tensormap(&tmaps.m[i]);
    if (p.b_resident) {
      // resident weights: fetched first thing (they are constants: no dependence on the previous kernel), so the copy
      // runs while warp 1 allocates TMEM -- which may have to wait for a co-resident CTA of the previous kernel
      const uint32_t bytes = static_cast<uint32_t>(p.nks) * p.b_stage_bytes;
      const uint32_t tail_bytes = p.tail_n ? static_cast<uint32_t>(p.tail_n) * static_cast<uint32_t>(p.Ntile) * 2u : 0u;   // W2: tail_n rows of Ntile channels
      const uint32_t b_dst = smem_u32(smem_b);
      // merged ConvTranspose: the image holds both row parities; this CTA's items all have parity blockIdx.x & 1 (even grid)
      const uint8_t* b_src = reinterpret_cast<const uint8_t*>(p.wpack) + (p.upm ? (blockIdx.x & 1u) * bytes : 0u);
      mbar_arrive_expect_tx(bres, bytes + tail_bytes);
      for (uint32_t off = 0; off < bytes; off += 32768u) {
        const uint32_t n = bytes - off < 32768u ? bytes - off : 32768u;
        bulk_copy_g2s(b_dst + off, b_src + off, n, bres);
      }
      if (tail_bytes) bulk_copy_g2s(smem_u32(smem + p.smem_off_w2), p.tail_w, tail_bytes, bres);
    }
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, static_cast<uint32_t>(p.tmem_cols));
    tmem_relinquish();
  }
  // bias for the epilogue; activated layers keep 0.5 * bias (epilogue_chunk16_hb: h = 0.5 acc + 0.5 bias in one FFMA)
  for (int i = tid; i < p.n_tiles * p.Ntile; i += TMA_THREADS) bias_s[i] = p.act ? 0.5f * p.bias[i] : p.bias[i];
  for (int i = tid; i < p.tail_n; i += TMA_THREADS) bias_s[256 + i] = p.tail_act ? 0.5f * p.tail_bias[i] : p.tail_bias[i];
  if (p.upm)   // merged ConvTranspose: the border corrections, added to the accumulator (tma_epilogue_loop_tail)
    for (int i = tid; i < 9 * 64; i += TMA_THREADS) reinterpret_cast<float*>(smem + p.smem_off_corr)[i] = p.bias[p.n_tiles * p.Ntile + i];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // Only now may the next kernel's CTAs start (PDL): a dependent CTA that became co-resident and grabbed TMEM columns
  // before this CTA had its own would wait for this kernel to finish while this CTA waits for its columns -- deadlock.
  pdl_launch_dependents();

  if (warp == 0) {
    // ======================================= TMA producer ========================================
    if (lane == 0) {
      const uint32_t a_u32 = smem_u32(smem_a);
      const uint32_t b_u32 = smem_u32(smem_b);
      const uint32_t a_tx = static_cast<uint32_t>(p.cps) * p.slots * 16u * (p.kps > 1 ? p.kps : 1) *   // slots * row bytes (* K-blocks)
                            (p.mode == MODE_S2_TMA ? 4u : 1u);                                           // (* parity planes)
      const uint32_t b_stride = p.sw ? static_cast<uint32_t>((p.b_stage_bytes + 1023) & ~1023) : static_cast<uint32_t>(p.b_stage_bytes);
      pdl_wait();   // the weights above are constants; the activations below are the previous kernels' output
      // ring position kept incrementally (slot = it % S, round = it / S): the divisions by the kernel parameter S cost the
      // single producer / issuer thread ~60 dependent instructions per stage hand-over
      int slot_c = 0;
      uint32_t round_c = 0;
      long long t_wait = 0, t0 = 0;
      const bool flat = p.mode == MODE_FLAT_TMA;
      const int S = p.S;
      for (int w = blockIdx.x; w < total_work; w += gridDim.x) {
        const int tile = w >> (p.upm ? 1 : (p.n_tiles == 4 ? 2 : (p.n_tiles == 2 ? 1 : 0)));   // upm: (row tile, row parity)
        const int n_tile = w & (p.n_tiles - 1);
        const int b = fd_div(p.fd_hp1, tile);
        const int y0 = (tile - b * p.tpi) * p.R;
        for (int ks = 0; ks < p.nks; ++ks) {
          const int slot = slot_c;
          const uint32_t round = round_c;
          if (++slot_c == S) { slot_c = 0; ++round_c; }
          if (PROBE) t0 = clock64();
          if (round > 0) mbar_wait(&empty[slot], (round - 1u) & 1u);
          if (PROBE) {
            t_wait += clock64() - t0;
            if (p.dbg_skip & 4) { mbar_arrive(&full[slot]); continue; }
          }
          mbar_arrive_expect_tx(&full[slot], a_tx + (p.b_resident ? 0u : static_cast<uint32_t>(p.b_stage_bytes)));
          const uint32_t a_dst = a_u32 + slot * p.a_stage_bytes;
          if (p.mode == MODE_S2_TMA) {
            // four parity planes: columns xs = -1 .. Wo-1, rows ys = y0 - py .. y0 - py + R  (y0 = first OUTPUT row)
            if (p.pair) {   // two row-parity planes of pixel-pair rows (nks == 1)
              for (int pl = 0; pl < 2; ++pl) tma_load_4d(a_dst + pl * p.lbo_a, &tmaps.m[pl], &full[slot], 0, -1, y0 - pl, b);
            } else {
              for (int pl = 0; pl < 4; ++pl)
                tma_load_4d(a_dst + pl * p.lbo_a, &tmaps.m[pl], &full[slot], ks * p.cb, -1, y0 - (pl >> 1), b);
            }
          } else if (flat) {
            // rows [tile*slots, +slots) of the activation matrix, hbox rows per box, kps K-blocks per stage; rows past
            // the end and channels past Cin arrive as zeros
            const uint32_t box_bytes = static_cast<uint32_t>(p.hbox) * p.cb * 2u;
            uint32_t dst = a_dst;
            for (int kb = 0; kb < p.kps; ++kb)
              for (int r0 = 0; r0 < p.slots; r0 += p.hbox, dst += box_bytes)
                tma_load_4d(dst, &tmap, &full[slot], (ks * p.kps + kb) * p.cb, tile * p.slots + r0, 0, 0);
          } else if (p.sw) {
            tma_load_4d(a_dst, &tmap, &full[slot], ks * p.cb, -1, y0 - 1, b);     // the whole K-block in one box
          } else {
            for (int c = 0; c < p.cps; ++c)
              tma_load_4d(a_dst + c * p.lbo_a, &tmap, &full[slot], ks * p.cb + c * 8, -1, y0 - 1, b);
          }
          if (!p.b_resident) {
            const uint8_t* src = reinterpret_cast<const uint8_t*>(p.wpack) +
                                 (static_cast<size_t>(n_tile) * p.nks + ks) * p.b_stage_bytes;
            const uint32_t b_dst = b_u32 + slot * b_stride;
            for (uint32_t off = 0; off < static_cast<uint32_t>(p.b_stage_bytes); off += 32768u) {
              const uint32_t n = p.b_stage_bytes - off < 32768u ? p.b_stage_bytes - off : 32768u;
              bulk_copy_g2s(b_dst + off, src + off, n, &full[slot]);
            }
          }
        }
      }
      if (PROBE && p.dbg_clk) p.dbg_clk[blockIdx.x * 12 + 0] = t_wait;
    }
  } else if (warp < TMA_FIRST_EPI_WARP) {
    // ======================================= MMA issuers =========================================
    // warp 1 + u owns sub-tile u (its own TMEM accumulator): same waits, its own MMAs, its own commits
    const int my_u = warp - 1;
    if (my_u < n_issuers)
    // all 32 lanes run the loop (uniform control flow); one elected lane issues the tcgen05 instructions
    {
      const uint32_t a_u32 = smem_u32(smem_a);
      const uint32_t b_u32 = smem_u32(smem_b);
      const uint32_t lbo_a16 = static_cast<uint32_t>(p.lbo_a) >> 4;
      const uint32_t lbo_b16 = static_cast<uint32_t>(p.Ntile);
      const uint32_t desc_hi = (128u >> 4) | (1u << 14);
      const int kj = p.cb >> 4;
      const uint32_t idesc = p.idesc;
      const uint32_t ntile_u = static_cast<uint32_t>(p.Ntile);
      const uint32_t rb = static_cast<uint32_t>(p.cb) * 2u;                 // swizzled row bytes of a K-block (weights; operand rows unless paired)
      const uint32_t rba = p.pair ? 2u * rb : rb;                            // operand row bytes (pixel-pair rows: two K-blocks wide)
      const uint32_t row16 = rba >> 4;                                       // one operand row in 16-byte units
      const uint32_t sub16 = 128u * row16;                                   // one 128-row sub-tile
      const uint32_t tap16 = (ntile_u * rb) >> 4;                            // one tap's weight tile
      const uint32_t b_stride_sw = static_cast<uint32_t>((p.b_stage_bytes + 1023) & ~1023);
      const uint32_t layout = p.sw == 3 ? 2u : (p.sw == 2 ? 4u : 6u);
      const uint64_t hi_sw = static_cast<uint64_t>(((8u * rb) >> 4) | (1u << 14) | (layout << 29)) << 32;
      const uint32_t layout_a = p.pair ? (p.sw == 2 ? 2u : 4u) : layout;   // pair: the swizzle one step wider than the weights'
      const uint64_t hi_a = static_cast<uint64_t>(((8u * rba) >> 4) | (1u << 14) | (layout_a << 29)) << 32;
      const bool mma_on = !PROBE || !(p.dbg_skip & 1);
      long long t_start = 0, t_bres = 0, t_tempty = 0, t_full = 0, t_issue = 0, t_fence = 0, t_commit = 0, t0 = 0;
      long long g_start = 0;
      if (PROBE) {
        t_start = clock64();
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g_start));
      }
      if (p.b_resident) mbar_wait(bres, 0);
      if (PROBE) t_bres = clock64() - t_start;
      // Fused trailing 1x1 (tail): item j's packed intermediate sits in this sub-tile's accumulator columns 64 u + {0, 24, 32, 56}
      // (8 columns = one K step of 16 channels each); D2 = A[TMEM] x W2^T as two N = 16 halves into the freed column runs
      // [8, 24) and [40, 56).  W2: [32 rows][128 bytes], 128-byte swizzle; a half starts 16 rows = 2048 bytes further.
      // blocking = false: only if the epilogue has already delivered item j (polled between the K stages of the next item, so
      // that the 1x1's accumulators are read out and the buffer is free again BEFORE the next item's MMAs finish -- otherwise
      // the tensor pipe idles through the whole second epilogue pass of every item)
      auto issue_tail = [&](int j, bool blocking) -> bool {
        const int jb = j & 1;
        const uint32_t ph = static_cast<uint32_t>(j >> 1) & 1u;
        if (blocking) mbar_wait(&tready[jb], ph);
        else if (!__any_sync(0xffffffffu, mbar_test_wait(&tready[jb], ph))) return false;
        tc_fence_after();
        if (elect_one()) {
          const int N1 = p.Ntile;
          const uint32_t accj = tmem_base + static_cast<uint32_t>((jb * p.nsub + my_u) * N1);
          const uint32_t w2 = smem_u32(smem + p.smem_off_w2);
          // W2: [N2 rows][N1 channels] fp16, K-major, rows of N1 * 2 bytes in the hardware swizzle of that width
          const uint32_t rb2 = static_cast<uint32_t>(N1) * 2u;
          const uint64_t hi2 = static_cast<uint64_t>(((8u * rb2) >> 4) | (1u << 14) | ((rb2 == 128u ? 2u : 4u) << 29)) << 32;
          const uint32_t idesc16 = umma_idesc_f16(16, 0);
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            const uint32_t b_lo2 = (((w2 + static_cast<uint32_t>(hh) * 16u * rb2) >> 4) & 0x3FFFu) | (1u << 16);
            const uint32_t d2 = accj + (hh ? 40u : 8u);
#pragma unroll
            for (int j2 = 0; j2 < 4; ++j2)
              umma_f16_ts(d2, accj + tail_pack_col(j2), hi2 | (b_lo2 + 2u * j2), idesc16, j2 > 0 ? 1u : 0u);
          }
          umma_commit(&t2full[jb]);
        }
        __syncwarp();
        return true;
      };
      // Per-launch constants of the swizzled issue loop.  The issuing warps all wait for the same operand barrier, so whatever
      // they execute between that barrier and their first tcgen05.mma is time the tensor pipe may run dry: the per-stage
      // arithmetic is reduced to two multiply-adds here, and issue_taps keeps the descriptor arithmetic of tap t + 1 BEHIND the
      // MMAs of tap t (the compiler used to hoist all 18..72 descriptor words of a stage above its first MMA: ~280 instructions
      // in lockstep on all four issuers per 1152 cycles of tensor work in proto.cv2 -- ncu source page, gpurun_out s11).
      uint32_t c_a_stage16 = static_cast<uint32_t>(p.a_stage_bytes) >> 4;
      uint32_t c_b_step16 = (p.b_resident ? static_cast<uint32_t>(p.b_stage_bytes) : b_stride_sw) >> 4;
      uint32_t c_a_lo = (((a_u32 >> 4) & 0x3FFFu) | (1u << 16)) + static_cast<uint32_t>(my_u) * sub16;
      uint32_t c_b_lo = ((b_u32 >> 4) & 0x3FFFu) | (1u << 16);
      uint32_t c_d_off = static_cast<uint32_t>(my_u) * ntile_u;
      uint32_t c_sel = static_cast<uint32_t>((p.mode == MODE_HALO_TMA ? 0 : p.mode == MODE_S2_TMA ? 4 : 8) + (kj == 4 ? 2 : kj == 2 ? 1 : 0));
      uint32_t c_bres = p.b_resident ? 1u : 0u;
      const uint32_t c_wp16 = static_cast<uint32_t>(p.Wp) * row16;
      if (p.upm) {
        // merged ConvTranspose: warp my_u = 2 u + dx computes column parity dx of sub-tile u for the CTA's row parity dy; its tap
        // (0, 0) is halo row j + dy Wp + dx - 1, its weights the dx half of the resident stage (four taps)
        const uint32_t dy = blockIdx.x & 1u, dx = static_cast<uint32_t>(my_u) & 1u;
        c_a_lo = (((a_u32 >> 4) & 0x3FFFu) | (1u << 16)) + (static_cast<uint32_t>(my_u) >> 1) * sub16 + dy * c_wp16 + dx * row16 - row16;
        c_b_lo += dx * 4u * tap16;
        c_sel = 12;
      }
      const uint32_t c_planex16 = p.pair ? (rb >> 4) : static_cast<uint32_t>(p.lbo_a) >> 4;      // x parity: odd pixel inside the row / one plane buffer
      const uint32_t c_plane16 = p.pair ? static_cast<uint32_t>(p.lbo_a) >> 4 : 2u * (static_cast<uint32_t>(p.lbo_a) >> 4);   // y parity
      const uint32_t c_blk16 = static_cast<uint32_t>(p.slots) * row16;
      const int c_kps = p.kps > 1 ? p.kps : 1;
      int tail_pending = -1;                      // item whose 1x1 has not been issued yet
      int tcount = 0;
      int slot_c = 0, buf_c = 0, use_c = 0;       // ring slot / accumulator set, kept incrementally (no divisions by S / nbuf)
      uint32_t round_c = 0;
      const int S = p.S;
      for (int w = blockIdx.x; w < total_work; w += gridDim.x, ++tcount) {
        const int buf = buf_c;
        const int use = use_c;
        if (++buf_c == nbuf) { buf_c = 0; ++use_c; }
        if (PROBE) t0 = clock64();
        if (use >= 1) mbar_wait(&tempty[buf], static_cast<uint32_t>(use - 1) & 1u);
        if (PROBE) t_tempty += clock64() - t0;
        tc_fence_after();
        const uint32_t d_base = tmem_base + static_cast<uint32_t>(buf * p.nsub * p.Ntile);
        for (int ks = 0; ks < p.nks; ++ks) {
          const int slot = slot_c;
          const uint32_t round = round_c;
          if (++slot_c == S) { slot_c = 0; ++round_c; }
          if (PROBE) t0 = clock64();
          mbar_wait(&full[slot], round & 1u);
          if (PROBE) { t_full += clock64() - t0; t0 = clock64(); }
          tc_fence_after();
          if (PROBE) { t_fence += clock64() - t0; t0 = clock64(); }
          const uint32_t a_base = a_u32 + slot * p.a_stage_bytes;
          if (p.sw) {
            // swizzled operands: row = K-block of cb channels (rb bytes); tap = row shift; k16 step = +32 bytes.
            // Measured on B200: the UMMA swizzle is a function of the ABSOLUTE shared-memory address bits (like the
            // TMA write side), so a descriptor may start at any row with the base-offset field left 0; filling that
            // field with (addr >> 7) & 7 for unaligned starts produces wrong results.
            // descriptor low words: start address >> 4 plus offsets in 16-byte units (never carries out of bits 0-13; the
            // stage buffers are 1024-byte aligned and a weight stage is a multiple of 16 bytes, so the shifts distribute)
            uint32_t b_lo = c_b_lo + static_cast<uint32_t>(c_bres ? ks : slot) * c_b_step16;
            // Loop order: sub-tile innermost, so that consecutive MMAs target different accumulators.  Everything is
            // unrolled with guards folded into the issue predicate: a handful of uniform adds per MMA, no branches.
            if (elect_one()) {   // one branch per stage; inside, a single lane issues the whole MMA batch
              if (mma_on) {
                const uint32_t a_sub = c_a_lo + static_cast<uint32_t>(slot) * c_a_stage16;
                const uint32_t d_tmem = d_base + c_d_off;
                const uint32_t acc0 = ks > 0 ? 1u : 0u;
                // straight-line issue code per (mode, k16 steps): the issuing thread is the bottleneck of thin layers, so
                // everything but the two descriptor adds per MMA is resolved at compile time
                switch (c_sel) {
                  case 0: issue_taps<0, 1>(d_tmem, a_sub, b_lo, hi_sw, idesc, acc0, row16, tap16, c_wp16, c_plane16, c_blk16, c_kps, hi_a, c_planex16); break;
                  case 1: issue_taps<0, 2>(d_tmem, a_sub, b_lo, hi_sw, idesc, acc0, row16, tap16, c_wp16, c_plane16, c_blk16, c_kps, hi_a, c_planex16); break;
                  case 2: issue_taps<0, 4>(d_tmem, a_sub, b_lo, hi_sw, idesc, acc0, row16, tap16, c_wp16, c_plane16, c_blk16, c_kps, hi_a, c_planex16); break;
                  case 4: issue_taps<1, 1>(d_tmem, a_sub, b_lo, hi_sw, idesc, acc0, row16, tap16, c_wp16, c_plane16, c_blk16, c_kps, hi_a, c_planex16); break;
                  case 5: issue_taps<1, 2>(d_tmem, a_sub, b_lo, hi_sw, idesc, acc0, row16, tap16, c_wp16, c_plane16, c_blk16, c_kps, hi_a, c_planex16); break;
                  case 6: issue_taps<1, 4>(d_tmem, a_sub, b_lo, hi_sw, idesc, acc0, row16, tap16, c_wp16, c_plane16, c_blk16, c_kps, hi_a, c_planex16); break;
                  case 8: issue_taps<2, 1>(d_tmem, a_sub, b_lo, hi_sw, idesc, acc0, row16, tap16, c_wp16, c_plane16, c_blk16, c_kps, hi_a, c_planex16); break;
                  case 9: issue_taps<2, 2>(d_tmem, a_sub, b_lo, hi_sw, idesc, acc0, row16, tap16, c_wp16, c_plane16, c_blk16, c_kps, hi_a, c_planex16); break;
                  case 12: issue_taps<3, 4>(d_tmem, a_sub, b_lo, hi_sw, idesc, acc0, row16, tap16, c_wp16, c_plane16, c_blk16, c_kps, hi_a, c_planex16); break;
                  default: issue_taps<2, 4>(d_tmem, a_sub, b_lo, hi_sw, idesc, acc0, row16, tap16, c_wp16, c_plane16, c_blk16, c_kps, hi_a, c_planex16); break;
                }
              }
              umma_commit(&empty[slot]);
            }
            __syncwarp();
            if (tail_pending >= 0 && issue_tail(tail_pending, false)) tail_pending = -1;
            if (PROBE) t_issue += clock64() - t0;
            continue;
          }
          const uint32_t b_base = b_u32 + (p.b_resident ? ks : slot) * p.b_stage_bytes;
          const uint32_t a_lo0 = ((a_base >> 4) & 0x3FFFu) | (lbo_a16 << 16);
          const uint32_t b_lo0 = ((b_base >> 4) & 0x3FFFu) | (lbo_b16 << 16);
          for (int u = 0; u < p.nsub; ++u) {
            const uint32_t d_tmem = d_base + static_cast<uint32_t>(u * p.Ntile);
            uint32_t b_lo = b_lo0;
            uint32_t acc = ks > 0 ? 1u : 0u;
            for (int kh = 0; kh < 3; ++kh) {
#pragma unroll
              for (int kw = 0; kw < 3; ++kw) {
                // row of tap (kh,kw) for position j = 128u + i:  j + kh*(W+2) + kw - 1   (one row = one 16-byte unit)
                uint32_t a_lo = a_lo0 + static_cast<uint32_t>(128 * u + kh * p.Wp + kw - 1);
                for (int j = 0; j < kj; ++j) {
                  if (elect_one()) umma_f16(d_tmem, (static_cast<uint64_t>(desc_hi) << 32) | a_lo,
                           (static_cast<uint64_t>(desc_hi) << 32) | b_lo, p.idesc, acc);
                  acc = 1;
                  a_lo += 2 * lbo_a16;
                  b_lo += 2 * lbo_b16;
                }
              }
            }
          }
          __syncwarp();
          if (elect_one()) umma_commit(&empty[slot]);
        }
        if (elect_one()) umma_commit(&tfull[buf]);
        if (tail_pending >= 0) issue_tail(tail_pending, true);   // not delivered during this item's stages: queued behind its MMAs
        tail_pending = p.tail_n ? tcount : -1;
      }
      if (tail_pending >= 0) issue_tail(tail_pending, true);     // the last item's
      if (PROBE && p.dbg_clk && lane == 0 && warp == 1) {
        p.dbg_clk[blockIdx.x * 12 + 1] = t_bres;
        p.dbg_clk[blockIdx.x * 12 + 2] = t_tempty;
        p.dbg_clk[blockIdx.x * 12 + 3] = t_full;
        p.dbg_clk[blockIdx.x * 12 + 4] = t_issue;
        p.dbg_clk[blockIdx.x * 12 + 5] = clock64() - t_start;
        p.dbg_clk[blockIdx.x * 12 + 8] = t_fence;
        p.dbg_clk[blockIdx.x * 12 + 9] = t_commit;
        long long g_end;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g_end));
        p.dbg_clk[blockIdx.x * 12 + 10] = g_end - g_start;       // the MMA warp's lifetime in ns (mma_total is the same span in cycles)
      }
    }
  } else {
    // ======================================= epilogue ============================================
    // one specialised instantiation per (destination kind, activation, residual): see tma_epilogue_loop
    if (p.tail_n && p.upm) {
      tma_epilogue_loop_tail<PROBE, true>(p, tmem_base, tfull, tempty, tready, t2full, bias_s, warp, lane, total_work);
    } else if (p.tail_n) {
      tma_epilogue_loop_tail<PROBE, false>(p, tmem_base, tfull, tempty, tready, t2full, bias_s, warp, lane, total_work);
    } else {
    const int kind = p.transposed ? 2 : (p.split_n ? 1 : 0);
    const int nch_ = p.Ntile >> 4;
    const bool breg = p.n_tiles == 1 && nch_ <= TMA_EPI_GROUPS && TMA_EPI_GROUPS % nch_ == 0;
    const int sel = (breg ? 16 : 0) + kind * 4 + (p.act ? 2 : 0) + (p.res ? 1 : 0);
#define XR_EPI_CASE(id, K, A, R, B) \
  case id: tma_epilogue_loop<PROBE, K, A, R, B>(p, tmem_base, tfull, tempty, bias_s, nbuf, warp, lane, total_work); break;
    switch (sel) {
      XR_EPI_CASE(0, 0, false, false, false) XR_EPI_CASE(1, 0, false, true, false) XR_EPI_CASE(2, 0, true, false, false)
      XR_EPI_CASE(3, 0, true, true, false) XR_EPI_CASE(4, 1, false, false, false) XR_EPI_CASE(6, 1, true, false, false)
      XR_EPI_CASE(8, 2, false, false, false) XR_EPI_CASE(10, 2, true, false, false)
      XR_EPI_CASE(16, 0, false, false, true) XR_EPI_CASE(17, 0, false, true, true) XR_EPI_CASE(18, 0, true, false, true)
      XR_EPI_CASE(19, 0, true, true, true) XR_EPI_CASE(20, 1, false, false, true) XR_EPI_CASE(22, 1, true, false, true)
      XR_EPI_CASE(24, 2, false, false, true) XR_EPI_CASE(26, 2, true, false, true)
      default: asm volatile("trap;"); break;       // split / transposed launches never carry a residual (checked at plan time)
    }
#undef XR_EPI_CASE
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, static_cast<uint32_t>(p.tmem_cols));
  }
}

static inline void conv_tma_prepare_device() {
  XR_CUDA(cudaFuncSetAttribute(conv_halo_tma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, CONV_SMEM_MAX));
#ifdef XRSEG_DEBUG_API
  XR_CUDA(cudaFuncSetAttribute(conv_halo_tma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, CONV_SMEM_MAX));
#endif
}

static inline void launch_conv_halo_tma(const ConvParams& p_in, const TmapSet& maps, cudaStream_t stream) {
  ConvParams p = p_in;                        // values the kernel would otherwise compute and keep (or spill) per thread
  p.total_work = p.m_tiles * p.n_tiles;
  if (p.nbuf < 2) p.nbuf = 2;
  if (p.upm) p.grid &= ~1;                    // a CTA's items must share one row parity (its resident weights)
  XR_CHECK(!p.upm || (p.tail_n && p.grid >= 2), "a merged ConvTranspose launch needs the fused 1x1 tail and an even grid");
#ifdef XRSEG_DEBUG_API
  if (p.dbg_skip || p.dbg_clk) {   // probe instantiation: only reachable through xrseg_debug_conv
    launch_k(conv_halo_tma_kernel<true>, p.grid, TMA_THREADS, p.smem_bytes, stream, p, maps);
    return;
  }
#endif
  launch_k(conv_halo_tma_kernel<false>, p.grid, TMA_THREADS, p.smem_bytes, stream, p, maps);
}
static inline void launch_conv_halo_tma(const ConvParams& p, const CUtensorMap& map, cudaStream_t stream) {
  TmapSet t{};
  t.m[0] = map;
  launch_conv_halo_tma(p, t, stream);
}
#endif  // __CUDACC__

// ---- host emulation of this kernel's data movement (fp32; test infrastructure only) -------------------------------
static inline void emulate_conv_halo_tma(const ConvParams& p, const float* in, const float* wpack_f, const float* bias,
                                         const float* res, float* out) {
  const int bchunks = p.b_stage_bytes / (p.Ntile * 16);
  const int lbo_slots = p.lbo_a / 16;
  const int pre = 8;  // rows readable before the stage buffer (the kernel reads row -1 for invalid positions)
  std::vector<float> a((static_cast<size_t>(p.cps) * lbo_slots + 2 * 128 + pre) * 8);
  std::vector<float> acc(static_cast<size_t>(p.nsub) * 128 * p.Ntile);
  for (int w = 0; w < p.m_tiles * p.n_tiles; ++w) {
    const int tile = w / p.n_tiles, n_tile = w % p.n_tiles;
    const int b = tile / p.tpi;
    const int y0 = (tile % p.tpi) * p.R;
    std::fill(acc.begin(), acc.end(), 0.f);
    for (int ks = 0; ks < p.nks; ++ks) {
      std::fill(a.begin(), a.end(), 0.f);
      for (int c = 0; c < p.cps; ++c)          // one TMA box per chunk: coords (ks*cb + 8c, -1, y0-1, b)
        for (int by = 0; by < p.hbox; ++by)
          for (int bx = 0; bx < p.Wp; ++bx) {
            const int y = y0 - 1 + by, x = -1 + bx;
            if (y < 0 || y >= p.H || x < 0 || x >= p.W) continue;   // OOB -> zero fill
            const size_t pixi = (static_cast<size_t>(b) * p.H + y) * p.W + x;
            for (int e = 0; e < 8; ++e)
              a[(pre + static_cast<size_t>(c) * lbo_slots + by * p.Wp + bx) * 8 + e] =
                  in[pixi * p.in_pitch + ks * p.cb + c * 8 + e];
          }
      const float* bst = wpack_f + (p.sw ? (static_cast<size_t>(n_tile) * p.nks + ks) * (p.b_stage_bytes / 2)
                                         : (static_cast<size_t>(n_tile) * p.nks + ks) * bchunks * p.Ntile * 8);
      for (int u = 0; u < p.nsub; ++u)
        for (int t = 0; t < 9; ++t) {
          const int shift = 128 * u + (t / 3) * p.Wp + (t % 3) - 1;
          for (int j = 0; j < p.cb / 16; ++j)
            for (int hk = 0; hk < 2; ++hk) {
              const int ac = 2 * j + hk, bc = t * p.cps + 2 * j + hk;
              for (int i = 0; i < 128; ++i)
                for (int n = 0; n < p.Ntile; ++n) {
                  float sacc = 0.f;
                  for (int e = 0; e < 8; ++e) {
                    const float bv = p.sw ? bst[sw_phys((static_cast<size_t>(t) * p.Ntile + n) * (p.cb * 2) + (ac * 8 + e) * 2, p.sw) / 2]
                                          : bst[(static_cast<size_t>(bc) * p.Ntile + n) * 8 + e];
                    sacc += a[(pre + static_cast<size_t>(ac) * lbo_slots + i + shift) * 8 + e] * bv;
                  }
                  acc[(static_cast<size_t>(u) * 128 + i) * p.Ntile + n] += sacc;
                }
            }
        }
    }
    for (int u = 0; u < p.nsub; ++u)
      for (int i = 0; i < 128; ++i) {
        const int j = 128 * u + i;
        const int yy = j / p.Wp, cc = j % p.Wp, y = y0 + yy;
        if (!(yy < p.R && y < p.H && cc >= 1 && cc <= p.W)) continue;
        const size_t pix = (static_cast<size_t>(b) * p.H + y) * p.W + (cc - 1);
        for (int n = 0; n < p.Ntile; ++n) {
          const int ng = n_tile * p.Ntile + n;
          float yv = acc[(static_cast<size_t>(u) * 128 + i) * p.Ntile + n] + bias[ng];
          if (p.act) yv = yv / (1.0f + expf(-yv));
          if (res) yv += res[pix * p.res_pitch + ng];
          out[pix * p.out_pitch + ng] = yv;
        }
      }
  }
}

// ---- host emulation of the flat (1x1) mode ---------------------------------------------------------------------------
static inline void emulate_conv_flat_tma(const ConvParams& p, const float* in, const float* wpack_f, const float* bias,
                                         const float* res, float* out) {
  const int rb = p.cb * 2;
  std::vector<float> a(static_cast<size_t>(p.slots) * p.cb);
  std::vector<float> acc(static_cast<size_t>(p.slots) * p.Ntile);
  for (int w = 0; w < p.m_tiles * p.n_tiles; ++w) {
    const int tile = w / p.n_tiles, n_tile = w % p.n_tiles;
    std::fill(acc.begin(), acc.end(), 0.f);
    const int nkb = p.nks * (p.kps > 1 ? p.kps : 1);
    for (int ks = 0; ks < nkb; ++ks) {
      std::fill(a.begin(), a.end(), 0.f);
      for (int r = 0; r < p.slots; ++r) {            // TMA boxes: rows past flat_rows and channels past Cin are zero
        const long m = static_cast<long>(tile) * p.slots + r;
        if (m >= p.flat_rows) continue;
        for (int c = 0; c < p.cb; ++c) {
          const int ci = ks * p.cb + c;
          if (ci < p.Cin) a[static_cast<size_t>(r) * p.cb + c] = in[static_cast<size_t>(m) * p.in_pitch + ci];
        }
      }
      const float* bst = wpack_f + (static_cast<size_t>(n_tile) * nkb + ks) * (static_cast<size_t>(p.Ntile) * p.cb);
      for (int r = 0; r < p.slots; ++r)
        for (int n = 0; n < p.Ntile; ++n) {
          float sacc = 0.f;
          for (int c = 0; c < p.cb; ++c)
            sacc += a[static_cast<size_t>(r) * p.cb + c] * bst[sw_phys(static_cast<size_t>(n) * rb + c * 2, p.sw) / 2];
          acc[static_cast<size_t>(r) * p.Ntile + n] += sacc;
        }
    }
    for (int r = 0; r < p.slots; ++r) {
      const long m = static_cast<long>(tile) * p.slots + r;
      if (m >= p.flat_rows) continue;
      for (int n = 0; n < p.Ntile; ++n) {
        const int ng = n_tile * p.Ntile + n;
        float yv = acc[static_cast<size_t>(r) * p.Ntile + n] + bias[ng];
        if (p.act) yv = yv / (1.0f + expf(-yv));
        if (p.transposed) {
          const int pos = ng / p.Cout, co = ng % p.Cout;
          const long tb = m / (p.H * p.W), rem = m % (p.H * p.W), th = rem / p.W, tw = rem % p.W;
          const size_t opix = (static_cast<size_t>(tb) * p.Ho + (2 * th + (pos >> 1))) * p.Wo + (2 * tw + (pos & 1));
          out[opix * p.out_pitch + co] = yv;
          continue;
        }
        if (res) yv += res[static_cast<size_t>(m) * p.res_pitch + ng];
        out[static_cast<size_t>(m) * p.out_pitch + ng] = yv;
      }
    }
  }
}

// ---- host emulation of the stride-2 parity-plane mode ----------------------------------------------------------------
// `in` is the NHWC input [B, 2*p.H, 2*p.W, in_pitch]; follows the kernel literally: four plane boxes per K-block, taps as
// row shifts, epilogue on position-linear indices.  Valid outputs must never read outside their plane buffer.
static inline bool emulate_conv_s2_tma(const ConvParams& p, const float* in, const float* wpack_f, const float* bias,
                                       const float* res, float* out) {
  const int H = 2 * p.H, W = 2 * p.W, rb = p.cb * 2;
  const int plane_rows = p.slots;
  std::vector<float> a(static_cast<size_t>(4) * plane_rows * p.cb);
  std::vector<float> acc(static_cast<size_t>(p.nsub) * 128 * p.Ntile);
  for (int w = 0; w < p.m_tiles * p.n_tiles; ++w) {
    const int tile = w / p.n_tiles, n_tile = w % p.n_tiles;
    const int b = tile / p.tpi, y0 = (tile % p.tpi) * p.R;
    std::fill(acc.begin(), acc.end(), 0.f);
    for (int ks = 0; ks < p.nks; ++ks) {
      std::fill(a.begin(), a.end(), 0.f);
      for (int pl = 0; pl < 4; ++pl) {
        const int py = pl >> 1, px = pl & 1;
        for (int by = 0; by < p.hbox; ++by)
          for (int bx = 0; bx < p.Wp; ++bx) {
            const int ys = y0 - py + by, xs = -1 + bx;
            if (ys < 0 || ys >= H / 2 || xs < 0 || xs >= W / 2) continue;     // OOB -> zero fill
            const size_t pix = (static_cast<size_t>(b) * H + 2 * ys + py) * W + 2 * xs + px;
            for (int c = 0; c < p.cb; ++c)
              a[(static_cast<size_t>(pl) * plane_rows + by * p.Wp + bx) * p.cb + c] = in[pix * p.in_pitch + ks * p.cb + c];
          }
      }
      const float* bst = wpack_f + (static_cast<size_t>(n_tile) * p.nks + ks) * (p.b_stage_bytes / 2);
      for (int j = 0; j < p.nsub * 128; ++j) {
        const int yy = j / p.Wp, cc = j % p.Wp;
        const bool valid = yy < p.R && y0 + yy < p.H && cc >= 1;
        if (!valid) continue;
        for (int t = 0; t < 9; ++t) {
          const int kh = t / 3, kw = t % 3;
          const int pl = (kh != 1 ? 2 : 0) + (kw != 1 ? 1 : 0);
          const int row = j + (kh == 2 ? p.Wp : 0) - (kw == 0 ? 1 : 0);
          if (row < 0 || row >= plane_rows) return false;                     // a valid output left its plane buffer
          for (int n = 0; n < p.Ntile; ++n) {
            float sacc = 0.f;
            for (int c = 0; c < p.cb; ++c)
              sacc += a[(static_cast<size_t>(pl) * plane_rows + row) * p.cb + c] *
                      bst[sw_phys((static_cast<size_t>(t) * p.Ntile + n) * rb + c * 2, p.sw) / 2];
            acc[static_cast<size_t>(j) * p.Ntile + n] += sacc;
          }
        }
      }
    }
    for (int j = 0; j < p.nsub * 128; ++j) {
      const int yy = j / p.Wp, cc = j % p.Wp, y = y0 + yy;
      if (!(yy < p.R && y < p.H && cc >= 1 && cc <= p.W)) continue;
      const size_t pix = (static_cast<size_t>(b) * p.H + y) * p.W + (cc - 1);
      for (int n = 0; n < p.Ntile; ++n) {
        const int ng = n_tile * p.Ntile + n;
        float yv = acc[static_cast<size_t>(j) * p.Ntile + n] + bias[ng];
        if (p.act) yv = yv / (1.0f + expf(-yv));
        if (res) yv += res[pix * p.res_pitch + ng];
        out[pix * p.out_pitch + ng] = yv;
      }
    }
  }
  return true;
}

}  // namespace xrseg
