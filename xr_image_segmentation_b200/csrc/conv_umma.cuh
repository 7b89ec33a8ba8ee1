// conv_umma.cuh -- implicit-GEMM convolution on the 5th-gen tensor cores (tcgen05.mma, accumulators in TMEM).
//
// Replaces the `Conv` / `ConvTranspose` (+ `Swish`, + residual `Add`) layers that the reference executes through
// Worker.ScheduleIterable / MoveNext (Assets/Scripts/InferenceEngine/IEExecutor.cs:371,397); layer list in
// SURVEY.md Appendix A/B.
//
// GEMM view:  D[M = output positions, N = Cout] = A[M, K] * W[N, K]^T,  K = taps * Cin, fp16 operands, fp32 accum.
// Activations are NHWC fp16 (channel counts padded to multiples of 16), so a K-chunk of 8 channels is one 16-byte
// vector.  Both operands sit in shared memory in the K-major SWIZZLE_NONE canonical layout:
//       element (row r, K-chunk c)  ->  base + c * LBO + r * 16 bytes            (SBO = 128 B: rows are uniform)
// Because rows are uniformly 16 B apart, a descriptor may START at any row.  Two A-operand modes use this:
//   MODE_GATHER  every (row, K-chunk) is fetched by an im2col address computation (any kernel / stride / ConvT).
//   MODE_HALO    3x3 stride-1: the input halo of the tile is loaded ONCE in "padded-linear" pixel order
//                (index = (b*(H+1) + y) * (W+2) + x + 1, one shared zero row between images, zero columns left
//                and right) and the nine taps are nine MMAs whose A descriptors start kh*(W+2)+kw rows further --
//                no 9x im2col re-read.  Output rows that fall on padding positions are computed and discarded.
//
// Warp roles (288 threads): warps 0-3 producers (cp.async 16 B, zero-fill for padding), warps 4-7 epilogue
// (tcgen05.ld -> +bias -> SiLU -> +residual -> fp16 NHWC store into the channel slice of the destination, which is
// how Concat/Split cost nothing), warp 8 TMEM allocator + single-thread MMA issuer.  CTAs are persistent over
// (M-tile, N-tile) work items; the accumulator is double-buffered in TMEM so the epilogue of tile i overlaps the
// main loop of tile i+1.  Weights are pre-packed on the host into the exact shared-memory image.
#pragma once

#include <vector>

#include "common.cuh"

namespace xrseg {

enum { MODE_GATHER = 0, MODE_HALO = 1 };
enum {
  CONV_HDR_BYTES = 2304, CONV_SMEM_MAX = 232448, CONV_MAX_STAGES = 8,
  CONV_NPROD = 256,                      // producer threads (warps 0-7)
  CONV_NEPI = 256,                       // epilogue threads (warps 8-15)
  CONV_MMA_WARP = 16,                    // TMEM allocator + MMA issuer
  CONV_THREADS = CONV_NPROD + CONV_NEPI + 32
};

// Division by a runtime-constant divisor (n < 2^31): q = (umulhi(n, mul) + n) >> shr.
struct FastDiv {
  uint32_t mul, shr;
  int d;
};
static inline FastDiv make_fastdiv(int d) {
  FastDiv f;
  f.d = d < 1 ? 1 : d;
  uint32_t L = 0;
  while ((1u << L) < static_cast<uint32_t>(f.d)) ++L;
  f.shr = L;
  f.mul = static_cast<uint32_t>(((static_cast<uint64_t>(1) << 32) * ((static_cast<uint64_t>(1) << L) - f.d)) / f.d + 1);
  return f;
}
__host__ __device__ __forceinline__ int fd_div(const FastDiv& f, int n) {
#ifdef __CUDA_ARCH__
  return static_cast<int>((__umulhi(static_cast<uint32_t>(n), f.mul) + static_cast<uint32_t>(n)) >> f.shr);
#else
  return static_cast<int>(((static_cast<uint64_t>(static_cast<uint32_t>(n)) * f.mul >> 32) + static_cast<uint32_t>(n)) >> f.shr);
#endif
}

// profiling switches of the probe builds (libxrseg_debug.so); constant false in the product library
#ifdef XRSEG_DEBUG_API
#define XR_DBG_SKIP(p, bit) (((p).dbg_skip & (bit)) != 0)
#else
#define XR_DBG_SKIP(p, bit) false
#endif

struct ConvParams {
  const __half* in;
  __half* out;
  const __half* res;
  const __half* wpack;
  const float* bias;
  int B, H, W, Cin, in_pitch;       // Cin: padded channel count of the input view (multiple of 16)
  int Ho, Wo, Cout, out_pitch;      // Cout: padded output channels (per position when transposed)
  int res_pitch;
  int k, stride, pad, act, transposed;
  int mode, Wp, Hp1, M_total;
  int m_tiles, n_tiles, Ntile;
  int K_total, nks, cps, taps, cb;  // cps: A chunks per stage; taps: MMA tap loop count (9 in halo mode, else 1)
  int slots, lbo_a, a_stage_bytes, b_stage_bytes, b_resident;
  int S, lag;
  uint32_t idesc;
  int tmem_cols;
  int smem_off_b, smem_off_a, smem_bytes;
  int grid;
  FastDiv fd_wp, fd_hp1, fd_hw, fd_wo, fd_cin, fd_cout;
  int R, nsub, tpi, hbox;           // MODE_HALO_TMA (conv_tma.cuh): rows per tile, sub-tiles, tiles per image, box rows
  long long* dbg_clk;               // optional [grid][8] cycle counters per role phase (debug builds of the probe)
  int dbg_skip;                     // profiling experiment: 1 skip MMA issue, 2 skip epilogue math+stores, 4 skip loads
  int sw;                           // operand swizzle: 0 none, 1/2/3 = 32/64/128-byte (row = 16/32/64 channels)
  int flat_rows;                    // MODE_FLAT_TMA: B*H*W rows of the activation matrix
  int kps;                          // MODE_FLAT_TMA: K-blocks (of cb channels) per pipeline stage; 0 / 1 elsewhere
  int nbuf;                         // TMA kernel: TMEM accumulator sets in flight (0 = 2)
  int total_work;                   // TMA kernel: m_tiles * n_tiles, filled in by launch_conv_halo_tma (a kernel-parameter read instead of a
                                    // computed value the register allocator spills: the reload sat on the item loop's back edge)
  int pair;                         // s2 TMA mode: operand rows hold a PIXEL PAIR (2 cb channels, conv_tma.cuh plan_conv_s2_tma_impl)
  // Sibling fusion (TMA kernel): two convolutions that read the same input run as ONE GEMM with N = Cout_a + Cout_b;
  // output columns >= split_n go to out2 (pixel pitch out2_pitch), relative to split_n.  split_n == 0: single output.
  __half* out2;
  int split_n, out2_pitch;
  // Fused trailing 1x1 convolution (conv_tma.cuh "tail"): the 64-channel output of a 3x3 layer never leaves the SM -- the epilogue
  // writes it back into tensor memory as packed fp16, a second set of MMAs (A from TMEM, W2 from shared memory) produces the
  // tail_n = 32 output channels of the 1x1 layer in the freed accumulator columns, a second epilogue pass stores those.
  // `out` / `out_pitch` are then the TAIL's destination.  tail_n == 0: off.
  int tail_n, tail_act, smem_off_w2;
  const __half* tail_w;             // [32][64] fp16, K-major 128-byte swizzle (pack_conv_weights_sw image of the 1x1 layer)
  const float* tail_bias;           // [32]
  // ConvTranspose 2x2 / stride 2 merged into this 3x3 (conv_tma.cuh plan_conv_upmerge_tma): H / W are the map BEFORE the
  // upsampling, Ho / Wo = 2H / 2W.  Virtual sub-tile v = 2 u + dx (u = 128-row sub-tile, dx = output column parity); the row
  // parity dy of an item is w & 1.  The bias holds [Cout] interior values and nine [Cout] border corrections at smem_off_corr.
  int upm, smem_off_corr;
};

struct ConvDesc {
  int B, H, W, Cin, in_pitch;
  int Cout, out_pitch;
  int k, stride, act, transposed;
  int res_pitch;                    // 0 = no residual
  int upm;                          // 1: a 2x2 / stride-2 ConvTranspose of this input runs inside the 3x3 (ConvParams::upm)
};

// ---------------------------------------------------------------------------------------------------------------
// index math shared by the device loaders, the epilogue and the host emulator
// ---------------------------------------------------------------------------------------------------------------
struct PixRef {
  int valid;
  long pix;  // pixel index into the NHWC tensor (multiply by pitch for the element offset)
};

// MODE_HALO: biased padded-linear index Lb = L + Hp1*Wp (always >= 0) -> input pixel.
__host__ __device__ inline PixRef halo_pixel(const ConvParams& p, long Lb) {
  long G = Lb / p.Wp;
  int cc = static_cast<int>(Lb - G * p.Wp);
  long b1 = G / p.Hp1;
  int r = static_cast<int>(G - b1 * p.Hp1);
  PixRef o;
  o.valid = (b1 >= 1 && b1 <= p.B && r < p.H && cc >= 1 && cc <= p.W) ? 1 : 0;
  o.pix = ((b1 - 1) * p.H + r) * static_cast<long>(p.W) + (cc - 1);
  return o;
}

// MODE_GATHER: output position m and K element index -> input pixel and channel.
__host__ __device__ inline PixRef gather_pixel(const ConvParams& p, long m, int kelem, int* c0) {
  PixRef o;
  o.valid = 0;
  o.pix = 0;
  *c0 = 0;
  if (m >= p.M_total || kelem >= p.K_total) return o;
  int tap = kelem / p.Cin;
  *c0 = kelem - tap * p.Cin;
  int kk = p.transposed ? 1 : p.k;
  int kh = tap / kk, kw = tap - kh * kk;
  int hw = p.transposed ? p.H * p.W : p.Ho * p.Wo;
  long b = m / hw;
  int rem = static_cast<int>(m - b * hw);
  int wo = p.transposed ? p.W : p.Wo;
  int oh = rem / wo, ow = rem - oh * wo;
  int st = p.transposed ? 1 : p.stride;
  int pad = p.transposed ? 0 : p.pad;
  int ih = oh * st - pad + kh, iw = ow * st - pad + kw;
  if (ih < 0 || ih >= p.H || iw < 0 || iw >= p.W) return o;
  o.valid = 1;
  o.pix = (b * p.H + ih) * static_cast<long>(p.W) + iw;
  return o;
}

// Output position m (+ column n of the GEMM) -> output pixel, channel.
__host__ __device__ inline PixRef out_pixel(const ConvParams& p, long m, int n, int* co) {
  PixRef o;
  o.valid = 0;
  o.pix = 0;
  *co = n;
  if (m >= p.M_total) return o;
  if (p.mode == MODE_HALO) {
    long G = m / p.Wp;
    int cc = static_cast<int>(m - G * p.Wp);
    long b = G / p.Hp1;
    int r = static_cast<int>(G - b * p.Hp1);
    if (r >= p.H || cc < 1 || cc > p.W) return o;
    o.valid = 1;
    o.pix = (b * p.H + r) * static_cast<long>(p.W) + (cc - 1);
    return o;
  }
  if (p.transposed) {
    int pos = n / p.Cout;
    *co = n - pos * p.Cout;
    int hw = p.H * p.W;
    long b = m / hw;
    int rem = static_cast<int>(m - b * hw);
    int h = rem / p.W, w = rem - h * p.W;
    o.valid = 1;
    o.pix = (b * p.Ho + (2 * h + (pos >> 1))) * static_cast<long>(p.Wo) + (2 * w + (pos & 1));
    return o;
  }
  o.valid = 1;
  o.pix = m;
  return o;
}

// ---------------------------------------------------------------------------------------------------------------
// planning (host)
// ---------------------------------------------------------------------------------------------------------------
#define XR_CUDA_CHECK_PLAN(p)                                                                          \
  XR_CHECK((p).cps == 2 || (p).cps == 4 || (p).cps == 8, "chunks per stage must be a power of two (%d)", (p).cps); \
  XR_CHECK(static_cast<long>((p).M_total) + static_cast<long>((p).Hp1) * (p).Wp + 256 < (1L << 31), "M too large")

static inline int pow2_ceil(int v) {
  int r = 32;
  while (r < v) r <<= 1;
  return r;
}

// variant: 0 / 2 = thread-loaded halo for 3x3 s1, 1 = force MODE_GATHER (cross-check path)
static inline ConvParams plan_conv(const ConvDesc& d, int num_sms, int variant = 0) {
  ConvParams p{};
  XR_CHECK(d.Cin % 16 == 0 && d.Cout % 16 == 0, "channels must be padded to 16 (cin %d cout %d)", d.Cin, d.Cout);
  p.B = d.B; p.H = d.H; p.W = d.W; p.Cin = d.Cin; p.in_pitch = d.in_pitch;
  p.Cout = d.Cout; p.out_pitch = d.out_pitch; p.res_pitch = d.res_pitch;
  p.k = d.k; p.stride = d.stride; p.pad = d.k / 2; p.act = d.act; p.transposed = d.transposed;
  if (d.transposed) {
    XR_CHECK(d.k == 2 && d.stride == 2, "only 2x2 stride-2 ConvTranspose is on the path");
    p.Ho = d.H * 2; p.Wo = d.W * 2; p.pad = 0;
  } else {
    p.Ho = (d.H + 2 * p.pad - d.k) / d.stride + 1;
    p.Wo = (d.W + 2 * p.pad - d.k) / d.stride + 1;
  }
  const int ncols = d.transposed ? 4 * d.Cout : d.Cout;
  p.Ntile = ncols <= 256 ? ncols : 256;
  XR_CHECK(ncols % p.Ntile == 0, "N %d not tileable", ncols);
  p.n_tiles = ncols / p.Ntile;
  p.idesc = umma_idesc_f16(p.Ntile, 0);
  p.tmem_cols = pow2_ceil(2 * p.Ntile);
  const bool halo = (d.k == 3 && d.stride == 1 && !d.transposed && variant != 1);
  p.mode = halo ? MODE_HALO : MODE_GATHER;
  const int budget = CONV_SMEM_MAX - CONV_HDR_BYTES;
  if (halo) {
    p.Wp = d.W + 2; p.Hp1 = d.H + 1;
    long mt = static_cast<long>(d.B) * p.Hp1 * p.Wp;
    XR_CHECK(mt < (1L << 31), "M too large");
    p.M_total = static_cast<int>(mt);
    p.slots = 130 + 2 * p.Wp;
    p.lbo_a = (p.slots | 1) * 16;
    p.taps = 9;
    p.K_total = 9 * d.Cin;
    int cb = 64;
    while (cb > 16 && (d.Cin % cb != 0 || p.lbo_a * (cb / 8) > 40960)) cb >>= 1;
    const long total_b = 9L * d.Cin * p.Ntile * 2;
    p.b_resident = (p.n_tiles == 1 && total_b <= 98304) ? 1 : 0;
    if (!p.b_resident)
      while (cb > 16 && 9 * cb * p.Ntile * 2 > 40960) cb >>= 1;
    p.cb = cb;
    p.cps = cb / 8;
    p.nks = d.Cin / cb;
    p.a_stage_bytes = p.lbo_a * p.cps;
    p.b_stage_bytes = 9 * cb * p.Ntile * 2;
  } else {
    long mt = d.transposed ? static_cast<long>(d.B) * d.H * d.W : static_cast<long>(d.B) * p.Ho * p.Wo;
    XR_CHECK(mt < (1L << 31), "M too large");
    p.M_total = static_cast<int>(mt);
    p.slots = 128;
    p.lbo_a = 129 * 16;
    p.taps = 1;
    p.K_total = (d.transposed ? 1 : d.k * d.k) * d.Cin;
    p.cb = 64;
    p.cps = 8;
    p.nks = ceil_div(p.K_total, 64);
    p.a_stage_bytes = p.lbo_a * 8;
    p.b_stage_bytes = 8 * p.Ntile * 16;
    const long total_b = static_cast<long>(p.nks) * p.b_stage_bytes;
    p.b_resident = (p.n_tiles == 1 && total_b <= 98304) ? 1 : 0;
  }
  p.m_tiles = ceil_div(p.M_total, 128);
  XR_CHECK(static_cast<long>(d.B) * d.H * d.W * d.in_pitch < (1L << 31), "input tensor too large for 32-bit gather offsets");
  const int resident_bytes = p.b_resident ? p.nks * p.b_stage_bytes : 0;
  const int per_stage = p.a_stage_bytes + (p.b_resident ? 0 : p.b_stage_bytes);
  int S = (budget - resident_bytes) / per_stage;
  if (S > CONV_MAX_STAGES) S = CONV_MAX_STAGES;
  XR_CHECK(S >= 2, "conv does not fit shared memory (a %d b %d resident %d)", p.a_stage_bytes, p.b_stage_bytes,
           resident_bytes);
  p.S = S;
  p.lag = 0;
  p.smem_off_b = CONV_HDR_BYTES;
  const int b_region = p.b_resident ? resident_bytes : S * p.b_stage_bytes;
  p.smem_off_a = CONV_HDR_BYTES + round_up(b_region, 128);
  p.smem_bytes = p.smem_off_a + S * p.a_stage_bytes;
  XR_CHECK(p.smem_bytes <= CONV_SMEM_MAX, "smem plan overflow %d", p.smem_bytes);
  const int work = p.m_tiles * p.n_tiles;
  const int occ = 1;   // 544 threads and >= 100 registers per thread: one CTA per SM
  p.grid = work < num_sms * occ ? work : num_sms * occ;
  p.fd_wp = make_fastdiv(p.Wp);
  p.fd_hp1 = make_fastdiv(p.Hp1);
  p.fd_hw = make_fastdiv(d.transposed ? d.H * d.W : p.Ho * p.Wo);
  p.fd_wo = make_fastdiv(d.transposed ? d.W : p.Wo);
  p.fd_cin = make_fastdiv(d.Cin);
  p.fd_cout = make_fastdiv(d.Cout);
  XR_CUDA_CHECK_PLAN(p);
  return p;
}

// Number of halves in the packed weight image.
static inline size_t conv_wpack_elems(const ConvParams& p) {
  return static_cast<size_t>(p.n_tiles) * p.nks * p.b_stage_bytes / 2;
}

// K element consumed at (stage ks, B-chunk bc, element e) -> (tap, input channel); returns false for K padding.
static inline bool conv_k_index(const ConvParams& p, int ks, int bc, int e, int* tap, int* ci) {
  if (p.mode != MODE_GATHER) {
    *tap = bc / p.cps;
    *ci = ks * p.cb + (bc % p.cps) * 8 + e;
    return true;
  }
  int kelem = (ks * 8 + bc) * 8 + e;
  if (kelem >= p.K_total) return false;
  *tap = kelem / p.Cin;
  *ci = kelem % p.Cin;
  return true;
}

// Pack fp32 weights ([cout,cin,k,k], or [cin,cout,2,2] when transposed) into the smem image
// [n_tile][stage][B-chunk][n][8] (fp16) and the bias into fp32 [n_tiles * Ntile].
template <typename HalfT>
static inline void pack_conv_weights(const ConvParams& p, const float* w, const float* bias, int cin_real, int cout_real,
                                     std::vector<HalfT>& wp, std::vector<float>& bp) {
  const int bchunks = p.b_stage_bytes / (p.Ntile * 16);
  wp.assign(conv_wpack_elems(p), HalfT(0.0f));
  bp.assign(static_cast<size_t>(p.n_tiles) * p.Ntile, 0.0f);
  const int kk = p.transposed ? 2 : p.k;
  for (int nt = 0; nt < p.n_tiles; ++nt)
    for (int ks = 0; ks < p.nks; ++ks)
      for (int bc = 0; bc < bchunks; ++bc)
        for (int n = 0; n < p.Ntile; ++n)
          for (int e = 0; e < 8; ++e) {
            int tap, ci;
            if (!conv_k_index(p, ks, bc, e, &tap, &ci)) continue;
            if (ci >= cin_real) continue;
            const int ng = nt * p.Ntile + n;
            float v;
            if (p.transposed) {
              const int pos = ng / p.Cout, co = ng % p.Cout;
              if (co >= cout_real) continue;
              v = w[((static_cast<size_t>(ci) * cout_real + co) * 2 + (pos >> 1)) * 2 + (pos & 1)];
            } else {
              if (ng >= cout_real) continue;
              const int kh = tap / kk, kw = tap % kk;
              v = w[((static_cast<size_t>(ng) * cin_real + ci) * kk + kh) * kk + kw];
            }
            const size_t idx = ((static_cast<size_t>(nt) * p.nks + ks) * bchunks + bc) * p.Ntile * 8 +
                               static_cast<size_t>(n) * 8 + e;
            wp[idx] = HalfT(v);
          }
  for (int ng = 0; ng < p.n_tiles * p.Ntile; ++ng) {
    const int co = p.transposed ? ng % p.Cout : ng;
    if (co < cout_real && bias) bp[ng] = bias[co];
  }
}

#ifdef __CUDACC__
// ---------------------------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------------------------
// cp.async completion -> mbarrier: the arrive fires when all prior cp.async of this thread have landed and counts as
// one of the barrier's expected arrivals (.noinc), so a producer thread never blocks on its own copies.
__device__ __forceinline__ void cp_async_arrive_noinc(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__global__ void __launch_bounds__(CONV_THREADS, 1) conv_umma_kernel(const __grid_constant__ ConvParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem);       // [8]
  uint64_t* empty = full + 8;                               // [8]
  uint64_t* tfull = empty + 8;                              // [2]
  uint64_t* tempty = tfull + 2;                             // [2]
  uint64_t* bres = tempty + 2;                              // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bres + 1);
  float* bias_s = reinterpret_cast<float*>(smem + 256);     // [<=512]
  uint8_t* smem_b = smem + p.smem_off_b;
  uint8_t* smem_a = smem + p.smem_off_a;

  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // provably warp-uniform: role code uses the uniform datapath
  const int lane = tid & 31;
  const int total_work = p.m_tiles * p.n_tiles;

  if (tid == 0) {
    for (int i = 0; i < CONV_MAX_STAGES; ++i) {
      mbar_init(&full[i], CONV_NPROD);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], CONV_NEPI);
    }
    mbar_init(bres, CONV_NPROD);
    mbar_fence_init();
  }
  if (warp == CONV_MMA_WARP) {
    tmem_alloc(tmem_slot, static_cast<uint32_t>(p.tmem_cols));
    tmem_relinquish();
  }
  for (int i = tid; i < p.n_tiles * p.Ntile; i += CONV_THREADS) bias_s[i] = p.bias[i];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // Only now may the next kernel's CTAs start (PDL): a dependent CTA that became co-resident and grabbed TMEM columns
  // before this CTA had its own would wait for this kernel to finish while this CTA waits for its columns -- deadlock.
  pdl_launch_dependents();

  if (warp < CONV_NPROD / 32) {
    // ======================================= producers ===========================================
    const uint32_t a_u32 = smem_u32(smem_a);
    const uint32_t b_u32 = smem_u32(smem_b);
    if (p.b_resident) {
      const int bytes = p.nks * p.b_stage_bytes;
      const uint8_t* src = reinterpret_cast<const uint8_t*>(p.wpack);
      for (int i = tid * 16; i < bytes; i += CONV_NPROD * 16) cp_async16(b_u32 + i, src + i, 16);
      cp_async_arrive_noinc(bres);
    }
    pdl_wait();   // weights / bias are constants (loaded above); activations are the previous kernels' output
    int it = 0;
    for (int w = blockIdx.x; w < total_work; w += gridDim.x) {
      const int m_tile = p.n_tiles == 1 ? w : (w >> 1);
      const int n_tile = p.n_tiles == 1 ? 0 : (w & 1);
      const int m0 = m_tile * 128;

      // per-tile row bookkeeping for the general MODE_GATHER path (4 rows per thread: r0 + 32 j)
      const int gc = tid & 7;
      const int r0 = tid >> 3;
      int g_pre[4], g_ih[4], g_iw[4];
      const bool fast1x1 = (p.mode == MODE_GATHER && p.k == 1 && p.stride == 1) || p.transposed;
      // K walk of this thread's chunk column (general gather): K element gc*8 + 64*ks -> (kh, kw, channel c0), advanced
      // incrementally per stage -- no division in the stage loop.  All offsets are 32-bit element offsets (plan checks).
      int w_c0 = gc * 8, w_kh = 0, w_kw = 0;
      if (p.mode == MODE_GATHER && !fast1x1) {
        while (w_c0 >= p.Cin) {
          w_c0 -= p.Cin;
          if (++w_kw == p.k) { w_kw = 0; ++w_kh; }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int m = m0 + r0 + 32 * j;
          const int b = fd_div(p.fd_hw, m);
          const int rem = m - b * p.fd_hw.d;
          const int oh = fd_div(p.fd_wo, rem), ow = rem - oh * p.fd_wo.d;
          g_ih[j] = m < p.M_total ? oh * p.stride - p.pad : -0x40000000;   // invalid rows fail the bounds test below
          g_iw[j] = ow * p.stride - p.pad;
          g_pre[j] = ((b * p.H + oh * p.stride - p.pad) * p.W + g_iw[j]) * p.in_pitch;   // element offset of tap (0,0)
        }
      }

      for (int ks = 0; ks < p.nks; ++ks, ++it) {
        const int slot = it % p.S;
        if (it >= p.S) mbar_wait(&empty[slot], static_cast<uint32_t>((it / p.S) - 1) & 1u);
        const uint32_t a_dst = a_u32 + slot * p.a_stage_bytes;

        if (p.mode == MODE_GATHER) {
          const int kelem = (ks * 8 + gc) * 8;
          if (kelem < p.K_total && !XR_DBG_SKIP(p, 4)) {
            if (fast1x1) {
              // A is the activation matrix itself: row m, channels kelem..kelem+7
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const int row = r0 + 32 * j;
                const int m = m0 + row;
                const bool ok = m < p.M_total;
                const __half* src = ok ? p.in + static_cast<size_t>(m) * p.in_pitch + kelem : p.in;
                cp_async16_ca(a_dst + gc * p.lbo_a + row * 16, src, ok ? 16u : 0u);
              }
            } else {
              const uint32_t dst0 = a_dst + gc * p.lbo_a + r0 * 16;
              const int tap_off = (w_kh * p.W + w_kw) * p.in_pitch + w_c0;
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const bool ok = static_cast<unsigned>(g_ih[j] + w_kh) < static_cast<unsigned>(p.H) &&
                                static_cast<unsigned>(g_iw[j] + w_kw) < static_cast<unsigned>(p.W);
                const int off = ok ? g_pre[j] + tap_off : 0;
                cp_async16_ca(dst0 + j * 512, p.in + off, ok ? 16u : 0u);
              }
            }
          }
          if (!fast1x1) {   // advance the K walk by one stage (64 K elements)
            w_c0 += 64;
            while (w_c0 >= p.Cin) {
              w_c0 -= p.Cin;
              if (++w_kw == p.k) { w_kw = 0; ++w_kh; }
            }
          }
        } else {
          // MODE_HALO: thread owns chunk c and walks the slots s0, s0 + step, ... of the padded-linear range
          const int c = tid & (p.cps - 1);
          const int s0 = tid / p.cps;
          const int step = CONV_NPROD / p.cps;
          const int q = m0 - 1 - p.Wp + s0 + p.Hp1 * p.Wp;       // biased by one virtual image: always >= 0
          int G = fd_div(p.fd_wp, q);
          int cc = q - G * p.Wp;
          int b1 = fd_div(p.fd_hp1, G);
          int r = G - b1 * p.Hp1;
          const __half* chan = p.in + ks * p.cb + c * 8;
          const size_t row_stride = static_cast<size_t>(p.W) * p.in_pitch;
          const __half* rowp = chan + (static_cast<size_t>(b1 - 1) * p.H + r) * row_stride;
          bool row_ok = static_cast<unsigned>(b1 - 1) < static_cast<unsigned>(p.B) && r < p.H;
          uint32_t dst = a_dst + c * p.lbo_a + s0 * 16;
          const uint32_t dst_step = step * 16;
          for (int s = s0; s < p.slots; s += step) {
            const bool ok = row_ok && static_cast<unsigned>(cc - 1) < static_cast<unsigned>(p.W);
            cp_async16_ca(dst, ok ? rowp + static_cast<size_t>(cc - 1) * p.in_pitch : p.in, ok ? 16u : 0u);
            dst += dst_step;
            cc += step;
            if (cc >= p.Wp) {
              do {
                cc -= p.Wp;
                if (++r == p.Hp1) { r = 0; ++b1; }
              } while (cc >= p.Wp);
              rowp = chan + (static_cast<size_t>(b1 - 1) * p.H + r) * row_stride;
              row_ok = static_cast<unsigned>(b1 - 1) < static_cast<unsigned>(p.B) && r < p.H;
            }
          }
        }
        if (!p.b_resident) {
          const uint8_t* src = reinterpret_cast<const uint8_t*>(p.wpack) +
                               (static_cast<size_t>(n_tile) * p.nks + ks) * p.b_stage_bytes;
          const uint32_t b_dst = b_u32 + slot * p.b_stage_bytes;
          for (int i = tid * 16; i < p.b_stage_bytes; i += CONV_NPROD * 16) cp_async16(b_dst + i, src + i, 16);
        }
        cp_async_arrive_noinc(&full[slot]);
      }
    }
    cp_async_wait<0>();   // nothing of this thread may still be in flight when the CTA exits
  } else if (warp == CONV_MMA_WARP) {
    // ======================================= MMA issuer ==========================================
    // all 32 lanes run the loop (uniform control flow); one elected lane issues the tcgen05 instructions
    {
      const uint32_t a_u32 = smem_u32(smem_a);
      const uint32_t b_u32 = smem_u32(smem_b);
      const uint32_t lbo_a16 = static_cast<uint32_t>(p.lbo_a) >> 4;
      const uint32_t lbo_b16 = static_cast<uint32_t>(p.Ntile);            // (Ntile * 16 B) >> 4
      const uint32_t desc_hi = (128u >> 4) | (1u << 14);                  // SBO = 128 B, descriptor version 1
      if (p.b_resident) {
        mbar_wait(bres, 0);
        fence_proxy_async_smem();
      }
      int it = 0, tcount = 0;
      for (int w = blockIdx.x; w < total_work; w += gridDim.x, ++tcount) {
        const int buf = tcount & 1;
        const int use = tcount >> 1;
        if (use >= 1) mbar_wait(&tempty[buf], static_cast<uint32_t>(use - 1) & 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(buf * p.Ntile);
        uint32_t acc = 0;
        for (int ks = 0; ks < p.nks; ++ks, ++it) {
          const int slot = it % p.S;
          mbar_wait(&full[slot], static_cast<uint32_t>(it / p.S) & 1u);
          fence_proxy_async_smem();   // cp.async (generic proxy) writes -> tcgen05.mma (async proxy) reads
          tc_fence_after();
          const uint32_t a_base = a_u32 + slot * p.a_stage_bytes;
          const uint32_t b_base = b_u32 + (p.b_resident ? ks : slot) * p.b_stage_bytes;
          // Descriptors are advanced by adding 16-byte units to their low word (start address field, bits 0-13);
          // the issue loop is a single thread, so it is kept to a handful of instructions per MMA.
          const uint32_t a_lo0 = ((a_base >> 4) & 0x3FFFu) | (lbo_a16 << 16);
          const uint32_t b_lo0 = ((b_base >> 4) & 0x3FFFu) | (lbo_b16 << 16);
          if (p.mode == MODE_GATHER) {
            int kj = (p.K_total - ks * 64) >> 4;
            if (kj > 4) kj = 4;
            uint32_t a_lo = a_lo0, b_lo = b_lo0;
            for (int j = 0; j < kj; ++j) {
              if (elect_one() && !XR_DBG_SKIP(p, 1)) umma_f16(d_tmem, (static_cast<uint64_t>(desc_hi) << 32) | a_lo, (static_cast<uint64_t>(desc_hi) << 32) | b_lo,
                       p.idesc, acc);
              acc = 1;
              a_lo += 2 * lbo_a16;
              b_lo += 2 * lbo_b16;
            }
          } else {
            const int kj = p.cb >> 4;
            uint32_t b_lo = b_lo0;
            for (int kh = 0; kh < 3; ++kh) {
#pragma unroll
              for (int kw = 0; kw < 3; ++kw) {
                uint32_t a_lo = a_lo0 + static_cast<uint32_t>(kh * p.Wp + kw);   // tap shift: one slot = one 16-byte unit
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
      }
    }
  } else {
    // ======================================= epilogue ============================================
    // 8 warps: quadrant q = TMEM lanes 32q..32q+31 (one output row per thread), `half` interleaves the 16-column chunks
    const int ew = warp - CONV_NPROD / 32;
    const int q = ew & 3;
    const int half = ew >> 2;
    const int row = q * 32 + lane;
    int tcount = 0;
    pdl_wait();   // before the first residual read / output store
    for (int w = blockIdx.x; w < total_work; w += gridDim.x, ++tcount) {
      const int m_tile = p.n_tiles == 1 ? w : (w >> 1);
      const int n_tile = p.n_tiles == 1 ? 0 : (w & 1);
      const int m = m_tile * 128 + row;
      // output pixel of this row (transposed conv: base pixel, the 2x2 position comes from the column chunk)
      bool valid = m < p.M_total;
      size_t pix = 0;
      int tb = 0, th = 0, tw = 0;
      if (p.mode == MODE_HALO) {
        const int G = fd_div(p.fd_wp, m);
        const int cc = m - G * p.Wp;
        const int b = fd_div(p.fd_hp1, G);
        const int r = G - b * p.Hp1;
        valid = valid && r < p.H && cc >= 1 && cc <= p.W;
        pix = (static_cast<size_t>(b) * p.H + r) * p.W + (cc - 1);
      } else if (p.transposed) {
        tb = fd_div(p.fd_hw, m);
        const int rem = m - tb * p.fd_hw.d;
        th = fd_div(p.fd_wo, rem);
        tw = rem - th * p.fd_wo.d;
      } else {
        pix = static_cast<size_t>(m);
      }
      const int buf = tcount & 1;
      const int use = tcount >> 1;
      mbar_wait(&tfull[buf], static_cast<uint32_t>(use) & 1u);
      tc_fence_after();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(buf * p.Ntile);
      for (int c0 = half * 16; c0 < p.Ntile; c0 += 32) {
        uint32_t v[16];
        tmem_ld16(t_row + c0, v);
        tmem_ld_wait();
        const int n = n_tile * p.Ntile + c0;
        int co = n;
        if (p.transposed) {
          const int pos = fd_div(p.fd_cout, n);
          co = n - pos * p.Cout;
          pix = (static_cast<size_t>(tb) * p.Ho + (2 * th + (pos >> 1))) * p.Wo + (2 * tw + (pos & 1));
        }
        if (valid && !XR_DBG_SKIP(p, 2))
          epilogue_chunk16(v, bias_s + n, p.act, p.res ? p.res + pix * p.res_pitch + co : nullptr,
                           p.out + pix * p.out_pitch + co);
      }
      tc_fence_before();
      mbar_arrive(&tempty[buf]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == CONV_MMA_WARP) {
    tc_fence_after();
    tmem_dealloc(tmem_base, static_cast<uint32_t>(p.tmem_cols));
  }
}

// Call once per device before the first launch.
static inline void conv_umma_prepare_device() {
  XR_CUDA(cudaFuncSetAttribute(conv_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CONV_SMEM_MAX));
}

static inline void launch_conv_umma(const ConvParams& p, cudaStream_t stream) {
  launch_k(conv_umma_kernel, p.grid, CONV_THREADS, p.smem_bytes, stream, p);
}
#endif  // __CUDACC__

// ---------------------------------------------------------------------------------------------------------------
// host emulation of the kernel's data movement (fp32 math): validates pack order, slot mapping and tap shifts.
// Test infrastructure only -- never on a product path.
// ---------------------------------------------------------------------------------------------------------------
static inline void emulate_conv_umma(const ConvParams& p, const float* in, const float* wpack_f, const float* bias,
                                     const float* res, float* out) {
  const int bchunks = p.b_stage_bytes / (p.Ntile * 16);
  const int lbo_a_slots = p.lbo_a / 16;
  std::vector<float> a(static_cast<size_t>(p.cps) * lbo_a_slots * 8);
  std::vector<float> acc(128 * static_cast<size_t>(p.Ntile));
  for (int w = 0; w < p.m_tiles * p.n_tiles; ++w) {
    const int m_tile = w / p.n_tiles, n_tile = w % p.n_tiles;
    const long m0 = static_cast<long>(m_tile) * 128;
    std::fill(acc.begin(), acc.end(), 0.0f);
    for (int ks = 0; ks < p.nks; ++ks) {
      std::fill(a.begin(), a.end(), 0.0f);
      // loader
      for (int c = 0; c < p.cps; ++c)
        for (int s = 0; s < p.slots; ++s) {
          PixRef pr;
          int c0;
          if (p.mode == MODE_GATHER) {
            pr = gather_pixel(p, m0 + s, (ks * 8 + c) * 8, &c0);
          } else {
            pr = halo_pixel(p, m0 - 1 - p.Wp + s + static_cast<long>(p.Hp1) * p.Wp);
            c0 = ks * p.cb + c * 8;
          }
          if (!pr.valid) continue;
          for (int e = 0; e < 8; ++e)
            a[(static_cast<size_t>(c) * lbo_a_slots + s) * 8 + e] = in[static_cast<size_t>(pr.pix) * p.in_pitch + c0 + e];
        }
      // MMA
      int kj = p.mode == MODE_GATHER ? std::min(4, (p.K_total - ks * 64) / 16) : p.cb / 16;
      const float* bst = wpack_f + (static_cast<size_t>(n_tile) * p.nks + ks) * bchunks * p.Ntile * 8;
      for (int t = 0; t < p.taps; ++t) {
        const int shift = p.mode == MODE_HALO ? (t / 3) * p.Wp + (t % 3) : 0;
        for (int j = 0; j < kj; ++j)
          for (int half_k = 0; half_k < 2; ++half_k) {
            const int ac = 2 * j + half_k;
            const int bc = t * p.cps + 2 * j + half_k;
            for (int i = 0; i < 128; ++i)
              for (int n = 0; n < p.Ntile; ++n) {
                float sacc = 0.f;
                for (int e = 0; e < 8; ++e)
                  sacc += a[(static_cast<size_t>(ac) * lbo_a_slots + i + shift) * 8 + e] *
                          bst[(static_cast<size_t>(bc) * p.Ntile + n) * 8 + e];
                acc[static_cast<size_t>(i) * p.Ntile + n] += sacc;
              }
          }
      }
    }
    // epilogue
    for (int i = 0; i < 128; ++i)
      for (int n = 0; n < p.Ntile; ++n) {
        int co;
        const int ng = n_tile * p.Ntile + n;
        PixRef o = out_pixel(p, m0 + i, ng, &co);
        if (!o.valid) continue;
        float y = acc[static_cast<size_t>(i) * p.Ntile + n] + bias[ng];
        if (p.act) y = y / (1.0f + expf(-y));
        if (res) y += res[static_cast<size_t>(o.pix) * p.res_pitch + co];
        out[static_cast<size_t>(o.pix) * p.out_pitch + co] = y;
      }
  }
}

}  // namespace xrseg
