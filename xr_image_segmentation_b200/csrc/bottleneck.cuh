// bottleneck.cuh -- the thin Bottleneck of a C3k2 block (c3k = False) as ONE kernel: Conv3x3+SiLU -> Conv3x3+SiLU (+ x).
//
// Replaces two launches of the graph per block (SURVEY.md Appendix A: chains b2.m0.cv1/cv2, b4.m0.cv1/cv2 and the neck's
// n13/n16/n19.m0.cv1/cv2, executed through IEExecutor.cs:371,397).  These layers have 8..64 channels: K = 72..576 and
// N = 8..64 keep neither the tensor pipe nor HBM busy as separate tcgen05 launches (b2.m0.cv2: 23 % of HBM peak, most of
// the time is the per-tile hand-over chain of a pipeline that has 9 small MMAs to run per tile), and the intermediate
// tensor makes a round trip through HBM.  Here a CTA owns a TH x TW tile of one frame:
//   1. the (TH+4) x (TW+4) input window (halo 2, zero fill outside the frame = the convs' padding) -> shared memory
//      with cp.async (16 B per request, pixel pitch padded so that ldmatrix rows fall into distinct bank groups);
//   2. conv 1 over the (TH+2) x (TW+2) window (halo 1), bias, SiLU, fp16 -> shared memory; positions outside the frame
//      are written as ZERO (they are conv 2's padding, not conv-1-of-padding);
//   3. conv 2 over the tile, bias, SiLU, + the block input (read back from the window of step 1), fp16 -> global.
// Both convs are implicit GEMMs on mma.sync m16n8k16 (fp16 in, fp32 accumulate): an M-tile is 16 consecutive pixels of
// the flattened window, its A fragment is ONE ldmatrix.x4 whose row addresses are the pixels shifted by the tap, K runs
// tap-major / channel-minor.  Weights are pre-packed on the host in B-fragment order (one 8-byte load per lane and
// n-tile).  Two M-tiles share every B fragment.  The 16..64-channel tiles are far too small for a TMEM pipeline
// (same reasoning as the stem and the attention kernel); the intermediate never leaves the SM.
// Numerics are those of the two separate launches: fp32 accumulation, bias in fp32, SiLU through tanh.approx.f16x2,
// fp16 intermediate, residual added in packed fp16 (common.cuh: epilogue_chunk16).
#pragma once

#include <vector>

#include "common.cuh"

namespace xrseg {

struct BneckParams {
  const __half* in; int in_pitch;      // [B,H,W,>=C1]  block input (and residual)
  __half* out; int out_pitch;          // [B,H,W,>=C2]
  const uint2* w1; const uint2* w2;    // fragment-ordered fp16 weights (pack_bneck_weights)
  const float* b1; const float* b2;    // [CM], [C2]
  int B, H, W;
};

// Tile geometry: the output tile is TH x 14 pixels, so the halo-1 window of the intermediate is exactly 16 pixels wide:
// an M-tile of conv 1 is one ROW of that window, an M-tile of conv 2 is one row of the tile (14 pixels + 2 discarded).
// Rows are warp-uniform, the pixel of a lane inside its row is lane % 16 -- no index arithmetic beyond a multiply-add.
// 14 divides the network's maps with <= 5 % overhang (160 -> 12 x 14, 80 -> 6 x 14, 40 -> 3 x 14).
constexpr int BNECK_TW = 14;

template <int C1, int CM, int C2, int TH>
struct BneckCfg {
  static constexpr int TW = BNECK_TW;
  static constexpr int IW = TW + 4, IH = TH + 4, MW = TW + 2, MH = TH + 2;
  static constexpr int P1 = C1 * 2 + (C1 >= 16 ? 16 : 0);   // bytes per pixel of the input window in shared memory
  static constexpr int PM = CM * 2 + (CM >= 16 ? 16 : 0);   // ... of the intermediate window
  static constexpr int KS1 = (9 * C1 + 15) / 16, KS2 = (9 * CM + 15) / 16;
  static constexpr int NT1 = CM / 8, NT2 = C2 / 8;
  static constexpr int W1_BYTES = KS1 * NT1 * 256, W2_BYTES = KS2 * NT2 * 256;
  static constexpr int IN_BYTES = (IH * IW * P1 + 127) / 128 * 128;
  static constexpr int MID_BYTES = ((MH * MW + 2) * PM + 127) / 128 * 128;   // + 2 pixels: conv 2's discarded columns read past the end
  static constexpr int BIAS_BYTES = (CM + C2) * 4;
  static constexpr int SMEM_BYTES = IN_BYTES + MID_BYTES + W1_BYTES + W2_BYTES + BIAS_BYTES;
  static_assert(C1 % 16 == 0 && CM % 8 == 0 && C2 % 16 == 0 && TH % 2 == 0 && MW == 16, "tile geometry");
};

#ifdef __CUDACC__

__device__ __forceinline__ void bneck_hmma(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void bneck_ldmatrix_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}

// acc[m][nt][4] += conv3x3 of two M-tiles.  a_base[m]: shared address of the lane's row pixel (window coordinates of
// the top-left tap), SW: window width in pixels, P: pixel pitch in bytes, C: channels per pixel (K = 9 C, tap-major).
// Lanes 16..31 supply the second 8-channel chunk of a k-step: for C >= 16 that is 16 bytes further in the same pixel,
// for C == 8 it is the NEXT tap's pixel (the ninth step pairs tap 8 with itself; its weights are zero).
template <int C, int NT, int SW, int P>
__device__ __forceinline__ void bneck_conv_tiles(float (&acc)[2][NT][4], const uint32_t (&a_base)[2], const uint2* s_w, int lane) {
  constexpr int KS = (9 * C + 15) / 16;
  const int hi = lane >> 4;
  const uint32_t base0 = a_base[0] + (C >= 16 ? hi * 16 : 0), base1 = a_base[1] + (C >= 16 ? hi * 16 : 0);
#pragma unroll
  for (int s = 0; s < KS; ++s) {
    uint32_t off;
    if constexpr (C >= 16) {
      constexpr int per_tap = C / 16;
      const int tap = s / per_tap, cc = s % per_tap;
      off = ((tap / 3) * SW + tap % 3) * P + cc * 32;
    } else {
      const int t0 = 2 * s, t1 = (2 * s + 1 < 9) ? 2 * s + 1 : 8;
      const int o0 = ((t0 / 3) * SW + t0 % 3) * P, o1 = ((t1 / 3) * SW + t1 % 3) * P;
      off = hi ? o1 : o0;
    }
    uint32_t a[2][4];
    bneck_ldmatrix_x4(a[0], base0 + off);
    bneck_ldmatrix_x4(a[1], base1 + off);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const uint2 bw = s_w[(s * NT + nt) * 32 + lane];
      bneck_hmma(acc[0][nt], a[0], bw.x, bw.y);
      bneck_hmma(acc[1][nt], a[1], bw.x, bw.y);
    }
  }
}

template <int C1, int CM, int C2, int TH, bool RES>
__global__ void __launch_bounds__(256) bottleneck_mma_kernel(const BneckParams p) {
  using Cfg = BneckCfg<C1, CM, C2, TH>;
  static_assert(!RES || C1 == C2, "the residual is the block input");
  constexpr int TW = Cfg::TW, IW = Cfg::IW, IH = Cfg::IH, MW = Cfg::MW, MH = Cfg::MH, P1 = Cfg::P1, PM = Cfg::PM;
  constexpr int NT1 = Cfg::NT1, NT2 = Cfg::NT2;
  extern __shared__ __align__(128) uint8_t bneck_smem[];
  uint8_t* s_in = bneck_smem;
  uint8_t* s_mid = s_in + Cfg::IN_BYTES;
  uint2* s_w1 = reinterpret_cast<uint2*>(s_mid + Cfg::MID_BYTES);
  uint2* s_w2 = reinterpret_cast<uint2*>(reinterpret_cast<uint8_t*>(s_w1) + Cfg::W1_BYTES);
  float* s_b1 = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(s_w2) + Cfg::W2_BYTES);
  float* s_b2 = s_b1 + CM;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int tx0 = blockIdx.x * TW, ty0 = blockIdx.y * TH, b = blockIdx.z;

  pdl_launch_dependents();
  // weights and biases are constants of the runner: fetched before waiting for the producer of the input
  for (int i = tid; i < Cfg::W1_BYTES / 16; i += 256)
    cp_async16(smem_u32(s_w1) + 16 * i, reinterpret_cast<const uint8_t*>(p.w1) + 16 * i, 16);
  for (int i = tid; i < Cfg::W2_BYTES / 16; i += 256)
    cp_async16(smem_u32(s_w2) + 16 * i, reinterpret_cast<const uint8_t*>(p.w2) + 16 * i, 16);
  cp_async_commit();
  for (int i = tid; i < CM + C2; i += 256) s_b1[i] = i < CM ? p.b1[i] : p.b2[i - CM];
  pdl_wait();

  // 1. input window: (row, pixel, 16-byte chunk) units, zero outside the frame.  Plain 16-byte loads into registers and
  //    16-byte shared stores: the pixels of a channel slice are 32..64-byte islands in global memory, and cp.async
  //    writes shared memory once per returning sector (ncu: 27 shared wavefronts per LDGSTS instead of 4).
  {
    constexpr int CH1 = C1 / 8, ROW = IW * CH1, TOTAL = IH * ROW, ITERS = (TOTAL + 255) / 256;
    const __half* img = p.in + static_cast<size_t>(b) * p.H * p.W * p.in_pitch;
    uint4 v[ITERS];
#pragma unroll
    for (int k = 0; k < ITERS; ++k) {
      const int i = tid + 256 * k;
      const int r = i / ROW, j = i - r * ROW;
      const int col = j / CH1, c = j - col * CH1;
      const int y = ty0 - 2 + r, x = tx0 - 2 + col;
      v[k] = make_uint4(0u, 0u, 0u, 0u);
      if (i < TOTAL && y >= 0 && y < p.H && x >= 0 && x < p.W)
        v[k] = __ldcg(reinterpret_cast<const uint4*>(img + (static_cast<size_t>(y) * p.W + x) * p.in_pitch + c * 8));
    }
#pragma unroll
    for (int k = 0; k < ITERS; ++k) {
      const int i = tid + 256 * k;
      const int r = i / ROW, j = i - r * ROW;
      const int col = j / CH1, c = j - col * CH1;
      if (i < TOTAL) *reinterpret_cast<uint4*>(s_in + (r * IW + col) * P1 + c * 16) = v[k];
    }
    cp_async_wait<0>();   // the weights
  }
  __syncthreads();

  // 2. conv 1: one M-tile per row of the halo-1 window -> s_mid (zero outside the frame)
  {
    float bias[NT1][2];
#pragma unroll
    for (int nt = 0; nt < NT1; ++nt) { bias[nt][0] = s_b1[nt * 8 + 2 * t]; bias[nt][1] = s_b1[nt * 8 + 2 * t + 1]; }
    for (int u = warp; u < MH / 2; u += 8) {
      float acc[2][NT1][4];
      uint32_t a_base[2];
#pragma unroll
      for (int m = 0; m < 2; ++m) {
#pragma unroll
        for (int nt = 0; nt < NT1; ++nt) acc[m][nt][0] = acc[m][nt][1] = acc[m][nt][2] = acc[m][nt][3] = 0.f;
        a_base[m] = smem_u32(s_in) + ((2 * u + m) * IW + (lane & 15)) * P1;
      }
      bneck_conv_tiles<C1, NT1, IW, P1>(acc, a_base, s_w1, lane);
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        const int qy = 2 * u + m, y = ty0 - 1 + qy;
        const bool row_ok = y >= 0 && y < p.H;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int qx = g + 8 * h, x = tx0 - 1 + qx;
          const bool ok = row_ok && x >= 0 && x < p.W;
          uint8_t* dst = s_mid + (qy * MW + qx) * PM + 4 * t;
#pragma unroll
          for (int nt = 0; nt < NT1; ++nt) {
            const uint32_t v = silu_pack_h2(acc[m][nt][2 * h] + bias[nt][0], acc[m][nt][2 * h + 1] + bias[nt][1]);
            *reinterpret_cast<uint32_t*>(dst + nt * 16) = ok ? v : 0u;
          }
        }
      }
    }
  }
  __syncthreads();

  // 3. conv 2: one M-tile per row of the tile (pixels 14, 15 of a row are discarded), + residual -> global
  {
    float bias[NT2][2];
#pragma unroll
    for (int nt = 0; nt < NT2; ++nt) { bias[nt][0] = s_b2[nt * 8 + 2 * t]; bias[nt][1] = s_b2[nt * 8 + 2 * t + 1]; }
    __half* img = p.out + static_cast<size_t>(b) * p.H * p.W * p.out_pitch;
    for (int u = warp; u < TH / 2; u += 8) {
      float acc[2][NT2][4];
      uint32_t a_base[2];
#pragma unroll
      for (int m = 0; m < 2; ++m) {
#pragma unroll
        for (int nt = 0; nt < NT2; ++nt) acc[m][nt][0] = acc[m][nt][1] = acc[m][nt][2] = acc[m][nt][3] = 0.f;
        a_base[m] = smem_u32(s_mid) + ((2 * u + m) * MW + (lane & 15)) * PM;
      }
      bneck_conv_tiles<CM, NT2, MW, PM>(acc, a_base, s_w2, lane);
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        const int oy = 2 * u + m, y = ty0 + oy;
        __half* row = img + (static_cast<size_t>(y) * p.W + tx0) * p.out_pitch;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int ox = g + 8 * h, x = tx0 + ox;
          const bool ok = y < p.H && ox < TW && x < p.W;
          uint32_t v[NT2];
#pragma unroll
          for (int nt = 0; nt < NT2; ++nt) {
            v[nt] = silu_pack_h2(acc[m][nt][2 * h] + bias[nt][0], acc[m][nt][2 * h + 1] + bias[nt][1]);
            if constexpr (RES) {
              const uint32_t rr = *reinterpret_cast<const uint32_t*>(s_in + ((oy + 2) * IW + ox + 2) * P1 + nt * 16 + 4 * t);
              const __half2 s2 = __hadd2(*reinterpret_cast<const __half2*>(&v[nt]), *reinterpret_cast<const __half2*>(&rr));
              v[nt] = *reinterpret_cast<const uint32_t*>(&s2);
            }
          }
          uint32_t* dst = reinterpret_cast<uint32_t*>(row + ox * p.out_pitch + 2 * t);
#pragma unroll
          for (int nt = 0; nt < NT2; ++nt)
            if (ok) dst[nt * 4] = v[nt];
        }
      }
    }
  }
}

#endif  // __CUDACC__

// B-fragment order of mma.sync m16n8k16 for W[k][n], k = tap * C + c (tap-major over the C channels of the shared-memory
// window, zero beyond the real channel counts and beyond K = 9 C): per (k-step, n-tile, lane) two 32-bit words
//   b0 = { W[16 s + 2 t][n], W[16 s + 2 t + 1][n] },  b1 = { W[16 s + 2 t + 8][n], W[16 s + 2 t + 9][n] },  n = 8 nt + lane / 4,
// t = lane % 4.  w: the layer's weights [cout][cin][3][3] (fp32; taps = 1: [cout][cin]), N: padded output channels (multiple of 8).
static inline void pack_bneck_weights(const float* w, int cin, int cout, int C, int N, std::vector<uint32_t>& out, int taps = 9) {
  const int K = taps * C, KS = (K + 15) / 16, NT = N / 8;
  out.assign(static_cast<size_t>(KS) * NT * 64, 0u);
  auto W = [&](int k, int n) -> float {
    if (k >= K || n >= cout) return 0.f;
    const int tap = k / C, c = k % C;
    if (c >= cin) return 0.f;
    return w[(static_cast<size_t>(n) * cin + c) * taps + tap];
  };
  auto pack = [](float lo, float hi) -> uint32_t {
    const __half l = __half(lo), h = __half(hi);
    uint16_t lb, hb;
    memcpy(&lb, &l, 2);
    memcpy(&hb, &h, 2);
    return static_cast<uint32_t>(lb) | (static_cast<uint32_t>(hb) << 16);
  };
  for (int s = 0; s < KS; ++s)
    for (int nt = 0; nt < NT; ++nt)
      for (int lane = 0; lane < 32; ++lane) {
        const int n = nt * 8 + (lane >> 2), k0 = 16 * s + 2 * (lane & 3);
        uint32_t* o = &out[((static_cast<size_t>(s) * NT + nt) * 32 + lane) * 2];
        o[0] = pack(W(k0, n), W(k0 + 1, n));
        o[1] = pack(W(k0 + 8, n), W(k0 + 9, n));
      }
}

}  // namespace xrseg
