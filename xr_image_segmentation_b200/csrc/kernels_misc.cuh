// kernels_misc.cuh -- the memory-bound CUDA-core kernels around the tensor-core convolutions:
// frame preprocessing (↔ TextureConverter.ToTensor, IEExecutor.cs:370), the K=27 stem convolution, depthwise 3x3
// convolutions, the fused SPPF max-pool chain, nearest x2 upsampling into a concat slice, the C2PSA attention, and a
// plain direct convolution used as the on-GPU cross-check of the tcgen05 path.  All activations are NHWC fp16.
#pragma once

#include "common.cuh"

namespace xrseg {

// A view of an NHWC fp16 tensor: channel slice [coff, coff + C) of a buffer whose pixel pitch is `pitch` elements.
struct TView {
  __half* ptr = nullptr;  // already offset to the first channel of the slice
  int B = 0, H = 0, W = 0, C = 0, pitch = 0;
};

#ifdef __CUDACC__

// ------------------------------------------------------------------------------------------------
// preprocess: u8 RGB/RGBA frames (any size) -> fp16 NHWC [B,640,640,4] (4th channel 0), values 0..1
// stretch: bilinear sample at (x+0.5)*sw/640-0.5, clamp; letterbox: scale r = min(640/h, 640/w), pad 114.
// ------------------------------------------------------------------------------------------------
struct PreParams {
  const uint8_t* src;
  __half* dst;
  int B, sw, sh, stride_bytes, bpp;
  int mode;         // 0 stretch, 1 letterbox
  float scale_x, scale_y;
  int left, top, nw, nh;   // letterbox placement
  int flip;                // 1: the frame's rows are stored bottom-up (Unity GetPixels32 / texture origin bottom-left)
};

__global__ void preprocess_kernel(const PreParams p) {
  XR_PDL_ENTRY();
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  const int b = blockIdx.z;
  if (x >= 640) return;
  const uint8_t* img = p.src + static_cast<size_t>(b) * p.sh * p.stride_bytes;
  float rgb[3];
  bool inside = true;
  int xx = x, yy = y;
  if (p.mode == 1) {
    xx = x - p.left;
    yy = y - p.top;
    inside = (xx >= 0 && xx < p.nw && yy >= 0 && yy < p.nh);
  }
  if (inside) {
    // two roundings in the oracle's order (oracle/preprocess._axis); left to nvcc, the product and the subtraction contract
    // into one FFMA
    const float fx = __fsub_rn(__fmul_rn(static_cast<float>(xx) + 0.5f, p.scale_x), 0.5f);
    const float fy = __fsub_rn(__fmul_rn(static_cast<float>(yy) + 0.5f, p.scale_y), 0.5f);
    const float x0f = floorf(fx), y0f = floorf(fy);
    const float tx = fx - x0f, ty = fy - y0f;
    int x0 = static_cast<int>(x0f), y0 = static_cast<int>(y0f);
    int x1 = x0 + 1, y1 = y0 + 1;
    x0 = min(max(x0, 0), p.sw - 1); x1 = min(max(x1, 0), p.sw - 1);
    y0 = min(max(y0, 0), p.sh - 1); y1 = min(max(y1, 0), p.sh - 1);
    const uint8_t* r0 = img + static_cast<size_t>(p.flip ? p.sh - 1 - y0 : y0) * p.stride_bytes;
    const uint8_t* r1 = img + static_cast<size_t>(p.flip ? p.sh - 1 - y1 : y1) * p.stride_bytes;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float a = static_cast<float>(r0[x0 * p.bpp + c]), bq = static_cast<float>(r0[x1 * p.bpp + c]);
      const float cq = static_cast<float>(r1[x0 * p.bpp + c]), d = static_cast<float>(r1[x1 * p.bpp + c]);
      const float top = __fadd_rn(__fmul_rn(a, 1.0f - tx), __fmul_rn(bq, tx));
      const float bot = __fadd_rn(__fmul_rn(cq, 1.0f - tx), __fmul_rn(d, tx));
      const float v = __fadd_rn(__fmul_rn(top, 1.0f - ty), __fmul_rn(bot, ty));
      rgb[c] = __fdiv_rn(v, 255.0f);
    }
  } else {
    rgb[0] = rgb[1] = rgb[2] = __fdiv_rn(114.0f, 255.0f);
  }
  __half2 lo = __floats2half2_rn(rgb[0], rgb[1]);
  __half2 hi = __floats2half2_rn(rgb[2], 0.0f);
  uint2 o;
  o.x = *reinterpret_cast<uint32_t*>(&lo);
  o.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(p.dst + ((static_cast<size_t>(b) * 640 + y) * 640 + x) * 4) = o;
}

// ------------------------------------------------------------------------------------------------
// stem: 3x3 stride-2 conv on the 4-channel fp16 image (K = 27 real taps), + bias + SiLU.  One thread per output
// pixel and 16 output channels; weights fp32 in shared memory as [tap(9)][ci(4)][co].
// ------------------------------------------------------------------------------------------------
struct StemParams {
  const __half* in;    // [B,H,W,4]
  __half* out;         // [B,H/2,W/2,Cout] pitch out_pitch
  const float* w;      // [9][4][Cout]
  const float* bias;   // [Cout]
  int B, H, W, Cout, out_pitch;
};

__global__ void __launch_bounds__(256) stem_conv_kernel(const StemParams p) {
  XR_PDL_ENTRY();
  extern __shared__ float sw[];  // 36*Cout weights + Cout bias
  for (int i = threadIdx.x; i < 36 * p.Cout; i += blockDim.x) sw[i] = p.w[i];
  for (int i = threadIdx.x; i < p.Cout; i += blockDim.x) sw[36 * p.Cout + i] = p.bias[i];
  __syncthreads();
  const int Ho = p.H / 2, Wo = p.W / 2;
  const int groups = p.Cout / 16;
  const long total = static_cast<long>(p.B) * Ho * Wo * groups;
  for (long idx = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long>(gridDim.x) * blockDim.x) {
    const int g = static_cast<int>(idx % groups);
    long pix = idx / groups;
    const int ow = static_cast<int>(pix % Wo);
    const int oh = static_cast<int>((pix / Wo) % Ho);
    const int b = static_cast<int>(pix / (static_cast<long>(Wo) * Ho));
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = sw[36 * p.Cout + g * 16 + i];
#pragma unroll
    for (int kh = 0; kh < 3; ++kh) {
      const int ih = oh * 2 - 1 + kh;
      if (ih < 0 || ih >= p.H) continue;
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const int iw = ow * 2 - 1 + kw;
        if (iw < 0 || iw >= p.W) continue;
        const uint2 raw = *reinterpret_cast<const uint2*>(p.in + ((static_cast<size_t>(b) * p.H + ih) * p.W + iw) * 4);
        const float2 f01 = __half22float2(*reinterpret_cast<const __half2*>(&raw.x));
        const float2 f23 = __half22float2(*reinterpret_cast<const __half2*>(&raw.y));
        const float xin[3] = {f01.x, f01.y, f23.x};
        const float* wt = sw + (kh * 3 + kw) * 4 * p.Cout + g * 16;
#pragma unroll
        for (int ci = 0; ci < 3; ++ci)
#pragma unroll
          for (int i = 0; i < 16; ++i) acc[i] = fmaf(xin[ci], wt[ci * p.Cout + i], acc[i]);
      }
    }
    uint4 o0, o1;
    __half2* q0 = reinterpret_cast<__half2*>(&o0);
    __half2* q1 = reinterpret_cast<__half2*>(&o1);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      q0[i] = __floats2half2_rn(silu_f(acc[2 * i]), silu_f(acc[2 * i + 1]));
      q1[i] = __floats2half2_rn(silu_f(acc[8 + 2 * i]), silu_f(acc[8 + 2 * i + 1]));
    }
    uint4* op = reinterpret_cast<uint4*>(p.out + static_cast<size_t>(pix) * p.out_pitch + g * 16);
    op[0] = o0;
    op[1] = o1;
  }
}

// ------------------------------------------------------------------------------------------------
// fused preprocess + stem for frames that already are 640x640 (no resample needed): reads the uint8 RGB / RGBA frame
// directly (u8 / 255 is folded into the weights), 3x3 stride-2 conv + bias + SiLU -> fp16 NHWC.  Saves the fp16 image
// round trip of the two-kernel path.  Block = 16x16 output pixels; the 33x33 input patch is staged in shared memory.
// ------------------------------------------------------------------------------------------------
struct StemU8Params {
  const uint8_t* src; int stride_bytes, bpp;   // [B,H,W,bpp]
  __half* out; int out_pitch;
  const float* w;      // [9][4][Cout], already divided by 255
  const float* bias;
  int B, H, W, Cout;
  int flip;            // rows stored bottom-up
};

__global__ void __launch_bounds__(256) stem_u8_kernel(const StemU8Params p) {
  XR_PDL_ENTRY();
  extern __shared__ float sw[];                 // 36*Cout weights + Cout bias, then the u8 patch
  uint8_t* patch = reinterpret_cast<uint8_t*>(sw + 37 * p.Cout);   // [33][33][4]
  for (int i = threadIdx.x; i < 36 * p.Cout; i += 256) sw[i] = p.w[i];
  for (int i = threadIdx.x; i < p.Cout; i += 256) sw[36 * p.Cout + i] = p.bias[i];
  const int Ho = p.H / 2, Wo = p.W / 2;
  const int ox0 = blockIdx.x * 16, oy0 = blockIdx.y * 16, b = blockIdx.z;
  const uint8_t* img = p.src + static_cast<size_t>(b) * p.H * p.stride_bytes;
  const int ix0 = ox0 * 2 - 1, iy0 = oy0 * 2 - 1;
  for (int i = threadIdx.x; i < 33 * 33; i += 256) {
    const int py = i / 33, px = i - py * 33;
    const int iy = iy0 + py, ix = ix0 + px;
    uint32_t v = 0;
    if (iy >= 0 && iy < p.H && ix >= 0 && ix < p.W) {
      const uint8_t* s = img + static_cast<size_t>(p.flip ? p.H - 1 - iy : iy) * p.stride_bytes + ix * p.bpp;
      v = s[0] | (s[1] << 8) | (s[2] << 16);
    }
    reinterpret_cast<uint32_t*>(patch)[i] = v;
  }
  __syncthreads();
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int ox = ox0 + tx, oy = oy0 + ty;
  if (ox >= Wo || oy >= Ho) return;
  const size_t pix = (static_cast<size_t>(b) * Ho + oy) * Wo + ox;
  for (int g = 0; g < p.Cout / 16; ++g) {
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = sw[36 * p.Cout + g * 16 + i];
#pragma unroll
    for (int kh = 0; kh < 3; ++kh)
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const uint32_t v = reinterpret_cast<const uint32_t*>(patch)[(2 * ty + kh) * 33 + 2 * tx + kw];
        const float xin[3] = {static_cast<float>(v & 0xFF), static_cast<float>((v >> 8) & 0xFF),
                              static_cast<float>((v >> 16) & 0xFF)};
        const float* wt = sw + (kh * 3 + kw) * 4 * p.Cout + g * 16;
#pragma unroll
        for (int ci = 0; ci < 3; ++ci)
#pragma unroll
          for (int i = 0; i < 16; ++i) acc[i] = fmaf(xin[ci], wt[ci * p.Cout + i], acc[i]);
      }
    uint32_t o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = silu_pack_h2(acc[2 * i], acc[2 * i + 1]);
    uint4* op = reinterpret_cast<uint4*>(p.out + pix * p.out_pitch + g * 16);
    op[0] = make_uint4(o[0], o[1], o[2], o[3]);
    op[1] = make_uint4(o[4], o[5], o[6], o[7]);
  }
}

// ------------------------------------------------------------------------------------------------
// depthwise 3x3 stride-1 pad-1 conv (+bias, optional SiLU, optional residual add).  weights fp32 [9][C], bias [C].
// A thread owns one (x, 8-channel group) column and walks DOWN a strip of rows with a 3x3 register window: per
// output it issues three coalesced 16-byte loads (x-1, x, x+1 of the incoming row; the side columns are L1 hits of
// the neighbouring threads' centre loads) instead of nine, and its 72 weights live in registers.  32-bit index math,
// one block = 128 consecutive (x, group) columns of one image strip.
// Channel remap: input channel of output channel c is (c / in_grp) * in_grp_stride + in_grp_off + c % in_grp when
// in_grp > 0 -- lets the C2PSA positional-encoding conv read V straight out of the interleaved qkv tensor.
// ------------------------------------------------------------------------------------------------
struct DwParams {
  const __half* in; int in_pitch;
  __half* out; int out_pitch;
  const __half* res; int res_pitch;   // optional, added after activation
  const float* w; const float* bias;
  int B, H, W, C, act;
  int rows;                           // rows per strip (grid.y = ceil(H / rows))
  int in_grp, in_grp_stride, in_grp_off;
};

__device__ __forceinline__ void dw_fma8(float (&acc)[8], const uint4 v, const float (&w)[8]) {
  const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __half22float2(h[i]);
    acc[2 * i] = fmaf(f.x, w[2 * i], acc[2 * i]);
    acc[2 * i + 1] = fmaf(f.y, w[2 * i + 1], acc[2 * i + 1]);
  }
}

// Arithmetic: each kernel ROW (three taps) is a packed-half HMUL2 + 2 HFMA2 chain, the three row sums and the bias are
// added in fp32.  Against a full fp32 accumulation this adds ~1e-3 relative error (the output is rounded to fp16 anyway)
// and cuts the instruction count per 8 outputs from ~150 (72 conversions + 72 FMAs) to ~50; with the weights held as
// 36 half2 registers the kernel also fits more blocks per SM.
// NV = half2 lanes per thread: a thread owns 2*NV channels of one pixel column; the network launches NV = 4 (eight channels,
// 16-byte accesses).  NV = 2 halves the per-thread state (~60 registers) and doubles the occupancy: measured equal.  Staging
// the input tile in shared memory (fetched once by cp.async) was measured slower on B200: h3.cls.0dw / 1dw 51.5 / 59.9 us
// against 48.2 / 51.6 us -- the barrier between fill and compute costs more than the L1 re-reads it saves.
template <int NV>
struct alignas(NV * 4) DwVec {
  uint32_t v[NV];
};

template <int NV>
__global__ void __launch_bounds__(128, NV == 2 ? 8 : 4) dwconv3x3_kernel(const DwParams p) {
  XR_PDL_ENTRY();
  constexpr int CPT = 2 * NV;                           // channels per thread
  using Vec = DwVec<NV>;
  const int cgs = p.C / CPT;
  const int col = blockIdx.x * 128 + threadIdx.x;       // (x, group) column, group fastest
  if (col >= p.W * cgs) return;
  const int x = col / cgs, g = col - x * cgs;
  const int b = blockIdx.z;
  const int y0 = blockIdx.y * p.rows;
  const int y1 = min(y0 + p.rows, p.H);
  const int c = g * CPT;
  const int cin = p.in_grp > 0 ? (c / p.in_grp) * p.in_grp_stride + p.in_grp_off + c % p.in_grp : c;
  __half2 w[9][NV];
  float bias[CPT];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float2 wf = *reinterpret_cast<const float2*>(p.w + t * p.C + c + 2 * i);
      w[t][i] = __floats2half2_rn(wf.x, wf.y);
    }
#pragma unroll
  for (int i = 0; i < CPT; ++i) bias[i] = p.bias[c + i];
  const bool has_l = x > 0, has_r = x + 1 < p.W;
  const size_t row_elems = static_cast<size_t>(p.W) * p.in_pitch;
  const __half* src = p.in + static_cast<size_t>(b) * p.H * row_elems + static_cast<size_t>(x) * p.in_pitch + cin;
  Vec zero;
#pragma unroll
  for (int i = 0; i < NV; ++i) zero.v[i] = 0u;
  // Output row y needs input rows y-1, y, y+1 against kernel rows 0, 1, 2.  An input row is loaded ONCE and its three
  // row sums (against kh = 0, 1, 2) are kept in a rolling window: rs[kh] of input rows y-1+kh.
  __half2 s_up0[NV], s_mid1[NV], s_mid0[NV], s_dn2[NV], s_dn1[NV], s_dn0[NV];
  // raw input row (left / centre / right pixel); rows outside the image are zero
  auto load_raw = [&](int y, Vec& vl, Vec& vc, Vec& vr) {
    if (y < 0 || y >= p.H) {
      vl = vc = vr = zero;
      return;
    }
    const __half* q = src + static_cast<size_t>(y) * row_elems;
    vc = *reinterpret_cast<const Vec*>(q);
    vl = has_l ? *reinterpret_cast<const Vec*>(q - p.in_pitch) : zero;
    vr = has_r ? *reinterpret_cast<const Vec*>(q + p.in_pitch) : zero;
  };
  auto sums_of = [&](const Vec& vl, const Vec& vc, const Vec& vr, __half2 (&a0)[NV], __half2 (&a1)[NV], __half2 (&a2)[NV]) {
    const __half2* hl = reinterpret_cast<const __half2*>(vl.v);
    const __half2* hc = reinterpret_cast<const __half2*>(vc.v);
    const __half2* hr = reinterpret_cast<const __half2*>(vr.v);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      a0[i] = __hfma2(hr[i], w[2][i], __hfma2(hc[i], w[1][i], __hmul2(hl[i], w[0][i])));
      a1[i] = __hfma2(hr[i], w[5][i], __hfma2(hc[i], w[4][i], __hmul2(hl[i], w[3][i])));
      a2[i] = __hfma2(hr[i], w[8][i], __hfma2(hc[i], w[7][i], __hmul2(hl[i], w[6][i])));
    }
  };
  __half2 dummy[NV];
  Vec rl, rc, rr;
  // prologue: input row y0-1 contributes kernel row 0 to output y0; input row y0 contributes row 1 to y0 and row 0 to y0+1
  load_raw(y0 - 1, rl, rc, rr);
  sums_of(rl, rc, rr, s_up0, dummy, dummy);
  load_raw(y0, rl, rc, rr);
  sums_of(rl, rc, rr, s_mid0, s_mid1, dummy);
  load_raw(y0 + 1, rl, rc, rr);                  // the loop always has the NEXT input row's loads in flight (two rows ahead:
  size_t opix = (static_cast<size_t>(b) * p.H + y0) * p.W + x;   // 107 registers, h3.cls.0dw 47.7 -> 45.5 us, 1dw 51.5 -> 53.2 us: no gain)
  for (int y = y0; y < y1; ++y, opix += p.W) {
    Vec nl, nc, nr;
    load_raw(y + 2, nl, nc, nr);                 // prefetch for the next iteration (zero rows past the image)
    sums_of(rl, rc, rr, s_dn0, s_dn1, s_dn2);    // input row y+1: kernel row 2 for output y, row 1 for y+1, row 0 for y+2
    rl = nl; rc = nc; rr = nr;
    float acc[CPT];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float2 a = __half22float2(s_up0[i]), m = __half22float2(s_mid1[i]), d = __half22float2(s_dn2[i]);
      acc[2 * i] = bias[2 * i] + a.x + m.x + d.x;
      acc[2 * i + 1] = bias[2 * i + 1] + a.y + m.y + d.y;
    }
    Vec o;
    if (p.act) {
#pragma unroll
      for (int i = 0; i < NV; ++i) o.v[i] = silu_pack_h2(acc[2 * i], acc[2 * i + 1]);
    } else {
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        __half2 hh = __floats2half2_rn(acc[2 * i], acc[2 * i + 1]);
        o.v[i] = *reinterpret_cast<uint32_t*>(&hh);
      }
    }
    if (p.res) {
      const Vec raw = *reinterpret_cast<const Vec*>(p.res + opix * p.res_pitch + c);
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        __half2 sum = __hadd2(*reinterpret_cast<__half2*>(&o.v[i]), *reinterpret_cast<const __half2*>(&raw.v[i]));
        o.v[i] = *reinterpret_cast<uint32_t*>(&sum);
      }
    }
    *reinterpret_cast<Vec*>(p.out + opix * p.out_pitch + c) = o;
    // roll: the row below becomes the middle row, the middle row becomes the row above
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      s_up0[i] = s_mid0[i];
      s_mid0[i] = s_dn0[i];
      s_mid1[i] = s_dn1[i];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// SPPF pooling chain (graph chains 144-147): y1 = maxpool5(y0), y2 = maxpool5(y1), y3 = maxpool5(y2), written into
// the three channel slices after y0 of the concat buffer.  One block per (image, 8-channel group); the HxW map
// (20x20) lives in shared memory.  Chained 5x5 pools equal 5x5, 9x9 and 13x13 windows of y0.
// ------------------------------------------------------------------------------------------------
struct SppfParams {
  __half* buf;   // concat buffer [B,H,W,4C]: slice 0 holds y0 (input), slices 1..3 are written
  int B, H, W, C, pitch;
};

__global__ void __launch_bounds__(256) sppf_pool_kernel(const SppfParams p) {
  XR_PDL_ENTRY();
  extern __shared__ uint4 sp4[];    // two ping-pong maps of [H*W] x 8 channels
  const int cg = p.C / 8;
  const int g = blockIdx.x % cg;
  const int b = blockIdx.x / cg;
  const int n = p.H * p.W;
  uint4* cur = sp4;
  uint4* tmp = sp4 + n;
  __half* base = p.buf + static_cast<size_t>(b) * n * p.pitch + g * 8;
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    cur[i] = *reinterpret_cast<const uint4*>(base + static_cast<size_t>(i) * p.pitch);
  __syncthreads();
  auto max4 = [](uint4 a, const uint4 c) {
    __half2* x = reinterpret_cast<__half2*>(&a);
    const __half2* y = reinterpret_cast<const __half2*>(&c);
#pragma unroll
    for (int k = 0; k < 4; ++k) x[k] = __hmax2(x[k], y[k]);
    return a;
  };
  // three chained 5x5 stride-1 pools (pad 2 = window clipped at the border), each done separably: rows, then columns
  for (int r = 0; r < 3; ++r) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const int y = i / p.W, x = i - y * p.W;
      uint4 m = cur[i];
      for (int dx = -2; dx <= 2; ++dx)
        if (dx != 0 && x + dx >= 0 && x + dx < p.W) m = max4(m, cur[i + dx]);
      tmp[i] = m;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const int y = i / p.W;
      uint4 m = tmp[i];
      for (int dy = -2; dy <= 2; ++dy)
        if (dy != 0 && y + dy >= 0 && y + dy < p.H) m = max4(m, tmp[i + dy * p.W]);
      cur[i] = m;   // safe: the column pass only reads tmp
      *reinterpret_cast<uint4*>(base + static_cast<size_t>(i) * p.pitch + (r + 1) * p.C) = m;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// nearest x2 upsample (graph chains 191, 212: out[i] = in[i / 2]) into a channel slice of the concat buffer.
// ------------------------------------------------------------------------------------------------
struct UpParams {
  const __half* in; int in_pitch;
  __half* out; int out_pitch;
  int B, H, W, C;  // input dims
};

// Input-centric: a thread loads one 16-byte channel group of one input pixel and stores it to the four output pixels it
// covers.  grid = (ceil(W * C/8 / 256), H, B): 32-bit index math only (the first version decoded a flat 64-bit index with
// four 64-bit divisions per 16 bytes and ran at half the bandwidth the copy needs).
__global__ void __launch_bounds__(256) upsample2x_kernel(const UpParams p) {
  XR_PDL_ENTRY();
  const int cg = p.C / 8;
  const int col = blockIdx.x * 256 + threadIdx.x;
  if (col >= p.W * cg) return;
  const int x = col / cg, g = col - x * cg;
  const int y = blockIdx.y, b = blockIdx.z;
  const uint4 v = *reinterpret_cast<const uint4*>(p.in + ((static_cast<size_t>(b) * p.H + y) * p.W + x) * p.in_pitch + g * 8);
  const int Wo = 2 * p.W;
  __half* o = p.out + ((static_cast<size_t>(b) * 2 * p.H + 2 * y) * Wo + 2 * x) * p.out_pitch + g * 8;
  *reinterpret_cast<uint4*>(o) = v;
  *reinterpret_cast<uint4*>(o + p.out_pitch) = v;
  o += static_cast<size_t>(Wo) * p.out_pitch;
  *reinterpret_cast<uint4*>(o) = v;
  *reinterpret_cast<uint4*>(o + p.out_pitch) = v;
}

// ------------------------------------------------------------------------------------------------
// C2PSA attention (graph chains 160-168): per (image, head): S = Q^T K * scale, softmax over keys, O = V A^T.
// qkv is the NHWC output of the qkv 1x1 conv: per token, head h occupies channels [h*(2kd+hd), (h+1)*(2kd+hd)):
// kd query dims, kd key dims, hd value dims.  One thread per query, K and V of the head staged in shared memory,
// online softmax in fp32.  kd = 32, hd = 64.
// ------------------------------------------------------------------------------------------------
struct AttnParams {
  const __half* qkv; int qkv_pitch;
  __half* out; int out_pitch;    // [B,N,heads*hd]
  int B, N, heads;
  float scale;
  // fused positional encoding (graph chains 169-170: x = attention(v) + pe(v), pe = depthwise 3x3 + bias on the V map):
  // pe_w [9][heads*hd] fp32 (tap-major, as DwParams::w), pe_b [heads*hd], map width W (N = H * W).  nullptr: attention only.
  const float* pe_w; const float* pe_b; int W;
};

constexpr int ATT_KD = 32, ATT_HD = 64;
constexpr int ATT_KSTRIDE = 40;   // halves per K row in smem (80 B: conflict-free 32-bit fragment loads)
constexpr int ATT_VSTRIDE = 72;   // halves per V row in smem (144 B: conflict-free ldmatrix)
constexpr int ATT_CHUNK = 80;     // keys per online-softmax step (400 = 5 x 80)

__device__ __forceinline__ void hmma_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

// Two CTAs per (image, head), 13 warps each; one warp per 16 queries (N must be a multiple of 16 and of ATT_CHUNK).  S = Q K^T and
// O = P V run on the tensor cores (mma.sync m16n8k16, fp32 accumulate) with a register-level online softmax: the
// accumulator fragment of S is re-used directly as the A fragment of P V.  The whole working set of a head is 77 KB
// of shared memory and 0.06 GFLOP per frame -- too small for a TMEM/tcgen05 pipeline to pay off.
// With pe_w set, the block's positional encoding rides in the epilogue: the head's V map is already in shared memory, so
// pe(v) = depthwise 3x3 (zero padding) + bias is nine shared-memory reads per output next to the normalised attention
// output -- the separate depthwise launch (15 us for 0.06 GFLOP) and the round trip of the attention output are gone.
__global__ void __launch_bounds__(416) attention_kernel(const AttnParams p) {
  XR_PDL_ENTRY();
  extern __shared__ __align__(16) uint8_t att_smem[];
  __shared__ float pe_ws[9][ATT_HD];
  __shared__ float pe_bs[ATT_HD];
  __half* ks = reinterpret_cast<__half*>(att_smem);                       // [N][ATT_KSTRIDE]
  __half* vs = ks + static_cast<size_t>(p.N) * ATT_KSTRIDE;               // [N][ATT_VSTRIDE]
  const int bh = blockIdx.x;
  const int h = bh % p.heads;
  const int b = bh / p.heads;
  const int per_head = 2 * ATT_KD + ATT_HD;
  if (p.pe_w) {                                                           // weights are constants: before the PDL wait would do too
    const int C = p.heads * ATT_HD;
    for (int i = threadIdx.x; i < 10 * ATT_HD; i += blockDim.x) {
      const int t = i / ATT_HD, c = i - t * ATT_HD;
      if (t < 9) pe_ws[t][c] = p.pe_w[t * C + h * ATT_HD + c];
      else pe_bs[c] = p.pe_b[h * ATT_HD + c];
    }
  }
  const __half* base = p.qkv + static_cast<size_t>(b) * p.N * p.qkv_pitch + h * per_head;
  for (int i = threadIdx.x; i < p.N * 12; i += blockDim.x) {
    const int tok = i / 12, part = i - tok * 12;
    const __half* src = base + static_cast<size_t>(tok) * p.qkv_pitch + ATT_KD + part * 8;
    const uint32_t dst = part < 4 ? smem_u32(ks + tok * ATT_KSTRIDE + part * 8) : smem_u32(vs + tok * ATT_VSTRIDE + (part - 4) * 8);
    cp_async16(dst, src, 16);
  }
  cp_async_commit();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int q0 = (blockIdx.y * (blockDim.x >> 5) + warp) * 16;
  const bool active = q0 < p.N;     // the last CTA of a head may have idle warps (they still helped stage K / V)
  // Q fragments (pre-scaled): 2 k-steps x 4 registers
  uint32_t qa[2][4];
  {
    const __half2 sc = __float2half2_rn(p.scale);
    const int qs = active ? q0 : 0;
    const __half* qr0 = base + static_cast<size_t>(qs + g) * p.qkv_pitch;
    const __half* qr1 = base + static_cast<size_t>(qs + g + 8) * p.qkv_pitch;
#pragma unroll
    for (int kk = 0; kk < 2; ++kk) {
      const int c = kk * 16 + 2 * t;
      __half2 v0 = __hmul2(*reinterpret_cast<const __half2*>(qr0 + c), sc);
      __half2 v1 = __hmul2(*reinterpret_cast<const __half2*>(qr1 + c), sc);
      __half2 v2 = __hmul2(*reinterpret_cast<const __half2*>(qr0 + c + 8), sc);
      __half2 v3 = __hmul2(*reinterpret_cast<const __half2*>(qr1 + c + 8), sc);
      qa[kk][0] = *reinterpret_cast<uint32_t*>(&v0);
      qa[kk][1] = *reinterpret_cast<uint32_t*>(&v1);
      qa[kk][2] = *reinterpret_cast<uint32_t*>(&v2);
      qa[kk][3] = *reinterpret_cast<uint32_t*>(&v3);
    }
  }
  cp_async_wait<0>();
  __syncthreads();
  if (!active) return;

  float o[8][4];
#pragma unroll
  for (int n = 0; n < 8; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;
  float mx0 = -1e30f, mx1 = -1e30f, sum0 = 0.f, sum1 = 0.f;
  const float LOG2E = 1.4426950408889634f;

  for (int k0 = 0; k0 < p.N; k0 += ATT_CHUNK) {
    float s[ATT_CHUNK / 8][4];
#pragma unroll
    for (int n = 0; n < ATT_CHUNK / 8; ++n) {
      s[n][0] = s[n][1] = s[n][2] = s[n][3] = 0.f;
      const __half* kr = ks + (k0 + n * 8 + g) * ATT_KSTRIDE + 2 * t;
#pragma unroll
      for (int kk = 0; kk < 2; ++kk) {
        const uint32_t b0 = *reinterpret_cast<const uint32_t*>(kr + kk * 16);
        const uint32_t b1 = *reinterpret_cast<const uint32_t*>(kr + kk * 16 + 8);
        hmma_16816(s[n], qa[kk], b0, b1);
      }
    }
    // online softmax over this chunk (rows g and g+8 of the warp's 16 queries)
    float cm0 = -1e30f, cm1 = -1e30f;
#pragma unroll
    for (int n = 0; n < ATT_CHUNK / 8; ++n) {
      cm0 = fmaxf(cm0, fmaxf(s[n][0], s[n][1]));
      cm1 = fmaxf(cm1, fmaxf(s[n][2], s[n][3]));
    }
    cm0 = fmaxf(cm0, __shfl_xor_sync(0xffffffffu, cm0, 1)); cm0 = fmaxf(cm0, __shfl_xor_sync(0xffffffffu, cm0, 2));
    cm1 = fmaxf(cm1, __shfl_xor_sync(0xffffffffu, cm1, 1)); cm1 = fmaxf(cm1, __shfl_xor_sync(0xffffffffu, cm1, 2));
    const float nm0 = fmaxf(mx0, cm0), nm1 = fmaxf(mx1, cm1);
    const float corr0 = exp2f((mx0 - nm0) * LOG2E), corr1 = exp2f((mx1 - nm1) * LOG2E);
    mx0 = nm0; mx1 = nm1;
    float ps0 = 0.f, ps1 = 0.f;
#pragma unroll
    for (int n = 0; n < ATT_CHUNK / 8; ++n) {
      s[n][0] = exp2f((s[n][0] - nm0) * LOG2E); s[n][1] = exp2f((s[n][1] - nm0) * LOG2E);
      s[n][2] = exp2f((s[n][2] - nm1) * LOG2E); s[n][3] = exp2f((s[n][3] - nm1) * LOG2E);
      ps0 += s[n][0] + s[n][1];
      ps1 += s[n][2] + s[n][3];
    }
    sum0 = sum0 * corr0 + ps0;
    sum1 = sum1 * corr1 + ps1;
#pragma unroll
    for (int n = 0; n < 8; ++n) {
      o[n][0] *= corr0; o[n][1] *= corr0;
      o[n][2] *= corr1; o[n][3] *= corr1;
    }
    // O += P V : 16 keys per k-step; the S accumulator fragments of two adjacent key tiles form the A fragment
#pragma unroll
    for (int kk = 0; kk < ATT_CHUNK / 16; ++kk) {
      uint32_t pa[4];
      pa[0] = pack_h2(s[2 * kk][0], s[2 * kk][1]);
      pa[1] = pack_h2(s[2 * kk][2], s[2 * kk][3]);
      pa[2] = pack_h2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
      pa[3] = pack_h2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
      const int key = k0 + kk * 16 + (lane & 15);
#pragma unroll
      for (int n2 = 0; n2 < 4; ++n2) {          // two 8-wide dim tiles per ldmatrix.x4
        uint32_t vb[4];
        ldmatrix_x4_trans(vb, smem_u32(vs + key * ATT_VSTRIDE + n2 * 16 + (lane >> 4) * 8));
        hmma_16816(o[2 * n2], pa, vb[0], vb[1]);
        hmma_16816(o[2 * n2 + 1], pa, vb[2], vb[3]);
      }
    }
  }
  sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1); sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
  sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1); sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
  const float inv0 = 1.0f / sum0, inv1 = 1.0f / sum1;
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    o[n][0] *= inv0; o[n][1] *= inv0;
    o[n][2] *= inv1; o[n][3] *= inv1;
  }
  if (p.pe_w) {
    // + pe(v): rows q0 + g and q0 + g + 8 of the map, channels n * 8 + 2t, + 1; fp32 accumulation in tap order
    const int H = p.N / p.W;
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
      const int tok = q0 + g + 8 * rr;
      const int y = tok / p.W, x = tok - y * p.W;
      float acc[8][2];
#pragma unroll
      for (int n = 0; n < 8; ++n) {
        acc[n][0] = pe_bs[n * 8 + 2 * t];
        acc[n][1] = pe_bs[n * 8 + 2 * t + 1];
      }
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        const int yy = y + tap / 3 - 1, xx = x + tap % 3 - 1;
        if (yy < 0 || yy >= H || xx < 0 || xx >= p.W) continue;
        const __half* vr = vs + (yy * p.W + xx) * ATT_VSTRIDE + 2 * t;
#pragma unroll
        for (int n = 0; n < 8; ++n) {
          const float2 v2 = __half22float2(*reinterpret_cast<const __half2*>(vr + n * 8));
          acc[n][0] = fmaf(pe_ws[tap][n * 8 + 2 * t], v2.x, acc[n][0]);
          acc[n][1] = fmaf(pe_ws[tap][n * 8 + 2 * t + 1], v2.y, acc[n][1]);
        }
      }
#pragma unroll
      for (int n = 0; n < 8; ++n) {
        o[n][2 * rr] += acc[n][0];
        o[n][2 * rr + 1] += acc[n][1];
      }
    }
  }
  __half* o0 = p.out + (static_cast<size_t>(b) * p.N + q0 + g) * p.out_pitch + h * ATT_HD + 2 * t;
  __half* o1 = o0 + static_cast<size_t>(8) * p.out_pitch;
#pragma unroll
  for (int n = 0; n < 8; ++n) {
    *reinterpret_cast<uint32_t*>(o0 + n * 8) = pack_h2(o[n][0], o[n][1]);
    *reinterpret_cast<uint32_t*>(o1 + n * 8) = pack_h2(o[n][2], o[n][3]);
  }
}

// ------------------------------------------------------------------------------------------------
// Stem on the tensor cores (↔ TextureConverter.ToTensor + graph chain 002, IEExecutor.cs:370-371): 3x3 stride-2 conv
// straight from the uint8 frame, + bias + SiLU -> fp16 NHWC.  K = 27 is too thin for a tcgen05 pipeline (one UMMA of
// K = 16 per 2 KB of output), so this is a register-level implicit GEMM on mma.sync m16n8k16: the K axis is laid out
// as (tap, RGBX) = 12 x 4 = 48 (taps 9..11 and channel X carry zero weights), so an A-fragment register is exactly two
// bytes of ONE pixel word of the staged RGBX patch -- one LDS + PRMT + HSUB2 ("0x6400 | byte" is the fp16 1024 + byte).
// Bytes stay exact integers in fp16; the 1/255 of ToTensor is applied to the fp32 accumulator.
// Block = 8 output rows x 32 output columns (one row per warp, two 16-pixel m-tiles); NT = Cout / 8 n-tiles.
// ------------------------------------------------------------------------------------------------
struct StemMmaParams {
  const uint8_t* src; int stride_bytes, bpp;   // [B,H,W,bpp] uint8, rows 4-byte aligned
  __half* out; int out_pitch;                  // [B,H/2,W/2,Cout]
  const __half* w16;                           // stem_mma_kernel: [Cout][12 taps][4] fp16, zero padded; stem_rows_kernel: [Cout][3][16]
  const float* bias;                           // [Cout]
  int B, H, W;
  float in_scale;                              // 1/255
  int flip;                                    // rows stored bottom-up (image row y lives at memory row H-1-y)
};

constexpr int STEM_PW = 65, STEM_PH = 17, STEM_RAW_WORDS = 56, STEM_RAW_CHUNKS = 14;

template <int NT>
__global__ void __launch_bounds__(256) stem_mma_kernel(const StemMmaParams p) {
  XR_PDL_ENTRY();
  __shared__ __align__(16) uint32_t raw[STEM_PH][STEM_RAW_WORDS];
  __shared__ uint32_t patch[STEM_PH * STEM_PW];
  const int Ho = p.H >> 1, Wo = p.W >> 1;
  const int ox0 = blockIdx.x * 32, oy0 = blockIdx.y * 8, b = blockIdx.z;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const uint8_t* img = p.src + static_cast<size_t>(b) * p.H * p.stride_bytes;
  const int ix0 = 2 * ox0 - 1, iy0 = 2 * oy0 - 1;
  const int c_lo = max(ix0, 0), c_hi = min(ix0 + STEM_PW - 1, p.W - 1);
  if (p.bpp == 4) {
    for (int i = tid; i < STEM_PH * STEM_PW; i += 256) {
      const int r = i / STEM_PW, c = i - r * STEM_PW;
      const int iy = iy0 + r, ix = ix0 + c;
      uint32_t v = 0;
      if (iy >= 0 && iy < p.H && ix >= 0 && ix < p.W)
        v = *reinterpret_cast<const uint32_t*>(img + static_cast<size_t>(p.flip ? p.H - 1 - iy : iy) * p.stride_bytes + ix * 4) & 0x00FFFFFFu;
      patch[i] = v;
    }
  } else {
    // pass 1: the bytes [3 c_lo, 3 (c_hi + 1)) of each patch row into shared memory
    const bool wide = ((reinterpret_cast<uintptr_t>(p.src) | static_cast<uintptr_t>(p.stride_bytes)) & 15) == 0 &&
                      ((p.W * 3) & 15) == 0;
    const int a0 = wide ? (c_lo * 3) & ~15 : (c_lo * 3) & ~3;
    if (wide) {
      // 16-byte path (the normal case: 640-wide frames, 16-byte aligned rows): ONE load per thread covers the 17 x 224
      // bytes of the patch -- staging latency, not arithmetic, bounded the previous 4-byte version
      if (tid < STEM_PH * STEM_RAW_CHUNKS) {
        const int r = tid / STEM_RAW_CHUNKS, j = tid - r * STEM_RAW_CHUNKS;
        const int iy = iy0 + r;
        const int off = a0 + 16 * j;
        if (iy >= 0 && iy < p.H && off < p.W * 3 && off < (c_hi + 1) * 3)
          *reinterpret_cast<uint4*>(&raw[r][4 * j]) =
              *reinterpret_cast<const uint4*>(img + static_cast<size_t>(p.flip ? p.H - 1 - iy : iy) * p.stride_bytes + off);
      }
    } else {
      const int nwords = ((c_hi + 1) * 3 - a0 + 3) >> 2;
      for (int i = tid; i < STEM_PH * STEM_RAW_WORDS; i += 256) {
        const int r = i / STEM_RAW_WORDS, j = i - r * STEM_RAW_WORDS;
        const int iy = iy0 + r;
        if (j < nwords && iy >= 0 && iy < p.H)
          raw[r][j] = *reinterpret_cast<const uint32_t*>(img + static_cast<size_t>(p.flip ? p.H - 1 - iy : iy) * p.stride_bytes + a0 + 4 * j);
      }
    }
    __syncthreads();
    // pass 2: RGB bytes -> one RGBX word per pixel (zero outside the image = the conv's zero padding).  A thread expands
    // five consecutive pixels (15 bytes): five word loads and one funnel shift per pixel instead of three byte loads.
    static_assert(STEM_PW % 5 == 0 && STEM_PH * (STEM_PW / 5) <= 256, "one (row, 5-pixel group) unit per thread");
    if (tid < STEM_PH * (STEM_PW / 5)) {
      const int r = tid / (STEM_PW / 5), q5 = tid - r * (STEM_PW / 5);
      const int iy = iy0 + r;
      const bool row_ok = iy >= 0 && iy < p.H;
      const int ob = 3 * (ix0 + 5 * q5) - a0;              // byte offset of the group's first pixel in raw[r] (may be < 0)
      const int wi = max(ob, 0) >> 2;
      uint32_t w5[6];
#pragma unroll
      for (int k = 0; k < 6; ++k) w5[k] = (wi + k < STEM_RAW_WORDS) ? raw[r][wi + k] : 0u;
#pragma unroll
      for (int k = 0; k < 5; ++k) {
        const int ix = ix0 + 5 * q5 + k;
        const int rel = ob + 3 * k - 4 * wi;               // >= 0 for every pixel inside the image
        uint32_t v = 0;
        if (row_ok && ix >= 0 && ix < p.W) {
          const int j = rel >> 2;                          // 0..4
          uint32_t lo = w5[0], hi = w5[1];
          if (j == 1) { lo = w5[1]; hi = w5[2]; }
          if (j == 2) { lo = w5[2]; hi = w5[3]; }
          if (j == 3) { lo = w5[3]; hi = w5[4]; }
          if (j == 4) { lo = w5[4]; hi = w5[5]; }
          v = __funnelshift_r(lo, hi, 8 * (rel & 3)) & 0x00FFFFFFu;
        }
        patch[r * STEM_PW + 5 * q5 + k] = v;
      }
    }
  }
  // weights + bias -> registers (constant for the whole block)
  uint32_t wb[3][NT][2];
  int off[3][2];
#pragma unroll
  for (int s = 0; s < 3; ++s)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int tap = 4 * s + 2 * h + (t >> 1);
      const int tc = min(tap, 8);
      off[s][h] = (tc / 3) * STEM_PW + tc % 3;
#pragma unroll
      for (int nt = 0; nt < NT; ++nt)
        wb[s][nt][h] = *reinterpret_cast<const uint32_t*>(p.w16 + ((nt * 8 + g) * 12 + tap) * 4 + (t & 1) * 2);
    }
  float bs[NT][2];
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    bs[nt][0] = p.bias[nt * 8 + 2 * t];
    bs[nt][1] = p.bias[nt * 8 + 2 * t + 1];
  }
  __syncthreads();
  const uint32_t sel = (t & 1) ? 0x4342u : 0x4140u;
  const int oy = oy0 + warp;
  const uint32_t* prow = patch + 2 * warp * STEM_PW;
  auto cvt = [&](uint32_t word) {
    uint32_t v = __byte_perm(word, 0x64646464u, sel);
    const uint32_t k1024 = 0x64006400u;
    __half2 r = __hsub2(*reinterpret_cast<__half2*>(&v), *reinterpret_cast<const __half2*>(&k1024));
    return *reinterpret_cast<uint32_t*>(&r);
  };
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
    float c[NT][4];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) c[nt][0] = c[nt][1] = c[nt][2] = c[nt][3] = 0.f;
    const int px = mt * 16 + g;
#pragma unroll
    for (int s = 0; s < 3; ++s) {
      uint32_t a[4];
      a[0] = cvt(prow[2 * px + off[s][0]]);
      a[1] = cvt(prow[2 * (px + 8) + off[s][0]]);
      a[2] = cvt(prow[2 * px + off[s][1]]);
      a[3] = cvt(prow[2 * (px + 8) + off[s][1]]);
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) hmma_16816(c[nt], a, wb[s][nt][0], wb[s][nt][1]);
    }
    if (oy < Ho) {
      __half* o0 = p.out + ((static_cast<size_t>(b) * Ho + oy) * Wo + ox0 + px) * p.out_pitch + 2 * t;
      __half* o1 = o0 + static_cast<size_t>(8) * p.out_pitch;
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        if (ox0 + px < Wo)
          *reinterpret_cast<uint32_t*>(o0 + nt * 8) =
              silu_pack_h2(fmaf(c[nt][0], p.in_scale, bs[nt][0]), fmaf(c[nt][1], p.in_scale, bs[nt][1]));
        if (ox0 + px + 8 < Wo)
          *reinterpret_cast<uint32_t*>(o1 + nt * 8) =
              silu_pack_h2(fmaf(c[nt][2], p.in_scale, bs[nt][0]), fmaf(c[nt][3], p.in_scale, bs[nt][1]));
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Stem, second version for packed RGB frames (the normal case: 16-byte aligned rows, 3 W a multiple of 16).  The first
// version expanded every RGB pixel of its patch into an RGBX word (~12 instructions per input pixel) and re-loaded its
// weight fragments for 32 pixels per thread: two thirds of its issue slots went into staging (ncu: issue-bound at
// 75 %, 145 us for 64 frames).  Here the K axis is (kernel row, 16 consecutive BYTES of the raw image row):
//   k-step kh covers bytes [6 ox - 3, 6 ox + 13) of image row 2 oy + kh - 1 -- the nine bytes of the three taps
//   (kw, c) = k, k < 9, followed by seven bytes that meet zero weights.
// so the patch is staged as RAW bytes (one 16-byte load, four funnel shifts and one 16-byte shared store per 5.3 pixels;
// the one-byte shift makes every tap window start at an even shared-memory offset) and an A-fragment register is one
// 16-bit shared load + PRMT + HSUB2 ("0x6400 | byte" = fp16 1024 + byte).  Block = 16 output rows x 64 output columns,
// a warp owns two rows = eight 16-pixel M-tiles against the same 12 weight-fragment registers.
// ------------------------------------------------------------------------------------------------
constexpr int STEM2_ROWS = 16, STEM2_COLS = 64;
constexpr int STEM2_PR = 2 * STEM2_ROWS + 1;            // patch rows
constexpr int STEM2_CHUNKS = 26;                        // 16-byte chunks per patch row (13 + 387 bytes -> 416)
constexpr int STEM2_PITCH = STEM2_CHUNKS * 16;          // shared bytes per patch row

template <int NT>
__global__ void __launch_bounds__(256, NT == 2 ? 4 : 3) stem_rows_kernel(const StemMmaParams p) {
  XR_PDL_ENTRY();
  __shared__ __align__(16) uint8_t patch[STEM2_PR * STEM2_PITCH];
  const int Ho = p.H >> 1, Wo = p.W >> 1;
  const int ox0 = blockIdx.x * STEM2_COLS, oy0 = blockIdx.y * STEM2_ROWS, b = blockIdx.z;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const uint8_t* img = p.src + static_cast<size_t>(b) * p.H * p.stride_bytes;
  const int row_bytes = p.W * 3;
  const int a0 = ((6 * ox0 - 3) & ~15);                // global byte of shared byte 1 of every patch row (may be -16)
  // weights + bias -> registers: b0 = W[2t, 2t+1][n], b1 = W[2t+8, 2t+9][n] of k-step kh, n = 8 nt + g
  uint32_t wb[3][NT][2];
  float bs[NT][2];
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
    for (int kh = 0; kh < 3; ++kh) {
      const __half* w = p.w16 + ((nt * 8 + g) * 3 + kh) * 16 + 2 * t;
      wb[kh][nt][0] = *reinterpret_cast<const uint32_t*>(w);
      wb[kh][nt][1] = *reinterpret_cast<const uint32_t*>(w + 8);
    }
    bs[nt][0] = p.bias[nt * 8 + 2 * t];
    bs[nt][1] = p.bias[nt * 8 + 2 * t + 1];
  }
  // stage the raw patch: shared byte s of row r = image byte a0 + s - 1 of row 2 oy0 - 1 + r (zero outside the image).
  // ALL of a thread's loads are issued before the first one is used: as a rolled loop (load, wait, shift, store, next) every
  // thread had one 16-byte load in flight and a quarter of the kernel's stall samples sat on the funnel shift behind it
  // (ncu source page, profiles/r2final_full_stem); four CTAs per SM instead of five pay for the registers.
  {
    constexpr int TOTAL = STEM2_PR * STEM2_CHUNKS, ITERS = (TOTAL + 255) / 256;
    uint4 v[ITERS];
    uint32_t prev[ITERS];
#pragma unroll
    for (int k = 0; k < ITERS; ++k) {
      const int u = tid + 256 * k;
      const int r = u / STEM2_CHUNKS, j = u - r * STEM2_CHUNKS;
      const int iy = 2 * oy0 - 1 + r;
      const int off = a0 + 16 * j;                      // first image byte of the 16-byte load
      v[k] = make_uint4(0u, 0u, 0u, 0u);
      prev[k] = 0u;
      if (u < TOTAL && iy >= 0 && iy < p.H) {
        const uint8_t* rowp = img + static_cast<size_t>(p.flip ? p.H - 1 - iy : iy) * p.stride_bytes;
        if (off >= 0 && off < row_bytes) v[k] = __ldg(reinterpret_cast<const uint4*>(rowp + off));
        if (off >= 4 && off - 4 < row_bytes) prev[k] = __ldg(reinterpret_cast<const uint32_t*>(rowp + off - 4));
      }
    }
#pragma unroll
    for (int k = 0; k < ITERS; ++k) {
      const int u = tid + 256 * k;
      const int r = u / STEM2_CHUNKS, j = u - r * STEM2_CHUNKS;
      uint4 o;
      o.x = __funnelshift_l(prev[k], v[k].x, 8);        // shift the byte stream up by one byte
      o.y = __funnelshift_l(v[k].x, v[k].y, 8);
      o.z = __funnelshift_l(v[k].y, v[k].z, 8);
      o.w = __funnelshift_l(v[k].z, v[k].w, 8);
      if (u < TOTAL) *reinterpret_cast<uint4*>(patch + r * STEM2_PITCH + 16 * j) = o;
    }
  }
  __syncthreads();
  auto cvt = [](uint32_t pair) {                        // two bytes -> two fp16 values
    uint32_t v = __byte_perm(pair, 0x64646464u, 0x4140u);
    const uint32_t k1024 = 0x64006400u;
    __half2 r = __hsub2(*reinterpret_cast<__half2*>(&v), *reinterpret_cast<const __half2*>(&k1024));
    return *reinterpret_cast<uint32_t*>(&r);
  };
  // tap window of tile column c starts at shared byte 6 c + 14 (image byte 6 ox - 3, shifted by a0 and the extra byte)
  const uint32_t lane_off = 6 * g + 14 + 2 * t;
#pragma unroll
  for (int rr = 0; rr < 2; ++rr) {
    const int orow = 2 * warp + rr, oy = oy0 + orow;
    const uint8_t* prow = patch + (2 * orow) * STEM2_PITCH + lane_off;
    const bool row_ok = oy < Ho;
    // this lane's first output pixel of the row (pixel ox0 + g, channels 2t, 2t + 1)
    __half* orow_out = p.out + ((static_cast<size_t>(b) * Ho + (row_ok ? oy : 0)) * Wo + ox0 + g) * p.out_pitch + 2 * t;
#pragma unroll
    for (int mt = 0; mt < STEM2_COLS / 16; ++mt) {
      float c[NT][4];
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) c[nt][0] = c[nt][1] = c[nt][2] = c[nt][3] = 0.f;
#pragma unroll
      for (int kh = 0; kh < 3; ++kh) {
        const uint8_t* q = prow + kh * STEM2_PITCH + 96 * mt;   // 16 pixels x 6 bytes per M-tile
        uint32_t a[4];
        a[0] = cvt(*reinterpret_cast<const uint16_t*>(q));
        a[1] = cvt(*reinterpret_cast<const uint16_t*>(q + 48));      // pixel g + 8
        a[2] = cvt(*reinterpret_cast<const uint16_t*>(q + 8));       // k + 8
        a[3] = cvt(*reinterpret_cast<const uint16_t*>(q + 56));
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) hmma_16816(c[nt], a, wb[kh][nt][0], wb[kh][nt][1]);
      }
      // values first, then plainly predicated stores (an if-block around the SiLU math costs a BSSY / BSYNC pair per store;
      // trading halves between lanes for 8-byte stores measured slower: 102 -> 117 us)
      const int px = ox0 + mt * 16 + g;
      uint32_t v0[NT], v1[NT];
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        v0[nt] = silu_pack_h2(fmaf(c[nt][0], p.in_scale, bs[nt][0]), fmaf(c[nt][1], p.in_scale, bs[nt][1]));
        v1[nt] = silu_pack_h2(fmaf(c[nt][2], p.in_scale, bs[nt][0]), fmaf(c[nt][3], p.in_scale, bs[nt][1]));
      }
      uint32_t* o0 = reinterpret_cast<uint32_t*>(orow_out + static_cast<size_t>(mt * 16) * p.out_pitch);
      uint32_t* o1 = reinterpret_cast<uint32_t*>(orow_out + static_cast<size_t>(mt * 16 + 8) * p.out_pitch);
      const bool ok0 = row_ok && px < Wo, ok1 = row_ok && px + 8 < Wo;
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        if (ok0) o0[nt * 4] = v0[nt];
        if (ok1) o1[nt * 4] = v1[nt];
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// direct convolution on CUDA cores: one thread per output element, fp32 accumulate.  Cross-check path only
// (xrseg_config.conv_impl = XRSEG_CONV_DIRECT); weights fp16 [Cout][k*k][Cin] (or [4 pos][Cout][Cin] transposed).
// ------------------------------------------------------------------------------------------------
struct DirectParams {
  const __half* in; int in_pitch;
  __half* out; int out_pitch;
  const __half* res; int res_pitch;
  const __half* w; const float* bias;
  int B, H, W, Cin, Ho, Wo, Cout, k, stride, pad, act, transposed;
};

__global__ void __launch_bounds__(256) conv_direct_kernel(const DirectParams p) {
  const long total = static_cast<long>(p.B) * p.Ho * p.Wo * p.Cout;
  for (long idx = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long>(gridDim.x) * blockDim.x) {
    const int co = static_cast<int>(idx % p.Cout);
    const long pix = idx / p.Cout;
    const int ow = static_cast<int>(pix % p.Wo);
    const int oh = static_cast<int>((pix / p.Wo) % p.Ho);
    const long b = pix / (static_cast<long>(p.Wo) * p.Ho);
    float acc = p.bias[co];
    if (p.transposed) {
      const int ih = oh >> 1, iw = ow >> 1, pos = (oh & 1) * 2 + (ow & 1);
      const __half* xi = p.in + ((b * p.H + ih) * p.W + iw) * p.in_pitch;
      const __half* wt = p.w + (static_cast<size_t>(pos) * p.Cout + co) * p.Cin;
      for (int ci = 0; ci < p.Cin; ++ci) acc = fmaf(__half2float(xi[ci]), __half2float(wt[ci]), acc);
    } else {
      for (int kh = 0; kh < p.k; ++kh) {
        const int ih = oh * p.stride - p.pad + kh;
        if (ih < 0 || ih >= p.H) continue;
        for (int kw = 0; kw < p.k; ++kw) {
          const int iw = ow * p.stride - p.pad + kw;
          if (iw < 0 || iw >= p.W) continue;
          const __half* xi = p.in + ((b * p.H + ih) * p.W + iw) * p.in_pitch;
          const __half* wt = p.w + (static_cast<size_t>(co) * p.k * p.k + kh * p.k + kw) * p.Cin;
          for (int ci = 0; ci < p.Cin; ci += 2) {
            const float2 xv = __half22float2(*reinterpret_cast<const __half2*>(xi + ci));
            const float2 wv = __half22float2(*reinterpret_cast<const __half2*>(wt + ci));
            acc = fmaf(xv.x, wv.x, acc);
            acc = fmaf(xv.y, wv.y, acc);
          }
        }
      }
    }
    if (p.act) acc = silu_f(acc);
    if (p.res) acc += __half2float(p.res[pix * p.res_pitch + co]);
    p.out[pix * p.out_pitch + co] = __float2half_rn(acc);
  }
}

// ------------------------------------------------------------------------------------------------
// layout converters for the debug / parity entry points
// ------------------------------------------------------------------------------------------------
__global__ void nchw_f32_to_nhwc_f16_kernel(const float* src, __half* dst, int B, int C, int H, int W, int Cpad,
                                            int pitch) {
  const long total = static_cast<long>(B) * H * W * Cpad;
  for (long idx = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(idx % Cpad);
    const long pix = idx / Cpad;
    const int x = static_cast<int>(pix % W);
    const int y = static_cast<int>((pix / W) % H);
    const long b = pix / (static_cast<long>(W) * H);
    const float v = c < C ? src[((b * C + c) * H + y) * W + x] : 0.f;
    dst[pix * pitch + c] = __float2half_rn(v);
  }
}

__global__ void nhwc_f16_to_nchw_f32_kernel(const __half* src, float* dst, int B, int C, int H, int W, int pitch) {
  const long total = static_cast<long>(B) * C * H * W;
  for (long idx = blockIdx.x * static_cast<long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long>(gridDim.x) * blockDim.x) {
    const int x = static_cast<int>(idx % W);
    const int y = static_cast<int>((idx / W) % H);
    const int c = static_cast<int>((idx / (static_cast<long>(W) * H)) % C);
    const long b = idx / (static_cast<long>(W) * H * C);
    dst[idx] = __half2float(src[((b * H + y) * W + x) * pitch + c]);
  }
}

static inline int grid_for(long total, int block = 256, int cap = 148 * 16) {
  long g = (total + block - 1) / block;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

#endif  // __CUDACC__
}  // namespace xrseg
