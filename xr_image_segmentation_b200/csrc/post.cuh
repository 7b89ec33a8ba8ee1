// post.cuh -- the Detect/Segment tail the reference bakes into its graph (IEModelEditorConverter.cs:31-106, graph
// chains 400-416 and 455-498) and the C# box / mask post-processing (IEExecutor.cs:529-559, IEBoxer.cs:37-81,
// IEMasker.cs:82-119,124-196,232-247) as memory-bound CUDA kernels:
//   decode   : 16-bin DFL softmax expectation + anchor/stride decode + 80-class sigmoid max/argmax + score filter
//   nms      : per-frame sort (score desc, index asc) -> IoU bitmask (smem staged) -> greedy reduce
//   gather   : compaction of boxes / labels / coefs over the batch (output_0..2)
//   masks    : coef x proto (32-term fp32 FMA chain) + sigmoid (output_3), fused crop / upsample / threshold variants
// Arithmetic that decides discrete results (IoU test, box predicate, thresholds) uses explicit IEEE intrinsics in a
// fixed order so that it matches oracle/postprocess.py bit for bit on identical inputs.
#pragma once

#include "common.cuh"

namespace xrseg {

constexpr int NUM_ANCHORS_MAX = 8400;
constexpr int NC = 80;            // the COCO class count: decode_filter_kernel is specialised for it
constexpr int NM = 32;
constexpr int PROTO_HW = 160;
constexpr int PROTO_PIX = PROTO_HW * PROTO_HW;

// One feature-map scale feeding the decode: element (b, a_local, c) at ptr + b*bstride + a_local*pitch + c.
template <typename T>
struct ScaleSrc {
  const T* box; long box_bstride; int box_pitch;
  const T* cls; long cls_bstride; int cls_pitch;
  const T* coef; long coef_bstride; int coef_pitch;
  int h, w, a_off;
  float stride;
};

template <typename T>
struct DecodeParams {
  ScaleSrc<T> s[3];
  int B, A;
  int nc;                    // classes; class tensors carry cls_pitch >= nc channels per anchor, the rest is never counted
  float score_thr;
  float logit_floor;         // anchors whose largest class logit is <= this cannot reach score_thr
  float* boxes;              // [B,A,4] cx,cy,w,h  (rows of candidates only; the rest is never read)
  float* scores;             // [B,A]
  int* labels;               // [B,A]
  unsigned long long* keys;  // [B,A] candidate sort keys
  int* cand_count;           // [B]
  int* filt_list;            // [B,A] anchors that survived the logit filter (unordered)
  int* filt_count;           // [B]
};

#ifdef __CUDACC__

__device__ __forceinline__ float ldf(const float* p) { return *p; }
__device__ __forceinline__ float ldf(const __half* p) { return __half2float(*p); }

// 16 consecutive values (64-byte aligned fp32 / 32-byte aligned fp16) with 128-bit loads
__device__ __forceinline__ void load16(const float* p, float (&v)[16]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 f = reinterpret_cast<const float4*>(p)[i];
    v[4 * i] = f.x; v[4 * i + 1] = f.y; v[4 * i + 2] = f.z; v[4 * i + 3] = f.w;
  }
}
__device__ __forceinline__ void load16(const __half* p, float (&v)[16]) {
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const uint4 raw = reinterpret_cast<const uint4*>(p)[i];
    const __half2* h = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = __half22float2(h[j]);
      v[8 * i + 2 * j] = f.x;
      v[8 * i + 2 * j + 1] = f.y;
    }
  }
}

// ---- decode, kernel 1 of 2: the streaming filter ---------------------------------------------------------------------
// Block = 256 consecutive anchors of one frame; every anchor's 80 class logits are read once and reduced to their
// maximum; an anchor whose largest LOGIT is below logit(score_thr) - 0.01 cannot pass the probability test and is
// dropped -- nothing downstream reads non-candidates.  Survivors (1-2 % of the anchors) are appended to the frame's list.
// Loads are warp-coalesced: a warp owns 32 consecutive anchors = one contiguous run of 32*NC logits, lane l reads the
// 16-byte chunks l, l+32, ... of the run and the per-anchor maximum is a segmented reduction through shared memory (a
// thread-per-anchor walk touches 32 different sectors per load instruction and was bound by the load/store unit).
template <typename T>
__global__ void __launch_bounds__(256) decode_filter_kernel(const DecodeParams<T> p) {
  XR_PDL_ENTRY();
  constexpr int EPC = 16 / static_cast<int>(sizeof(T));          // logits per 16-byte chunk
  constexpr int CPA = NC / EPC;                                   // chunks per anchor (10 fp16, 20 fp32)
  __shared__ float s_max[8][32 * CPA];
  __shared__ int s_list[256];
  __shared__ int s_n, s_base;
  const int b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  const int a0 = blockIdx.x * 256 + warp * 32;                    // first anchor of this warp
  const int a = a0 + lane;
  if (a0 < p.A) {
    const int a_last = min(a0 + 31, p.A - 1);
    int si = 0;
    if (a0 >= p.s[1].a_off) si = 1;
    if (a0 >= p.s[2].a_off) si = 2;
    int sl = 0;
    if (a_last >= p.s[1].a_off) sl = 1;
    if (a_last >= p.s[2].a_off) sl = 2;
    float lmax = -3.0e38f;
    if (si == sl && p.s[si].cls_pitch == NC) {
      // coalesced run: anchors a0 .. a_last of scale si
      const ScaleSrc<T>& s = p.s[si];
      const T* run = s.cls + b * s.cls_bstride + static_cast<long>(a0 - s.a_off) * NC;
      const int n_chunks = (a_last - a0 + 1) * CPA;
#pragma unroll
      for (int it = 0; it < CPA; ++it) {
        const int gi = it * 32 + lane;
        float m = -3.0e38f;
        if (gi < n_chunks) {
          const uint4 raw = reinterpret_cast<const uint4*>(run)[gi];
          if (sizeof(T) == 2) {
            const __half2* h = reinterpret_cast<const __half2*>(&raw);
            const __half2 m2 = __hmax2(__hmax2(h[0], h[1]), __hmax2(h[2], h[3]));
            m = fmaxf(__low2float(m2), __high2float(m2));
          } else {
            const float* f = reinterpret_cast<const float*>(&raw);
            m = fmaxf(fmaxf(f[0], f[1]), fmaxf(f[2], f[3]));
          }
        }
        s_max[warp][gi] = m;
      }
      __syncwarp();
      if (a <= a_last) {
#pragma unroll
        for (int k = 0; k < CPA; ++k) lmax = fmaxf(lmax, s_max[warp][lane * CPA + k]);
      }
    } else if (a < p.A) {
      // generic walk (a warp straddling two scales, or a padded class tensor)
      int sa = 0;
      if (a >= p.s[1].a_off) sa = 1;
      if (a >= p.s[2].a_off) sa = 2;
      const ScaleSrc<T>& s = p.s[sa];
      const T* cl = s.cls + b * s.cls_bstride + static_cast<long>(a - s.a_off) * s.cls_pitch;
#pragma unroll
      for (int c0 = 0; c0 < NC; c0 += 16) {
        float l[16];
        load16(cl + c0, l);
#pragma unroll
        for (int k = 0; k < 16; ++k) lmax = fmaxf(lmax, l[k]);
      }
    }
    if (a < p.A && lmax > p.logit_floor) s_list[atomicAdd(&s_n, 1)] = a;
  }
  __syncthreads();
  const int n = s_n;
  if (n == 0) return;
  if (threadIdx.x == 0) s_base = atomicAdd(&p.filt_count[b], n);   // one global atomic per block
  __syncthreads();
  if (static_cast<int>(threadIdx.x) < n) p.filt_list[static_cast<long>(b) * p.A + s_base + threadIdx.x] = s_list[threadIdx.x];
}

// Largest of the first `valid` logits of a 16-byte chunk (all of them when valid >= the chunk's element count).
template <typename T>
__device__ __forceinline__ float chunk_max(const uint4 raw, int valid) {
  constexpr int EPC = 16 / static_cast<int>(sizeof(T));
  if (valid >= EPC) {
    if (sizeof(T) == 2) {
      const __half2* h = reinterpret_cast<const __half2*>(&raw);
      const __half2 m2 = __hmax2(__hmax2(h[0], h[1]), __hmax2(h[2], h[3]));
      return fmaxf(__low2float(m2), __high2float(m2));
    }
    const float* f = reinterpret_cast<const float*>(&raw);
    return fmaxf(fmaxf(f[0], f[1]), fmaxf(f[2], f[3]));
  }
  const T* e = reinterpret_cast<const T*>(&raw);
  float m = -3.0e38f;
#pragma unroll
  for (int k = 0; k < EPC; ++k)
    if (k < valid) m = fmaxf(m, ldf(e + k));
  return m;
}

// Per-thread walk over one anchor's nc logits (a warp whose 32 anchors straddle two scales).
template <typename T>
__device__ __forceinline__ float anchor_max_walk(const DecodeParams<T>& p, int b, int a) {
  int sa = 0;
  if (a >= p.s[1].a_off) sa = 1;
  if (a >= p.s[2].a_off) sa = 2;
  const ScaleSrc<T>& s = p.s[sa];
  const T* cl = s.cls + b * s.cls_bstride + static_cast<long>(a - s.a_off) * s.cls_pitch;
  float m = -3.0e38f;
  for (int c = 0; c < p.nc; ++c) m = fmaxf(m, ldf(cl + c));
  return m;
}

// Appends the block's survivors to the frame's list (one global atomic per block).
__device__ __forceinline__ void filter_append(int* s_list, int& s_n, int& s_base, int* filt_count, int* filt_list, int A, int b) {
  __syncthreads();
  const int n = s_n;
  if (n == 0) return;
  if (threadIdx.x == 0) s_base = atomicAdd(&filt_count[b], n);
  __syncthreads();
  if (static_cast<int>(threadIdx.x) < n) filt_list[static_cast<long>(b) * A + s_base + threadIdx.x] = s_list[threadIdx.x];
}

// Any other class count, rows of at most 32 chunks (cls_pitch <= 256 fp16 / 128 fp32 channels): the same warp-coalesced run
// as decode_filter_kernel with the chunks per anchor (cpa = cls_pitch / chunk) read at run time -- chunk gi of the run is
// chunk gi % cpa of anchor gi / cpa -- and a segment table of 32 * cpa entries per warp in dynamic shared memory.  Only
// channels < nc count: the padding channels of the class tensor hold logit 0 (probability 0.5, above the 0.301 threshold),
// and chunks holding nothing but padding are not read.  cls_pitch is a multiple of the chunk (host-checked).
template <typename T>
__global__ void __launch_bounds__(256) decode_filter_nc_kernel(const DecodeParams<T> p) {
  XR_PDL_ENTRY();
  constexpr int EPC = 16 / static_cast<int>(sizeof(T));
  extern __shared__ float s_seg[];                                // [8 warps][32 * cpa]
  __shared__ int s_list[256];
  __shared__ int s_n, s_base;
  const int b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  const int a0 = blockIdx.x * 256 + warp * 32;
  const int a = a0 + lane;
  if (a0 < p.A) {
    const int a_last = min(a0 + 31, p.A - 1);
    int si = 0;
    if (a0 >= p.s[1].a_off) si = 1;
    if (a0 >= p.s[2].a_off) si = 2;
    int sl = 0;
    if (a_last >= p.s[1].a_off) sl = 1;
    if (a_last >= p.s[2].a_off) sl = 2;
    float lmax = -3.0e38f;
    if (si == sl) {
      const ScaleSrc<T>& s = p.s[si];
      const int cpa = s.cls_pitch / EPC;
      const int used = (p.nc + EPC - 1) / EPC;                    // chunks holding at least one class
      const uint4* run = reinterpret_cast<const uint4*>(s.cls + b * s.cls_bstride + static_cast<long>(a0 - s.a_off) * s.cls_pitch);
      const int n_chunks = (a_last - a0 + 1) * cpa;
      float* seg = s_seg + warp * 32 * cpa;
      for (int gi = lane; gi < n_chunks; gi += 32) {
        const int j = gi / cpa, c = gi - j * cpa;
        seg[gi] = c < used ? chunk_max<T>(run[gi], p.nc - c * EPC) : -3.0e38f;
      }
      __syncwarp();
      if (a <= a_last)
        for (int k = 0; k < cpa; ++k) lmax = fmaxf(lmax, seg[lane * cpa + k]);
    } else if (a < p.A) {
      lmax = anchor_max_walk(p, b, a);
    }
    if (a < p.A && lmax > p.logit_floor) s_list[atomicAdd(&s_n, 1)] = a;
  }
  filter_append(s_list, s_n, s_base, p.filt_count, p.filt_list, p.A, b);
}

// Wide rows (more than 32 chunks: over 256 fp16 classes), where 32 anchors' segment table no longer fits shared memory: a
// warp reads its 32 anchors one row at a time (row j: lane l reads chunks l, l + 32, ... -- one contiguous, coalesced row),
// keeps a per-lane partial maximum per anchor, and a butterfly reduce-scatter (31 shuffles for 32 anchors) leaves anchor
// a0 + l's maximum in lane l.  Rows hold at most 1024 channels (the host checks cls_pitch against it).
template <typename T>
__global__ void __launch_bounds__(256) decode_filter_wide_kernel(const DecodeParams<T> p) {
  XR_PDL_ENTRY();
  constexpr int EPC = 16 / static_cast<int>(sizeof(T));
  constexpr int ROW_ITERS = 1024 / EPC / 32;                      // chunk loads per lane and row at 1024 channels
  __shared__ int s_list[256];
  __shared__ int s_n, s_base;
  const int b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  const int a0 = blockIdx.x * 256 + warp * 32;
  const int a = a0 + lane;
  if (a0 < p.A) {
    const int a_last = min(a0 + 31, p.A - 1);
    int si = 0;
    if (a0 >= p.s[1].a_off) si = 1;
    if (a0 >= p.s[2].a_off) si = 2;
    int sl = 0;
    if (a_last >= p.s[1].a_off) sl = 1;
    if (a_last >= p.s[2].a_off) sl = 2;
    float lmax = -3.0e38f;
    if (si == sl) {
      const ScaleSrc<T>& s = p.s[si];
      const int used = (p.nc + EPC - 1) / EPC;
      const T* base = s.cls + b * s.cls_bstride + static_cast<long>(a0 - s.a_off) * s.cls_pitch;
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const uint4* row = reinterpret_cast<const uint4*>(base + static_cast<long>(min(j, a_last - a0)) * s.cls_pitch);
        float m = -3.0e38f;
#pragma unroll
        for (int k = 0; k < ROW_ITERS; ++k) {
          const int c = lane + 32 * k;
          if (c < used) m = fmaxf(m, chunk_max<T>(row[c], p.nc - c * EPC));
        }
        v[j] = m;
      }
      // reduce-scatter: at step o a lane keeps the half of its anchors whose index has its own bit o, compacted to v[0, o)
#pragma unroll
      for (int o = 16; o >= 1; o >>= 1) {
        const bool upper = (lane & o) != 0;
#pragma unroll
        for (int j = 0; j < o; ++j) {
          const float send = upper ? v[j] : v[j + o];
          const float keep = upper ? v[j + o] : v[j];
          v[j] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, o));
        }
      }
      lmax = v[0];
    } else if (a < p.A) {
      lmax = anchor_max_walk(p, b, a);
    }
    if (a <= a_last && lmax > p.logit_floor) s_list[atomicAdd(&s_n, 1)] = a;
  }
  filter_append(s_list, s_n, s_base, p.filt_count, p.filt_list, p.A, b);
}

// ---- decode, kernel 2 of 2: exact arithmetic on the survivors ----------------------------------------------------------
// One WARP per listed anchor: the nc class sigmoids are spread over the lanes and reduced with the graph's first-maximum
// rule (max probability, lowest index on ties); the four DFL sides go to four lanes, each keeping the sequential 16-bin
// order; lane 0 does the anchor / stride decode.  IEEE intrinsics in the oracle's operation order throughout.
// NCT: the class count when fixed at compile time (80: the COCO models), 0: p.nc.
template <typename T, int NCT>
__global__ void __launch_bounds__(256) decode_exact_kernel(const DecodeParams<T> p) {
  XR_PDL_ENTRY();
  const int nc = p.nc;
  const int b = blockIdx.y;
  const int n_list = min(p.filt_count[b], p.A);
  const int lane = threadIdx.x & 31;
  const int warps = gridDim.x * 8;
  for (int li = blockIdx.x * 8 + (threadIdx.x >> 5); li < n_list; li += warps) {
    const int a = p.filt_list[static_cast<long>(b) * p.A + li];
    int si = 0;
    if (a >= p.s[1].a_off) si = 1;
    if (a >= p.s[2].a_off) si = 2;
    const ScaleSrc<T>& s = p.s[si];
    const int al = a - s.a_off;
    const int gy = al / s.w, gx = al - gy * s.w;
    const float ax = static_cast<float>(gx) + 0.5f, ay = static_cast<float>(gy) + 0.5f;

    // ---- class sigmoid + max / first argmax (chains 416, 464, 471): like the graph, the maximum is taken over the
    // fp32 PROBABILITIES (two different logits can round to the same probability; the first index then wins).
    const T* cl = s.cls + b * s.cls_bstride + static_cast<long>(al) * s.cls_pitch;
    // the DFL logits are fetched together with the class logits (one memory round trip instead of two; 128 bytes per listed
    // anchor are wasted when its exact score misses the threshold)
    const T* bl = s.box + b * s.box_bstride + static_cast<long>(al) * s.box_pitch;
    const float l0 = ldf(bl + lane), l1 = ldf(bl + lane + 32);
    float best = -1.f;
    int besti = 0;
    auto take = [&](int c) {
      const float pr = __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-ldf(cl + c))));
      if (pr > best) {
        best = pr;
        besti = c;
      }
    };
    if constexpr (NCT != 0) {
      for (int c = lane; c < NCT; c += 32) take(c);
    } else {
#pragma unroll 1   // the compiler's partial unroll of the run-time trip count spilled
      for (int c = lane; c < nc; c += 32) take(c);
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
      if (ob > best || (ob == best && oi < besti)) {
        best = ob;
        besti = oi;
      }
    }
    if (!(best > p.score_thr)) continue;     // warp-uniform after the reduction

    // ---- DFL (chains 401-406): softmax over 16 bins, expectation with weights 0..15.  The 64 bins are spread over the
    // warp (lane -> bins lane and lane + 32, i.e. sides lane / 16 and 2 + lane / 16, bin lane % 16): the exponentials and
    // the IEEE divisions run in parallel, the two sums keep the oracle's sequential bin order (every lane of a 16-lane
    // group replays the additions on shuffled operands).  Four lanes doing 16 expf + 16 divisions each took 2.5x longer.
    float m0 = l0, m1 = l1;
#pragma unroll
    for (int o = 8; o >= 1; o >>= 1) {
      m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, o));
      m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, o));
    }
    const float e0 = expf(__fsub_rn(l0, m0)), e1 = expf(__fsub_rn(l1, m1));
    const int grp = lane & 16;
    float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      sum0 = __fadd_rn(sum0, __shfl_sync(0xffffffffu, e0, grp + k));
      sum1 = __fadd_rn(sum1, __shfl_sync(0xffffffffu, e1, grp + k));
    }
    const float kf = static_cast<float>(lane & 15);
    const float q0 = __fmul_rn(__fdiv_rn(e0, sum0), kf), q1 = __fmul_rn(__fdiv_rn(e1, sum1), kf);
    float x0 = 0.f, x1e = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      x0 = __fadd_rn(x0, __shfl_sync(0xffffffffu, q0, grp + k));
      x1e = __fadd_rn(x1e, __shfl_sync(0xffffffffu, q1, grp + k));
    }
    const float d0 = __shfl_sync(0xffffffffu, x0, 0), d1 = __shfl_sync(0xffffffffu, x0, 16);
    const float d2 = __shfl_sync(0xffffffffu, x1e, 0), d3 = __shfl_sync(0xffffffffu, x1e, 16);
    if (lane != 0) continue;
    // chains 407-415
    const float x1 = __fsub_rn(ax, d0), y1 = __fsub_rn(ay, d1);
    const float x2 = __fadd_rn(ax, d2), y2 = __fadd_rn(ay, d3);
    const float cx = __fmul_rn(__fmul_rn(__fadd_rn(x1, x2), 0.5f), s.stride);
    const float cy = __fmul_rn(__fmul_rn(__fadd_rn(y1, y2), 0.5f), s.stride);
    const float bw = __fmul_rn(__fsub_rn(x2, x1), s.stride);
    const float bh = __fmul_rn(__fsub_rn(y2, y1), s.stride);

    const long o = static_cast<long>(b) * p.A + a;
    reinterpret_cast<float4*>(p.boxes)[o] = make_float4(cx, cy, bw, bh);
    p.scores[o] = best;
    p.labels[o] = besti;
    const int slot = atomicAdd(&p.cand_count[b], 1);
    const unsigned long long key =
        (static_cast<unsigned long long>(0xFFFFFFFFu - __float_as_uint(best)) << 32) | static_cast<unsigned>(a);
    p.keys[static_cast<long>(b) * p.A + slot] = key;
  }
}

// Candidate keys straight from caller-provided scores (xrseg_debug_nms).
__global__ void scores_to_keys_kernel(const float* scores, int B, int A, float thr, unsigned long long* keys,
                                      int* cand_count) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (a >= A) return;
  const float s = scores[static_cast<long>(b) * A + a];
  if (s > thr) {
    const int slot = atomicAdd(&cand_count[b], 1);
    keys[static_cast<long>(b) * A + slot] =
        (static_cast<unsigned long long>(0xFFFFFFFFu - __float_as_uint(s)) << 32) | static_cast<unsigned>(a);
  }
}

// ------------------------------------------------------------------------------------------------
// sort: one block per frame, bitonic sort of up to 16384 keys in shared memory; writes the first
// min(count, max_cand) candidates: anchor index + corner box (x1,y1,x2,y2 = cx -/+ w*0.5 ..., chain 459).
// ------------------------------------------------------------------------------------------------
struct SortParams {
  const unsigned long long* keys;  // [B,A]
  const int* cand_count;           // [B]
  const float* boxes;              // [B,A,4] cxcywh  (or corners when corners_given)
  int corners_given;
  int A, max_cand;
  int* sorted_idx;                 // [B,max_cand]
  float4* sorted_corners;          // [B,max_cand]
  int* n_cand;                     // [B] = min(count, max_cand)
  int* overflow;                   // [1] bit 0 set when count > max_cand (bit 1: nms_reduce, kept > max_det)
};

__global__ void __launch_bounds__(1024) nms_sort_kernel(const SortParams p) {
  XR_PDL_ENTRY();
  extern __shared__ unsigned long long skeys[];
  const int b = blockIdx.x;
  const int cnt = min(p.cand_count[b], p.A);
  int n2 = 1;
  while (n2 < cnt) n2 <<= 1;
  for (int i = threadIdx.x; i < n2; i += blockDim.x)
    skeys[i] = i < cnt ? p.keys[static_cast<long>(b) * p.A + i] : 0xFFFFFFFFFFFFFFFFull;
  __syncthreads();
  for (int k = 2; k <= n2; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < n2; i += blockDim.x) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const unsigned long long x = skeys[i], y = skeys[ixj];
          const bool up = (i & k) == 0;
          if ((x > y) == up) {
            skeys[i] = y;
            skeys[ixj] = x;
          }
        }
      }
      __syncthreads();
    }
  const int n = min(cnt, p.max_cand);
  if (threadIdx.x == 0) {
    p.n_cand[b] = n;
    if (cnt > p.max_cand) atomicOr(p.overflow, 1);
  }
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int a = static_cast<int>(skeys[i] & 0xFFFFFFFFull);
    p.sorted_idx[static_cast<long>(b) * p.max_cand + i] = a;
    const float4 bx = reinterpret_cast<const float4*>(p.boxes)[static_cast<long>(b) * p.A + a];
    float4 c;
    if (p.corners_given) {
      c = bx;
    } else {
      const float hw = __fmul_rn(bx.z, 0.5f), hh = __fmul_rn(bx.w, 0.5f);
      c = make_float4(__fsub_rn(bx.x, hw), __fsub_rn(bx.y, hh), __fadd_rn(bx.x, hw), __fadd_rn(bx.y, hh));
    }
    p.sorted_corners[static_cast<long>(b) * p.max_cand + i] = c;
  }
}

// IoU exactly as oracle/postprocess.py::iou_f32 (one rounding per operation, no FMA).
__device__ __forceinline__ bool iou_gt(const float4 a, const float4 b, float thr) {
  const float iw = fmaxf(0.f, __fsub_rn(fminf(a.z, b.z), fmaxf(a.x, b.x)));
  const float ih = fmaxf(0.f, __fsub_rn(fminf(a.w, b.w), fmaxf(a.y, b.y)));
  const float inter = __fmul_rn(iw, ih);
  if (inter <= 0.f && thr >= 0.f) return false;   // disjoint boxes: 0 / union (or 0 / 0 = NaN) is never > thr -- same answer, no division
  const float area_a = __fmul_rn(__fsub_rn(a.z, a.x), __fsub_rn(a.w, a.y));
  const float area_b = __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));
  const float uni = __fsub_rn(__fadd_rn(area_a, area_b), inter);
  return __fdiv_rn(inter, uni) > thr;
}

// ------------------------------------------------------------------------------------------------
// bitmask: block (rb, frame), 64 threads, loops over the column blocks cb >= rb.  Row i = rb*64 + t against columns
// cb*64..+63 staged in smem;
// bit j is set when column candidate (cb*64 + j) comes later in the order and overlaps row i by more than thr.
// ------------------------------------------------------------------------------------------------
struct MaskBitsParams {
  const float4* sorted_corners;  // [B,max_cand]
  const int* n_cand;
  int max_cand, words;           // words = ceil(max_cand / 64)
  float iou_thr;
  unsigned long long* mask;      // [B,max_cand,words]
};

__global__ void __launch_bounds__(256) nms_bitmask_kernel(const MaskBitsParams p) {
  XR_PDL_ENTRY();
  const int rb = blockIdx.x, b = blockIdx.y;
  const int n = p.n_cand[b];
  if (rb * 64 >= n) return;
  __shared__ float4 cols[64];
  __shared__ unsigned long long part[4][64];
  // 256 threads: row t of the block against a quarter (16 columns) of each 64-column tile -- the per-thread chain of
  // exact divisions is what bounds this latency-bound kernel (~100 candidates per frame), so it is split four ways
  const int t = threadIdx.x & 63, s = threadIdx.x >> 6;
  const int i = rb * 64 + t;
  const float4 me = p.sorted_corners[static_cast<long>(b) * p.max_cand + min(i, n - 1)];
  const int nw = (n + 63) >> 6;
  for (int cb = rb; cb < nw; ++cb) {
    const int cj = cb * 64 + t;
    __syncthreads();
    if (s == 0 && cj < n) cols[t] = p.sorted_corners[static_cast<long>(b) * p.max_cand + cj];
    __syncthreads();
    unsigned long long bits = 0;
    if (i < n) {
      const int jn = min(64, n - cb * 64);
      const int j1 = min(jn, s * 16 + 16);
      for (int j = s * 16; j < j1; ++j) {
        const int gj = cb * 64 + j;
        if (gj > i && iou_gt(me, cols[j], p.iou_thr)) bits |= 1ull << j;
      }
    }
    part[s][t] = bits;
    __syncthreads();
    if (s == 0 && i < n)
      p.mask[(static_cast<long>(b) * p.max_cand + i) * p.words + cb] = part[0][t] | part[1][t] | part[2][t] | part[3][t];
  }
}

// ------------------------------------------------------------------------------------------------
// reduce: one block (128 threads) per frame.  Chunks of 64 candidate rows are staged in shared memory, warp 0
// resolves them in order: candidate i is kept unless an earlier kept candidate set its bit.
// ------------------------------------------------------------------------------------------------
struct ReduceParams {
  const unsigned long long* mask;
  const int* n_cand;
  const int* sorted_idx;
  int max_cand, words, max_det;
  int* keep_idx;   // [B,max_det] anchor indices in selection order
  int* keep_n;     // [B]
  int* overflow;
  // exclusive scan of keep_n over the frames [0, scan_upto) of the run -> offsets[scan_upto + 1], done by the block that
  // finishes last (ticket counter `done`, left at zero again): replaces a separate one-thread launch
  const int* keep_n_all; int* offsets; int* done; int scan_upto;
};

// One warp resolves a frame, 64 candidates (one bitmask row block) at a time; the other three warps only help to stage
// the next block.  State lives in registers: lane l holds the "removed" words l, l + 32, ... (NMS_RW words cover 8448
// candidates).  Per block: (1) the 64 x 64 diagonal word decides the block's own keepers in a register-only loop -- the
// 64 diagonal words are broadcast loads that do not depend on the loop-carried word, so the chain per row is one
// shift / test / OR; (2) the keepers' rows are OR-ed into the later words, lanes in parallel, rows by find-first-set;
// (3) kept indices are written with a popcount prefix.  The next block's rows are copied with cp.async meanwhile.
// (The first version re-read the removed word, the kept counter and the row from shared memory for every candidate:
// ~480 cycles per candidate, 215 us for the 854 candidates of the post-processing stress configuration.)
template <int NMS_RW, int NBUF>   // removed words per lane: 1 covers 2048 candidates (the default cap), 5 all 8400 anchors; NBUF-deep row ring
__global__ void __launch_bounds__(128) nms_reduce_kernel(const ReduceParams p) {
  XR_PDL_ENTRY();
  extern __shared__ unsigned long long rsm[];  // NBUF buffers of 64 rows x words
  const int b = blockIdx.x;
  const int n = p.n_cand[b];
  const int nw = (n + 63) / 64;
  const int lane = threadIdx.x & 31;
  const unsigned long long* gmask = p.mask + static_cast<long>(b) * p.max_cand * p.words;
  auto stage = [&](int blk) {                   // rows [64 blk, 64 blk + 64) x words [blk, nw) -> buffer blk % NBUF
    unsigned long long* dst = rsm + static_cast<size_t>(blk % NBUF) * 64 * p.words;
    const int rows = blk < nw ? min(64, n - 64 * blk) : 0, span = nw - blk;   // past the end: an empty group keeps the count uniform
    for (int i = threadIdx.x; i < rows * span; i += blockDim.x) {
      const int r = i / span, w = blk + i - r * span;
      const unsigned long long* src = gmask + static_cast<long>(64 * blk + r) * p.words + w;
      asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst + r * p.words + w)), "l"(src) : "memory");
    }
    cp_async_commit();
  };
  unsigned long long remv[NMS_RW];
#pragma unroll
  for (int j = 0; j < NMS_RW; ++j) remv[j] = 0ull;
  int kept = 0;
  for (int k = 0; k < NBUF - 1; ++k) stage(k);
  for (int blk = 0; blk < nw; ++blk) {
    cp_async_wait<NBUF - 2>();                  // groups are committed in block order: block blk has landed
    __syncthreads();                            // ... for every thread's copies; the buffer of block blk - 1 is free again
    stage(blk + NBUF - 1);
    if (threadIdx.x < 32) {
      const unsigned long long* chunk = rsm + static_cast<size_t>(blk % NBUF) * 64 * p.words;
      const int rows = min(64, n - 64 * blk);
      unsigned long long own = 0ull;            // removed word of this block
#pragma unroll
      for (int j = 0; j < NMS_RW; ++j)
        if ((blk >> 5) == j) own = remv[j];
      unsigned long long cur = __shfl_sync(0xffffffffu, own, blk & 31);
      // anchor ids of this lane's two rows: fetched now, used after the decision loop (hides the global latency)
      const int* sidx = p.sorted_idx + static_cast<long>(b) * p.max_cand + 64 * blk;
      const int id_lo = lane < rows ? sidx[lane] : 0, id_hi = lane + 32 < rows ? sidx[lane + 32] : 0;
      unsigned long long keepmask = 0ull;
      const unsigned long long* diag = chunk + blk;   // every lane reads the same word: one broadcast load per row, independent
#pragma unroll                                      // of the loop-carried `cur`, so the loads run ahead of the decision chain
      for (int r = 0; r < 64; ++r) {             // (fully unrolled: shifts by immediates)
        const unsigned long long d = diag[r * p.words];
        const bool take = r < rows && !((cur >> r) & 1ull);     // branch-free: a branch would sink the load under it and
        keepmask |= take ? (1ull << r) : 0ull;                  // put a shared-memory round trip into every step of the chain
        cur |= take ? d : 0ull;
      }
      // kept indices in selection order
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int r = lane + 32 * half;
        if ((keepmask >> r) & 1ull) {
          const int k = kept + __popcll(keepmask & ((1ull << r) - 1ull));
          if (k < p.max_det) p.keep_idx[static_cast<long>(b) * p.max_det + k] = half ? id_hi : id_lo;
          else if (k == p.max_det) atomicOr(p.overflow, 2);
        }
      }
      kept += __popcll(keepmask);
      // keepers' rows -> later removed words (word blk itself is final after this block): predicated, independent loads
#pragma unroll
      for (int j = 0; j < NMS_RW; ++j) {
        const int w = lane + 32 * j;
        if (w > blk && w < nw) {
          unsigned long long acc = 0ull;
#pragma unroll
          for (int r = 0; r < 64; ++r) {
            const unsigned long long row = chunk[r * p.words + w];   // rows past `rows` hold stale words: masked by keepmask
            acc |= ((keepmask >> r) & 1ull) ? row : 0ull;
          }
          remv[j] |= acc;
        }
      }
    }
  }
  __shared__ int s_last;
  if (threadIdx.x == 0) {
    p.keep_n[b] = min(kept, p.max_det);
    __threadfence();
    const int ticket = atomicAdd(p.done, 1);
    s_last = ticket == static_cast<int>(gridDim.x) - 1;
    if (s_last) *p.done = 0;
  }
  __syncthreads();
  if (s_last && threadIdx.x < 32) {
    __threadfence();
    int base = 0;
    for (int f0 = 0; f0 < p.scan_upto; f0 += 32) {
      const int f = f0 + lane;
      const int v = f < p.scan_upto ? __ldcg(p.keep_n_all + f) : 0;
      int incl = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += up;
      }
      if (f < p.scan_upto) p.offsets[f] = base + incl - v;
      base += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) p.offsets[p.scan_upto] = base;
  }
}

// ------------------------------------------------------------------------------------------------
// gather (chains 470, 472, 477): output_0 [N,4], output_1 [N], output_2 [N,32] + scores / anchor ids / frame ids.
// One warp per detection; lane k copies coefficient k.
// ------------------------------------------------------------------------------------------------
template <typename T>
struct GatherParams {
  ScaleSrc<T> s[3];
  const int* keep_idx; const int* keep_n; const int* offsets;
  const float* boxes; const float* scores; const int* labels;
  int B, A, max_det;
  float* out_boxes; int* out_labels; float* out_coefs; float* out_scores; int* out_anchor; int* out_frame;
};

template <typename T>
__global__ void __launch_bounds__(256) gather_kernel(const GatherParams<T> p) {
  XR_PDL_ENTRY();
  // grid = (16, frames) x 8 warps: the 128 warps of a frame stride over its detections (a grid of frames x max_det warps launched
  // thousands of blocks that found nothing to do at ~10 detections per frame)
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  const int n = p.keep_n[b];
  const int base = p.offsets[b];
  const int warps = gridDim.x * (blockDim.x >> 5);
  for (int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += warps) {
    const int a = p.keep_idx[static_cast<long>(b) * p.max_det + i];
    const int o = base + i;
    int si = 0;
    if (a >= p.s[1].a_off) si = 1;
    if (a >= p.s[2].a_off) si = 2;
    const ScaleSrc<T>& s = p.s[si];
    const float c = ldf(s.coef + b * s.coef_bstride + static_cast<long>(a - s.a_off) * s.coef_pitch + lane);
    p.out_coefs[static_cast<long>(o) * NM + lane] = c;
    if (lane < 4) p.out_boxes[static_cast<long>(o) * 4 + lane] = p.boxes[(static_cast<long>(b) * p.A + a) * 4 + lane];
    if (lane == 0) {
      p.out_labels[o] = p.labels[static_cast<long>(b) * p.A + a];
      p.out_scores[o] = p.scores[static_cast<long>(b) * p.A + a];
      p.out_anchor[o] = a;
      p.out_frame[o] = b;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// masks (chains 496-498): output_3[o, pix] = sigmoid(sum_k coef[o,k] * proto[b,k,pix]), k = 0..31 sequential fp32 FMA.
// Block = 256 pixels of one frame; each thread keeps its pixel's 32 prototype values in registers and loops over
// the frame's detections (coefficients broadcast from shared memory).  PLANAR selects proto layout [B,32,P] (fp32,
// the oracle's tensor) instead of NHWC fp16 [B,P,32].
// ------------------------------------------------------------------------------------------------
template <typename T, bool PLANAR>
struct MaskParams {
  const T* protos; long proto_bstride; int proto_pitch;
  const float* coefs;      // [N,32] compacted
  const int* keep_n; const int* offsets;
  int max_det;
  float* probs;            // [N,160,160]
};

template <typename T, bool PLANAR>
__global__ void __launch_bounds__(256) mask_prob_kernel(const MaskParams<T, PLANAR> p) {
  XR_PDL_ENTRY();
  __shared__ __align__(16) float sc[32][NM];    // broadcast reads (every thread the same address): 8 LDS.128 per detection
  const int b = blockIdx.y;
  const int n = p.keep_n[b];
  if (n == 0) return;
  const int off = p.offsets[b];
  const int pix = blockIdx.x * 256 + threadIdx.x;
  float pr[NM];
  if (PLANAR) {
#pragma unroll
    for (int k = 0; k < NM; ++k) pr[k] = ldf(p.protos + b * p.proto_bstride + static_cast<long>(k) * PROTO_PIX + pix);
  } else {
    const uint4* pp = reinterpret_cast<const uint4*>(p.protos + b * p.proto_bstride + static_cast<long>(pix) * p.proto_pitch);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint4 raw = pp[i];
      const __half2* h = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __half22float2(h[j]);
        pr[i * 8 + 2 * j] = f.x;
        pr[i * 8 + 2 * j + 1] = f.y;
      }
    }
  }
  for (int d0 = 0; d0 < n; d0 += 32) {
    const int nd = min(32, n - d0);
    __syncthreads();
    for (int i = threadIdx.x; i < nd * NM; i += 256) sc[i / NM][i % NM] = p.coefs[static_cast<long>(off + d0) * NM + i];
    __syncthreads();
    for (int d = 0; d < nd; ++d) {
      float acc = 0.f;
#pragma unroll
      for (int k4 = 0; k4 < NM / 4; ++k4) {      // sequential fp32 FMA chain k = 0..31 (the oracle's order)
        const float4 c = reinterpret_cast<const float4*>(sc[d])[k4];
        acc = __fmaf_rn(c.x, pr[4 * k4], acc);
        acc = __fmaf_rn(c.y, pr[4 * k4 + 1], acc);
        acc = __fmaf_rn(c.z, pr[4 * k4 + 2], acc);
        acc = __fmaf_rn(c.w, pr[4 * k4 + 3], acc);
      }
      // PLANAR = the oracle's own fp32 tensors: IEEE sigmoid (probabilities agree to 1e-6, thresholds bit for bit);
      // network path (fp16 prototypes, tolerance 0.1 % of mask pixels): ex2/rcp approximations, same sign behaviour
      const float prob = PLANAR ? __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-acc))) : __fdividef(1.0f, 1.0f + __expf(-acc));
      __stcs(p.probs + static_cast<long>(off + d0 + d) * PROTO_PIX + pix, prob);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// masks on the network path (fp16 prototypes, NHWC [B,P,32]): the same product as mask_prob_kernel, on mma.sync.
// The scalar kernel is bound by its own 32-FMA chain per output (issue slots, not HBM); here one m16n8k16 pair does
// 16 detections x 8 pixels x 32 prototypes with fp32 accumulation, coefficients rounded to fp16 (the prototypes already
// are).  The exact fp32 FMA-chain kernel stays the one fed with the oracle's tensors (PLANAR); this one is checked per
// probability against a float64 bound (tests/test_pipeline_ends.py).
// Block = 8 warps x MASK_MMA_GROUPS groups of 8 consecutive pixels of one frame; detections in tiles of 16.
// ------------------------------------------------------------------------------------------------
constexpr int MASK_MMA_GROUPS = 8;                           // 8-pixel groups per warp
constexpr int MASK_MMA_PIX = 8 * 8 * MASK_MMA_GROUPS;        // pixels per block (512)
constexpr int MASK_DET_STAGE = 64;                           // detections whose coefficients are staged per barrier pair

__device__ __forceinline__ void mask_hmma(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// sigmoid(x) = 0.5 tanh(x / 2) + 0.5: ONE MUFU per probability instead of two (ex2 + rcp).  With hundreds of detections per
// frame the kernel was bound by the special-function unit (2 x 7.7 M per frame), not by the 102 400 B it writes per
// detection.  Same sign behaviour as the exact form, so the 0.5 threshold falls on the same pixels.
__device__ __forceinline__ float mask_sigmoid(float x) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * x));
  return fmaf(0.5f, t, 0.5f);
}

// Loop order: a warp keeps the prototype (B) fragments of its 64 pixels in registers and sweeps over ALL detections of the
// frame, 16 at a time -- the prototypes are read from memory once per block, not once per detection tile (the first version
// re-read them for each of the 19 tiles of a 300-detection frame and ran at 34 % of HBM peak there).
__global__ void __launch_bounds__(256) mask_prob_mma_kernel(const MaskParams<__half, false> p) {
  XR_PDL_ENTRY();
  __shared__ __align__(16) __half sc[MASK_DET_STAGE][NM + 8];   // coefficients (fp16), padded rows
  const int b = blockIdx.y;
  const int n = p.keep_n[b];
  if (n == 0) return;
  const int off = p.offsets[b];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int pix_base = blockIdx.x * MASK_MMA_PIX + warp * (8 * MASK_MMA_GROUPS);
  const __half* pr = p.protos + b * p.proto_bstride;
  // B fragments (col-major 16 x 8): column = pixel pix0 + g, rows = prototypes; b0 = B[2t..2t+1], b1 = B[2t+8..2t+9]
  uint32_t bf[MASK_MMA_GROUPS][4];
#pragma unroll
  for (int grp = 0; grp < MASK_MMA_GROUPS; ++grp) {
    const __half* q = pr + static_cast<long>(pix_base + grp * 8 + g) * p.proto_pitch + 2 * t;
#pragma unroll
    for (int j = 0; j < 4; ++j) bf[grp][j] = *reinterpret_cast<const uint32_t*>(q + 8 * j);
  }
  for (int ds = 0; ds < n; ds += MASK_DET_STAGE) {
    const int ns = min(MASK_DET_STAGE, n - ds);
    __syncthreads();
    for (int i = threadIdx.x; i < MASK_DET_STAGE * NM; i += 256) {
      const int r = i / NM, k = i - r * NM;
      sc[r][k] = __float2half_rn(r < ns ? p.coefs[static_cast<long>(off + ds + r) * NM + k] : 0.f);
    }
    __syncthreads();
    for (int d0 = 0; d0 < ns; d0 += 16) {
      const int nd = min(16, ns - d0);
      // A fragments (row-major 16 x 16, two k-steps): a0 = A[g][2t..], a1 = A[g+8][2t..], a2 = A[g][2t+8..], a3 = A[g+8][2t+8..]
      uint32_t a[2][4];
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) {
        a[ks][0] = *reinterpret_cast<const uint32_t*>(&sc[d0 + g][16 * ks + 2 * t]);
        a[ks][1] = *reinterpret_cast<const uint32_t*>(&sc[d0 + g + 8][16 * ks + 2 * t]);
        a[ks][2] = *reinterpret_cast<const uint32_t*>(&sc[d0 + g][16 * ks + 2 * t + 8]);
        a[ks][3] = *reinterpret_cast<const uint32_t*>(&sc[d0 + g + 8][16 * ks + 2 * t + 8]);
      }
      float* out0 = p.probs + static_cast<long>(off + ds + d0 + g) * PROTO_PIX + pix_base + 2 * t;
      float* out1 = out0 + static_cast<long>(8) * PROTO_PIX;
#pragma unroll
      for (int grp = 0; grp < MASK_MMA_GROUPS; ++grp) {
        float c[4] = {0.f, 0.f, 0.f, 0.f};
        mask_hmma(c, a[0], bf[grp][0], bf[grp][1]);
        mask_hmma(c, a[1], bf[grp][2], bf[grp][3]);
        // c0,c1 = detection g, pixels pix0 + 2t, +1;  c2,c3 = detection g + 8
        if (g < nd) __stcs(reinterpret_cast<float2*>(out0 + grp * 8), make_float2(mask_sigmoid(c[0]), mask_sigmoid(c[1])));
        if (g + 8 < nd) __stcs(reinterpret_cast<float2*>(out1 + grp * 8), make_float2(mask_sigmoid(c[2]), mask_sigmoid(c[3])));
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// C# box conventions (IEExecutor.ParseBoxes IEE:529-559, IEBoxer.DrawBoxes IEB:37-81)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 box_convention(const float4 raw, int conv, float sw, float sh) {
  if (conv == 2) return raw;
  const float sx = __fdiv_rn(sw, 640.f), sy = __fdiv_rn(sh, 640.f);
  float4 o;
  if (conv == 0) {
    o.x = __fmul_rn(__fsub_rn(raw.x, 320.f), sx);
    o.y = __fmul_rn(__fsub_rn(320.f, raw.y), sy);
  } else {
    o.x = __fsub_rn(__fmul_rn(raw.x, sx), __fdiv_rn(sw, 2.f));
    o.y = __fsub_rn(__fmul_rn(raw.y, sy), __fdiv_rn(sh, 2.f));
  }
  o.z = __fmul_rn(raw.z, sx);
  o.w = __fmul_rn(raw.w, sy);
  return o;
}

struct BoxOut {
  float cx, cy, w, h;
  int label, frame;
};

// per-frame cap (50 / 200 / none) applied like the C# loops; writes rows compacted again over the batch.
// One block (one warp) per frame: its output base is the capped count of the frames before it (warp-reduced), then the
// lanes convert the frame's boxes in parallel.
__global__ void __launch_bounds__(32) boxes_to_screen_kernel(const float* boxes, const int* labels, const int* keep_n,
                                                             const int* offsets, int B, int conv, float sw, float sh, int cap,
                                                             BoxOut* out, int* out_n) {
  const int b = blockIdx.x, lane = threadIdx.x;
  int base = 0;
  for (int f = lane; f < b; f += 32) base += cap > 0 ? min(keep_n[f], cap) : keep_n[f];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) base += __shfl_xor_sync(0xffffffffu, base, o);
  const int n = cap > 0 ? min(keep_n[b], cap) : keep_n[b];
  const int first = offsets[b];
  for (int i = lane; i < n; i += 32) {
    const float4 r = box_convention(reinterpret_cast<const float4*>(boxes)[first + i], conv, sw, sh);
    BoxOut v;
    v.cx = r.x; v.cy = r.y; v.w = r.z; v.h = r.w;
    v.label = labels[first + i];
    v.frame = b;
    out[base + i] = v;
  }
  if (b == B - 1 && lane == 0) *out_n = base + n;
}

// IEMasker.PixelInBoundingBox (IEM:232-247) on a C#-convention box
__device__ __forceinline__ bool pixel_in_box(const float4 box, int x, int y, int image_w, int image_h) {
  const float xs = __fdiv_rn(160.f, static_cast<float>(image_w));
  const float ys = __fdiv_rn(160.f, static_cast<float>(image_h));
  const float cx = __fadd_rn(__fmul_rn(box.x, xs), 80.f);
  const float cy = __fsub_rn(80.f, __fmul_rn(box.y, ys));
  const float hw = __fdiv_rn(__fmul_rn(box.z, xs), 2.f);
  const float hh = __fdiv_rn(__fmul_rn(box.w, ys), 2.f);
  const float xf = static_cast<float>(x), yf = static_cast<float>(y);
  return xf >= __fsub_rn(cx, hw) && xf <= __fadd_rn(cx, hw) && yf >= __fsub_rn(cy, hh) && yf <= __fadd_rn(cy, hh);
}

// mode 0: IEMasker.DrawMask / DrawSingleMask loop (IEM:98-113,167-185): u8 [n,160,160] in texture row order.
// mode 1: geometric crop in image row order.   boxes: raw cx,cy,w,h rows (converted here) or C# boxes (conv < 0).
struct MaskThrParams {
  const float* probs;   // [n,160,160]
  const float* boxes;   // [n,4]
  int n, first;
  int mode, conv;
  float sw, sh;
  int image_w, image_h;
  float thr;
  uint8_t* out;         // [n,160,160]
};

__global__ void __launch_bounds__(256) mask_threshold_kernel(const MaskThrParams p) {
  const int d = blockIdx.y;
  const int pix = blockIdx.x * 256 + threadIdx.x;
  const int y = pix / PROTO_HW, x = pix - y * PROTO_HW;
  const float4 raw = reinterpret_cast<const float4*>(p.boxes)[p.first + d];
  const float v = p.probs[static_cast<long>(p.first + d) * PROTO_PIX + pix];
  if (p.mode == 0) {
    const float4 box = p.conv < 0 ? raw : box_convention(raw, p.conv, p.sw, p.sh);
    const int pos_y = PROTO_HW - y - 1;
    const bool on = (v > p.thr) && pixel_in_box(box, x, pos_y, p.image_w, p.image_h);
    p.out[static_cast<long>(d) * PROTO_PIX + pos_y * PROTO_HW + x] = on ? 1 : 0;
  } else {
    const float s = 0.25f;
    const float x1 = __fmul_rn(__fsub_rn(raw.x, __fmul_rn(raw.z, 0.5f)), s), x2 = __fmul_rn(__fadd_rn(raw.x, __fmul_rn(raw.z, 0.5f)), s);
    const float y1 = __fmul_rn(__fsub_rn(raw.y, __fmul_rn(raw.w, 0.5f)), s), y2 = __fmul_rn(__fadd_rn(raw.y, __fmul_rn(raw.w, 0.5f)), s);
    const float xf = static_cast<float>(x), yf = static_cast<float>(y);
    const bool on = (v > p.thr) && xf >= x1 && xf < x2 && yf >= y1 && yf < y2;
    p.out[static_cast<long>(d) * PROTO_PIX + pix] = on ? 1 : 0;
  }
}

// mode 3: crop mask bit-packed, one u32 per 32 pixels of a row: [n,160,5]
__global__ void __launch_bounds__(160) mask_bits_kernel(const MaskThrParams p) {
  const int d = blockIdx.y;
  const int y = blockIdx.x;
  const int x = threadIdx.x;
  const float4 raw = reinterpret_cast<const float4*>(p.boxes)[p.first + d];
  const float v = p.probs[static_cast<long>(p.first + d) * PROTO_PIX + y * PROTO_HW + x];
  const float s = 0.25f;
  const float x1 = __fmul_rn(__fsub_rn(raw.x, __fmul_rn(raw.z, 0.5f)), s), x2 = __fmul_rn(__fadd_rn(raw.x, __fmul_rn(raw.z, 0.5f)), s);
  const float y1 = __fmul_rn(__fsub_rn(raw.y, __fmul_rn(raw.w, 0.5f)), s), y2 = __fmul_rn(__fadd_rn(raw.y, __fmul_rn(raw.w, 0.5f)), s);
  const float xf = static_cast<float>(x), yf = static_cast<float>(y);
  const bool on = (v > p.thr) && xf >= x1 && xf < x2 && yf >= y1 && yf < y2;
  const unsigned bits = __ballot_sync(0xFFFFFFFFu, on);
  if ((x & 31) == 0) reinterpret_cast<uint32_t*>(p.out)[(static_cast<long>(d) * PROTO_HW + y) * 5 + (x >> 5)] = bits;
}

// ------------------------------------------------------------------------------------------------
// RGB-D point extraction (SURVEY.md §8f N3): ↔ IEExecutor.ExtractDepthData + DepthExtractionJob.Execute (IEE:561-651,
// 86-156) and CollectJobResults' in-order compaction (IEE:653-667).  One sample per (160 / step)^2 grid point of the
// target's mask: mask > thr -> box-relative image position -> depth lookup (half -> float, 0.1 m < d < 3.0 m) ->
// unproject with the camera intrinsics -> rotate by the depth camera pose.  The reference copies the 160x160 mask to the
// host and runs a Burst job; here the mask never leaves the device and only the compacted points do.
// Arithmetic follows the C# expression order with IEEE intrinsics (no FMA contraction); math.normalize / math.mul
// (quaternion, float3) are restated from Unity.Mathematics (rsqrt(dot) * v; v + q.w * t + cross(q.xyz, t), t = 2 cross(q.xyz, v)).
// ------------------------------------------------------------------------------------------------
struct DepthParams {
  const float* probs;          // output_3 row of the target: [160*160]
  const float* box;            // output_0 row of the target: raw cx, cy, w, h
  const uint16_t* depth;       // [depth_h * depth_w] half floats (device copy of the depth texture)
  int depth_w, depth_h, step, max_points;
  float thr, screen_w, screen_h;
  float pos[3], rot[4], focal[2], principal[2], sensor[2];
  float4* out;                 // [max_points] world x, y, z, depth in metres
  int* out_n;
};

__global__ void __launch_bounds__(1024) depth_extract_kernel(const DepthParams p) {
  __shared__ int s_warp[32];
  __shared__ int s_base;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_base = 0;
  __syncthreads();
  // ParseBoxes box (IEE:529-559) and back to raw 640-space exactly as ExtractDepthData does (IEE:586-589)
  const float sx = __fdiv_rn(p.screen_w, 640.f), sy = __fdiv_rn(p.screen_h, 640.f);
  const float bx = __fmul_rn(__fsub_rn(p.box[0], 320.f), sx), by = __fmul_rn(__fsub_rn(320.f, p.box[1]), sy);
  const float bw = __fmul_rn(p.box[2], sx), bh = __fmul_rn(p.box[3], sy);
  const float rcx = __fadd_rn(__fdiv_rn(bx, sx), 320.f), rcy = __fsub_rn(320.f, __fdiv_rn(by, sy));
  const float rw = __fdiv_rn(bw, sx), rh = __fdiv_rn(bh, sy);
  const int total_x = PROTO_HW / p.step;
  const int total = total_x * total_x;
  for (int i0 = 0; i0 < total; i0 += 1024) {
    const int index = i0 + tid;
    bool valid = false;
    float4 res = make_float4(0.f, 0.f, 0.f, 0.f);
    if (index < total) {
      const int ly = index / total_x, lx = index - ly * total_x;
      const int y = ly * p.step, x = lx * p.step;
      if (y < PROTO_HW && x < PROTO_HW && p.probs[y * PROTO_HW + x] > p.thr) {
        const float nx = __fdiv_rn(static_cast<float>(x), static_cast<float>(PROTO_HW));
        const float ny = __fdiv_rn(static_cast<float>(y), static_cast<float>(PROTO_HW));
        const float ipx = __fadd_rn(__fsub_rn(rcx, __fmul_rn(rw, 0.5f)), __fmul_rn(nx, rw));
        const float ipy = __fadd_rn(__fsub_rn(rcy, __fmul_rn(rh, 0.5f)), __fmul_rn(ny, rh));
        const float u = fminf(fmaxf(__fdiv_rn(ipx, 640.f), 0.f), 1.f);
        const float v = fminf(fmaxf(__fdiv_rn(ipy, 640.f), 0.f), 1.f);
        const float omv = __fsub_rn(1.0f, v);
        const int dx = static_cast<int>(__fmul_rn(u, static_cast<float>(p.depth_w - 1)));
        const int dy = static_cast<int>(__fmul_rn(omv, static_cast<float>(p.depth_h - 1)));
        const int di = dy * p.depth_w + dx;
        if (di >= 0 && di < p.depth_w * p.depth_h) {
          const float d = __half2float(__ushort_as_half(p.depth[di]));
          if (d > 0.1f && d < 3.0f) {
            const float cpx = __fmul_rn(u, p.sensor[0]), cpy = __fmul_rn(omv, p.sensor[1]);
            float dxc = __fdiv_rn(__fsub_rn(cpx, p.principal[0]), p.focal[0]);
            float dyc = __fdiv_rn(__fsub_rn(cpy, p.principal[1]), p.focal[1]);
            float dzc = 1.0f;
            const float dot = __fadd_rn(__fadd_rn(__fmul_rn(dxc, dxc), __fmul_rn(dyc, dyc)), __fmul_rn(dzc, dzc));
            const float inv = __fdiv_rn(1.0f, __fsqrt_rn(dot));
            dxc = __fmul_rn(inv, dxc); dyc = __fmul_rn(inv, dyc); dzc = __fmul_rn(inv, dzc);
            // t = 2 * cross(q.xyz, v)
            const float qx = p.rot[0], qy = p.rot[1], qz = p.rot[2], qw = p.rot[3];
            const float tx = __fmul_rn(2.f, __fsub_rn(__fmul_rn(qy, dzc), __fmul_rn(qz, dyc)));
            const float ty = __fmul_rn(2.f, __fsub_rn(__fmul_rn(qz, dxc), __fmul_rn(qx, dzc)));
            const float tz = __fmul_rn(2.f, __fsub_rn(__fmul_rn(qx, dyc), __fmul_rn(qy, dxc)));
            // v + q.w * t + cross(q.xyz, t)
            const float wx = __fadd_rn(__fadd_rn(dxc, __fmul_rn(qw, tx)), __fsub_rn(__fmul_rn(qy, tz), __fmul_rn(qz, ty)));
            const float wy = __fadd_rn(__fadd_rn(dyc, __fmul_rn(qw, ty)), __fsub_rn(__fmul_rn(qz, tx), __fmul_rn(qx, tz)));
            const float wz = __fadd_rn(__fadd_rn(dzc, __fmul_rn(qw, tz)), __fsub_rn(__fmul_rn(qx, ty), __fmul_rn(qy, tx)));
            res = make_float4(__fadd_rn(p.pos[0], __fmul_rn(wx, d)), __fadd_rn(p.pos[1], __fmul_rn(wy, d)),
                              __fadd_rn(p.pos[2], __fmul_rn(wz, d)), d);
            valid = true;
          }
        }
      }
    }
    // order-preserving compaction (the C# loop appends valid samples in index order and stops at _maxPoints)
    const unsigned bal = __ballot_sync(0xffffffffu, valid);
    if (lane == 0) s_warp[warp] = __popc(bal);
    __syncthreads();
    int before = 0, chunk_total = 0;
    for (int w = 0; w < 32; ++w) {
      const int c = s_warp[w];
      if (w < warp) before += c;
      chunk_total += c;
    }
    const int slot = s_base + before + __popc(bal & ((1u << lane) - 1u));
    if (valid && slot < p.max_points) p.out[slot] = res;
    __syncthreads();
    if (tid == 0) s_base += chunk_total;
    __syncthreads();
  }
  if (tid == 0) *p.out_n = min(s_base, p.max_points);
}

// Target association (IEE:488-507): nearest box of the locked class (ParseBoxes coordinates) among the first `cap`
// detections of a frame; strict `<` keeps the first of equal distances; accepted when the distance is below max_dist.
__global__ void associate_kernel(const float* boxes, const int* labels, int first, int n, int cap, float screen_w, float screen_h,
                                 float lx, float ly, int llabel, float max_dist, int* best_index, float* best_dist) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const float sx = __fdiv_rn(screen_w, 640.f), sy = __fdiv_rn(screen_h, 640.f);
  int best = -1;
  float mind = 3.402823466e+38f;
  const int m = n < cap ? n : cap;
  for (int i = 0; i < m; ++i) {
    if (labels[first + i] != llabel) continue;
    const float cx = __fmul_rn(__fsub_rn(boxes[4 * (first + i)], 320.f), sx);
    const float cy = __fmul_rn(__fsub_rn(320.f, boxes[4 * (first + i) + 1]), sy);
    const float dx = __fsub_rn(cx, lx), dy = __fsub_rn(cy, ly);
    const float dist = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
    if (dist < mind) { mind = dist; best = i; }
  }
  *best_index = (best != -1 && mind < max_dist) ? best : -1;
  *best_dist = mind;
}

// ------------------------------------------------------------------------------------------------
// mode 2 (extension, BASELINE.json config 5): fused coef x proto -> bilinear 160->640 of the LOGITS -> box crop ->
// threshold (logit > 0) -> u8 [n,640,640].  Block = one detection x one 64x64 output tile: the 18x18 logit patch it
// needs is computed once into shared memory from the frame's prototypes.
// ------------------------------------------------------------------------------------------------
struct Mask640Params {
  const __half* protos; long proto_bstride; int proto_pitch;
  const float* coefs; const float* boxes; const int* frames;
  int first;
  uint8_t* out;   // [n,640,640]
  float logit_thr;  // logit of the probability threshold (0 for 0.5)
};

__global__ void __launch_bounds__(256) mask640_kernel(const Mask640Params p) {
  __shared__ float patch[18][19];
  __shared__ float sc[NM];
  const int d = blockIdx.z;
  const int o = p.first + d;
  const int tx = blockIdx.x, ty = blockIdx.y;  // 10 x 10 tiles of 64
  const float4 raw = reinterpret_cast<const float4*>(p.boxes)[o];
  const float x1 = __fsub_rn(raw.x, __fmul_rn(raw.z, 0.5f)), x2 = __fadd_rn(raw.x, __fmul_rn(raw.z, 0.5f));
  const float y1 = __fsub_rn(raw.y, __fmul_rn(raw.w, 0.5f)), y2 = __fadd_rn(raw.y, __fmul_rn(raw.w, 0.5f));
  {
    // A tile the box does not touch is all zeros whatever the logits are (the crop test below is xf >= x1 && xf < x2, same for
    // y): write it without computing the patch.  Most of a 640x640 mask lies outside its box -- the kernel was bound by the ~40
    // strictly ordered fp32 operations per output pixel, not by the 7.9 GB it writes at 300 detections x 64 frames.
    const float tx0 = static_cast<float>(tx * 64), tx1 = static_cast<float>(tx * 64 + 63);
    const float ty0 = static_cast<float>(ty * 64), ty1 = static_cast<float>(ty * 64 + 63);
    if (!(tx1 >= x1 && tx0 < x2 && ty1 >= y1 && ty0 < y2)) {
      const int ry = threadIdx.x >> 2, seg = threadIdx.x & 3;
      __stcs(reinterpret_cast<uint4*>(p.out + (static_cast<long>(d) * 640 + ty * 64 + ry) * 640 + tx * 64 + seg * 16), make_uint4(0, 0, 0, 0));
      return;
    }
  }
  if (threadIdx.x < NM) sc[threadIdx.x] = p.coefs[static_cast<long>(o) * NM + threadIdx.x];
  const int b = p.frames[o];
  __syncthreads();
  // source coordinate of output pixel X: (X + 0.5) * 0.25 - 0.5 ; tile covers X in [64 tx, 64 tx + 63]
  const int sx0 = tx * 16 - 1, sy0 = ty * 16 - 1;  // first source index touched (may be -1 -> clamped)
  for (int i = threadIdx.x; i < 18 * 18; i += 256) {
    const int py = i / 18, px = i - py * 18;
    const int sy = min(max(sy0 + py, 0), PROTO_HW - 1), sx = min(max(sx0 + px, 0), PROTO_HW - 1);
    const uint4* pp = reinterpret_cast<const uint4*>(p.protos + b * p.proto_bstride +
                                                     static_cast<long>(sy * PROTO_HW + sx) * p.proto_pitch);
    float acc = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint4 raw = pp[q];
      const __half2* h = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __half22float2(h[j]);
        acc = __fmaf_rn(sc[q * 8 + 2 * j], f.x, acc);
        acc = __fmaf_rn(sc[q * 8 + 2 * j + 1], f.y, acc);
      }
    }
    patch[py][px] = acc;
  }
  __syncthreads();
  // each thread: 16 consecutive output pixels of one row (64 rows x 4 segments)
  const int ry = threadIdx.x >> 2, seg = threadIdx.x & 3;
  const int Y = ty * 64 + ry;
  float fy = __fsub_rn(__fmul_rn(__fadd_rn(static_cast<float>(Y), 0.5f), 0.25f), 0.5f);
  fy = fmaxf(fy, 0.f);
  int iy0 = min(static_cast<int>(floorf(fy)), PROTO_HW - 1);
  const int iy1 = min(iy0 + 1, PROTO_HW - 1);
  const float wy = __fsub_rn(fy, static_cast<float>(iy0));
  uint32_t packed[4] = {0, 0, 0, 0};
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const int X = tx * 64 + seg * 16 + i;
    float fx = __fsub_rn(__fmul_rn(__fadd_rn(static_cast<float>(X), 0.5f), 0.25f), 0.5f);
    fx = fmaxf(fx, 0.f);
    const int ix0 = min(static_cast<int>(floorf(fx)), PROTO_HW - 1);
    const int ix1 = min(ix0 + 1, PROTO_HW - 1);
    const float wx = __fsub_rn(fx, static_cast<float>(ix0));
    const float a = patch[iy0 - sy0][ix0 - sx0], bq = patch[iy0 - sy0][ix1 - sx0];
    const float c = patch[iy1 - sy0][ix0 - sx0], dq = patch[iy1 - sy0][ix1 - sx0];
    const float top = __fadd_rn(__fmul_rn(a, __fsub_rn(1.f, wx)), __fmul_rn(bq, wx));
    const float bot = __fadd_rn(__fmul_rn(c, __fsub_rn(1.f, wx)), __fmul_rn(dq, wx));
    const float val = __fadd_rn(__fmul_rn(top, __fsub_rn(1.f, wy)), __fmul_rn(bot, wy));
    const float xf = static_cast<float>(X), yf = static_cast<float>(Y);
    const bool on = (val > p.logit_thr) && xf >= x1 && xf < x2 && yf >= y1 && yf < y2;
    packed[i >> 2] |= (on ? 1u : 0u) << ((i & 3) * 8);
  }
  uint4 v = make_uint4(packed[0], packed[1], packed[2], packed[3]);
  __stcs(reinterpret_cast<uint4*>(p.out + (static_cast<long>(d) * 640 + Y) * 640 + tx * 64 + seg * 16), v);
}

#endif  // __CUDACC__
}  // namespace xrseg
