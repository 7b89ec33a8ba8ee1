// common.cuh -- error handling, sm_100a PTX wrappers (mbarrier, cp.async, tcgen05/TMEM) and small helpers
// shared by every kernel of libxrseg.so.  Written for sm_100a only; there is no other code path.
#pragma once

#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <string>
#include <utility>

namespace xrseg {

// ------------------------------------------------------------------------------------------------
// host-side error plumbing: kernels and CUDA calls report through a thread-local string
// ------------------------------------------------------------------------------------------------
struct CudaError {
  std::string msg;
};

#define XR_CUDA(call)                                                                              \
  do {                                                                                             \
    cudaError_t _e = (call);                                                                       \
    if (_e != cudaSuccess) {                                                                       \
      char _b[512];                                                                                \
      snprintf(_b, sizeof(_b), "%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
      throw ::xrseg::CudaError{_b};                                                                \
    }                                                                                              \
  } while (0)

#define XR_CHECK(cond, ...)                                                                        \
  do {                                                                                             \
    if (!(cond)) {                                                                                 \
      char _b[512];                                                                                \
      int _n = snprintf(_b, sizeof(_b), "%s:%d: check failed: %s: ", __FILE__, __LINE__, #cond);   \
      snprintf(_b + _n, sizeof(_b) - _n, __VA_ARGS__);                                             \
      throw ::xrseg::CudaError{_b};                                                                \
    }                                                                                              \
  } while (0)

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline long ceil_div_l(long a, long b) { return (a + b - 1) / b; }
static inline int round_up(int a, int b) { return ceil_div(a, b) * b; }

#ifdef __CUDACC__

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ float silu_f(float y) { return __fdividef(y, 1.0f + __expf(-y)); }

// SiLU of two values, packed to fp16: silu(y) = h * tanh(h) + h with h = y / 2 -- one MUFU (tanh.approx.f32) and one FFMA
// per output, evaluated in fp32 with a single rounding to fp16 at the end (the reference applies Swish to an fp32 conv
// output, SURVEY.md fact 6).  Measured on B200 against the packed-fp16 form (tanh.approx.f16x2 + HFMA2, half the MUFU
// work but three roundings): no launch changes by more than noise (profiles/r2a_*), while the per-layer relative L2 error
// against the fp32 oracle drops by a third to a half and the worst class-logit error from 0.21 to 0.08
// (profiles/r2a_layer_sweep_*.md).
__device__ __forceinline__ uint32_t silu_pack_h2(float a, float b) {
  const float ha = 0.5f * a, hb = 0.5f * b;
  float ta, tb;
  asm("tanh.approx.f32 %0, %1;" : "=f"(ta) : "f"(ha));
  asm("tanh.approx.f32 %0, %1;" : "=f"(tb) : "f"(hb));
  __half2 r = __floats2half2_rn(fmaf(ha, ta, ha), fmaf(hb, tb, hb));
  return *reinterpret_cast<uint32_t*>(&r);
}

// 256-bit global accesses (sm_100): one full 32-byte sector per lane and instruction.
__device__ __forceinline__ void st_global_256(void* ptr, const uint32_t (&o)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(ptr), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]),
               "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7])
               : "memory");
}
__device__ __forceinline__ void ld_global_256(const void* ptr, uint32_t (&v)[8]) {
  asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "l"(ptr)
               : "memory");
}

// Epilogue of 16 consecutive output channels of one pixel: accumulator + bias -> (SiLU) -> (+ residual) -> fp16 -> two
// 16-byte stores.  bias16: shared memory, 64-byte aligned.  res / out: global, 32-byte aligned.
__device__ __forceinline__ void epilogue_chunk16(const uint32_t (&v)[16], const float* bias16, int act, const __half* res,
                                                 __half* out) {
  float y[16];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 b4 = reinterpret_cast<const float4*>(bias16)[i];
    y[4 * i] = __uint_as_float(v[4 * i]) + b4.x;
    y[4 * i + 1] = __uint_as_float(v[4 * i + 1]) + b4.y;
    y[4 * i + 2] = __uint_as_float(v[4 * i + 2]) + b4.z;
    y[4 * i + 3] = __uint_as_float(v[4 * i + 3]) + b4.w;
  }
  uint32_t o[8];
  if (act) {
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = silu_pack_h2(y[2 * i], y[2 * i + 1]);
    if (res) {
      uint32_t rr[8];
      ld_global_256(res, rr);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        __half2 s = __hadd2(*reinterpret_cast<__half2*>(&o[i]), *reinterpret_cast<const __half2*>(&rr[i]));
        o[i] = *reinterpret_cast<uint32_t*>(&s);
      }
    }
  } else {
    if (res) {
      uint32_t rr[8];
      ld_global_256(res, rr);
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
  st_global_256(out, o);
}

// The same for the TMA convolution kernel's lean epilogue: hb16 (shared memory) holds 0.5 * bias when `act` is set, so the
// half-argument of silu(y) = h tanh(h) + h is ONE FFMA on the accumulator (h = 0.5 acc + 0.5 bias): three FP32-pipe
// instructions and one MUFU per output, plus half a pack.
__device__ __forceinline__ uint32_t silu_pack_from_half_arg(float ha, float hb) {
  float ta, tb;
  asm("tanh.approx.f32 %0, %1;" : "=f"(ta) : "f"(ha));
  asm("tanh.approx.f32 %0, %1;" : "=f"(tb) : "f"(hb));
  __half2 r = __floats2half2_rn(fmaf(ha, ta, ha), fmaf(hb, tb, hb));
  return *reinterpret_cast<uint32_t*>(&r);
}
// probe (PROBE instantiation of the kernel only; 0 in the product): 1 = compute but do not store, 2 = store without the
// bias / SiLU math (raw accumulators rounded to fp16)
__device__ __forceinline__ void epilogue_chunk16_hb(const uint32_t (&v)[16], const float* hb16, bool act, const __half* res,
                                                    __half* out, int probe = 0) {
  uint32_t o[8];
  if (probe & 2) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      __half2 h = __floats2half2_rn(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1]));
      o[i] = *reinterpret_cast<uint32_t*>(&h);
    }
    st_global_256(out, o);
    return;
  }
  if (act) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 b4 = reinterpret_cast<const float4*>(hb16)[i];
      o[2 * i] = silu_pack_from_half_arg(fmaf(__uint_as_float(v[4 * i]), 0.5f, b4.x), fmaf(__uint_as_float(v[4 * i + 1]), 0.5f, b4.y));
      o[2 * i + 1] = silu_pack_from_half_arg(fmaf(__uint_as_float(v[4 * i + 2]), 0.5f, b4.z), fmaf(__uint_as_float(v[4 * i + 3]), 0.5f, b4.w));
    }
    if (res) {
      uint32_t rr[8];
      ld_global_256(res, rr);
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
      const float4 b4 = reinterpret_cast<const float4*>(hb16)[i];
      y[4 * i] = __uint_as_float(v[4 * i]) + b4.x;
      y[4 * i + 1] = __uint_as_float(v[4 * i + 1]) + b4.y;
      y[4 * i + 2] = __uint_as_float(v[4 * i + 2]) + b4.z;
      y[4 * i + 3] = __uint_as_float(v[4 * i + 3]) + b4.w;
    }
    if (res) {
      uint32_t rr[8];
      ld_global_256(res, rr);
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
  if (probe & 1) {                       // keep the math alive without the store
    if ((o[0] ^ o[1] ^ o[2] ^ o[3] ^ o[4] ^ o[5] ^ o[6] ^ o[7]) == 0x12345678u) st_global_256(out, o);
    return;
  }
  st_global_256(out, o);
}

// ---- programmatic dependent launch (PDL) ---------------------------------------------------------
// Every kernel of the per-frame pipeline is launched with cudaLaunchAttributeProgrammaticStreamSerialization, so its
// CTAs may become resident while the previous kernel drains.  pdl_launch_dependents(): this CTA no longer objects to
// the next kernel starting; pdl_wait(): block until the previous kernel has fully completed and its writes are
// visible -- must precede the first access to anything a previous kernel wrote (or still reads, if we write it).
// Both are no-ops when the kernel was launched without the attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
#define XR_PDL_ENTRY()         \
  do {                         \
    pdl_launch_dependents();   \
    pdl_wait();                \
  } while (0)

// ---- mbarrier ----------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Non-blocking probe (mbarrier.test_wait): try_wait may suspend the thread for a system-dependent time when the phase is not
// complete, which is what a wait loop wants but not a poll between two batches of tcgen05.mma.
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (CUDA error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) {
      if ((threadIdx.x & 31) == 0)
        printf("xrseg: mbarrier wait timeout (block %d of %d, thread %d, barrier @%u parity %u)\n", blockIdx.x, gridDim.x,
               threadIdx.x, smem_u32(bar) & 0xFFFFu, parity);
      __trap();
    }
  }
}

// ---- cp.async (LDGSTS), 16-byte, zero-fill when src_bytes == 0 --------------------------------
__device__ __forceinline__ void cp_async16(uint32_t dst_smem, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst_smem), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async16_ca(uint32_t dst_smem, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(dst_smem), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void cp_async_wait_dyn(int n) {   // wait until at most n groups of this thread are pending
  switch (n) {
    case 0: cp_async_wait<0>(); break;
    case 1: cp_async_wait<1>(); break;
    case 2: cp_async_wait<2>(); break;
    case 3: cp_async_wait<3>(); break;
    case 4: cp_async_wait<4>(); break;
    case 5: cp_async_wait<5>(); break;
    case 6: cp_async_wait<6>(); break;
    default: cp_async_wait<7>(); break;
  }
}
// generic-proxy writes -> visible to the async proxy (tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- tcgen05 / TMEM ----------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// One lane of a fully converged warp.  The MMA-issuing warp runs its loop with all 32 lanes (so the compiler keeps the
// descriptor arithmetic in uniform registers) and predicates only the tcgen05 instructions on the elected lane.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
  return pred != 0;
}

// D[tmem] (+)= A[smem] * B[smem]; kind::f16 covers fp16 and bf16 operands with fp32 accumulation.
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate));   // ordered by the volatile barrier asm around it
}
// D[tmem] (+)= A[tmem] * B[smem]: the A operand comes from tensor memory -- lane = row, 16 K values = 8 consecutive columns
// of packed half2 (element k of a row sits in column k / 2, half k % 2), written there by tcgen05.st.
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate));
}
// Same, executed by every lane of the warp but issued only where `issue` != 0: no branch around the instruction.
__device__ __forceinline__ void umma_f16_pred(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                              uint32_t accumulate, uint32_t issue) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 q, %5, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(issue));
}
__device__ __forceinline__ void umma_commit_pred(uint64_t* bar, uint32_t issue) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "setp.ne.b32 q, %1, 0;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
      ::"r"(smem_u32(bar)), "r"(issue)
      : "memory");
}
// Arrive on an mbarrier once every previously issued tcgen05.mma of this thread has completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 16 consecutive fp32 columns: thread i of the warp receives lane (quadrant*32 + i).
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 32 lanes x 8 consecutive 32-bit columns, registers -> tensor memory (thread i of the warp writes lane quadrant*32 + i).
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]),
               "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor, K-major, SWIZZLE_NONE ("interleaved" core matrices of 8 rows x 16 B):
//   bits [0,14)  start address >> 4        bits [16,30) leading-dim byte offset >> 4 (K-adjacent core matrices)
//   bits [32,46) stride-dim byte offset >> 4 (M/N-adjacent core matrices)      bits [46,48) version = 1 (sm_100)
//   bits [61,64) layout type = 0 (no swizzle)
__device__ __forceinline__ uint64_t umma_desc_kmajor_noswz(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  return d;
}

// Instruction descriptor for kind::f16: fp32 accumulate, A and B K-major, M = 128.
//   bits [4,6) c_format (1 = f32)  [7,10) a_format  [10,13) b_format (0 = f16, 1 = bf16)
//   bit 15 a_major, bit 16 b_major (0 = K)  [17,23) N >> 3  [24,29) M >> 4
__host__ __device__ __forceinline__ uint32_t umma_idesc_f16(int n, int is_bf16) {
  uint32_t d = 0;
  d |= 1u << 4;
  d |= (is_bf16 ? 1u : 0u) << 7;
  d |= (is_bf16 ? 1u : 0u) << 10;
  d |= static_cast<uint32_t>(n >> 3) << 17;
  d |= static_cast<uint32_t>(128 >> 4) << 24;
  return d;
}

// Launch with programmatic stream serialization (PDL): only for kernels that call pdl_wait() before touching data
// produced by earlier kernels.  XRSEG_PDL=0 in the environment turns the attribute off (A/B measurements).
inline bool pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("XRSEG_PDL");
    return !(e && e[0] == '0');
  }();
  return on;
}
template <typename... KArgs, typename... Args>
inline void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  XR_CUDA(cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...));
}

#endif  // __CUDACC__

}  // namespace xrseg
