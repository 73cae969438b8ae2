// Shared device/host helpers for the b2c (B200 captioner) kernels.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>

#include "../../include/b2c.h"

namespace b2c {

typedef __nv_bfloat16 bf16;
typedef __half f16;          // teacher operands only (B2C_F16): the student never computes in fp16

// ------------------------------------------------------------------ errors
// Thread-local message; every entry point returns 0 or a negative B2C_E* code and never aborts.
inline char* err_buf() { static thread_local char buf[512] = {0}; return buf; }
inline int set_err(int code, const char* fmt, ...) {
  va_list ap; va_start(ap, fmt); vsnprintf(err_buf(), 512, fmt, ap); va_end(ap); return code;
}
#define B2C_CHECK_ARG(cond, ...) do { if (!(cond)) return b2c::set_err(B2C_EINVAL, __VA_ARGS__); } while (0)
#define B2C_CUDA(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) \
    return b2c::set_err(B2C_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)
inline unsigned long long& launch_counter() { static unsigned long long n = 0; return n; }
#define B2C_LAUNCH_CHECK(name) do { ++b2c::launch_counter(); cudaError_t e_ = cudaGetLastError(); if (e_ != cudaSuccess) \
    return b2c::set_err(B2C_ECUDA, "launch of %s failed: %s (%s:%d)", name, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)
#define B2C_TRY(expr) do { int r_ = (expr); if (r_ != 0) return r_; } while (0)

// ------------------------------------------------------------------ numeric type helpers
template <typename T> __device__ __forceinline__ float to_f(T v);
template <> __device__ __forceinline__ float to_f<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f<bf16>(bf16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f<f16>(f16 v) { return __half2float(v); }
template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f<bf16>(float v) { return __float2bfloat16_rn(v); }

// Accurate math in fp32 mode (parity 1e-4 / exact argmax), fast approximations in bf16 mode.
template <typename T> struct Math;
template <> struct Math<float> {
  static __device__ __forceinline__ float tanh_(float x) { return tanhf(x); }
  static __device__ __forceinline__ float sigmoid_(float x) { return 1.0f / (1.0f + expf(-x)); }
  static __device__ __forceinline__ float exp_(float x) { return expf(x); }
  static __device__ __forceinline__ float log_(float x) { return logf(x); }
  static __device__ __forceinline__ float dtanh_(float x) { const float t = tanhf(x); return fmaf(-t, t, 1.0f); }      // 1 - tanh^2
};
// bf16 mode: MUFU ex2/rcp based forms (abs error ~1e-7).  tanh.approx (rel 2^-11) is NOT used: the attention score is a sum
// of E tanh values, and its error goes straight into the softmax weights and from there into ReLU-mask flips downstream.
__device__ __forceinline__ float ex2_ftz_(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_ftz_(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
template <> struct Math<bf16> {
  // tanh(x) = 1 - 2 / (1 + e^{2x}),  sigmoid(x) = 1 / (1 + e^{-x}):  FMUL + MUFU.EX2 + FADD + MUFU.RCP + FFMA, no range fix-ups
  // (x -> +inf: e^{2x} = inf, rcp = 0 -> 1;  x -> -inf: e^{2x} = 0 -> 1 - 2 = -1)
  static __device__ __forceinline__ float tanh_(float x) { return fmaf(-2.0f, rcp_ftz_(1.0f + ex2_ftz_(2.8853900817779268f * x)), 1.0f); }
  static __device__ __forceinline__ float sigmoid_(float x) { return rcp_ftz_(1.0f + ex2_ftz_(-1.4426950408889634f * x)); }
  static __device__ __forceinline__ float exp_(float x) { return ex2_ftz_(1.4426950408889634f * x); }
  static __device__ __forceinline__ float log_(float x) { return __logf(x); }
  // 1 - tanh^2(x) for the BACKWARD only: one MUFU (tanh.approx, rel. error 2^-11 ~ a quarter of a bf16 ulp).  A relative error in
  // the derivative only rescales one gradient contribution; the forward (scores -> softmax) keeps the ex2 / rcp form above.
  static __device__ __forceinline__ float dtanh_(float x) { float t; asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(x)); return fmaf(-t, t, 1.0f); }
};

// 2^x, one MUFU (flush-to-zero: no denormal range fix-up code around it)
__device__ __forceinline__ float ex2_ftz(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Counter-based dropout: keep-mask from a 32-bit mix of (seed, stream id, element index).
// Stateless so backward regenerates the same mask; no mask tensor is stored.
__device__ __forceinline__ uint32_t mix32(uint64_t seed, uint32_t stream, uint64_t idx) {
  uint64_t z = seed + 0x9E3779B97F4A7C15ull * (idx + 1) + ((uint64_t)stream << 40);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z = z ^ (z >> 31);
  return (uint32_t)(z >> 32);
}
// effective seed: the by-value seed (frozen inside a captured CUDA graph) mixed with an optional device-side step counter
__device__ __forceinline__ uint64_t drop_seed(uint64_t seed, const unsigned long long* seed_dev) {
  return seed_dev ? seed + 0xD6E8FEB86659FD93ull * __ldg(seed_dev) : seed;
}
// returns 0 (dropped) or 1/(1-p) (kept)
__device__ __forceinline__ float dropout_scale(uint64_t seed, uint32_t stream, uint64_t idx, float p, float inv_keep) {
  const uint32_t thr = (uint32_t)(p * 4294967296.0f);
  return mix32(seed, stream, idx) >= thr ? inv_keep : 0.0f;
}

// ------------------------------------------------------------------ programmatic dependent launch (PDL)
// The recurrence is a chain of ~280 dependent small kernels per training step.  Kernels on that chain are launched with
// cudaLaunchAttributeProgrammaticStreamSerialization: each calls pdl_launch_dependents() first (the next kernel may start its
// prologue: barrier init, TMEM allocation, descriptor prefetch) and pdl_wait() before it touches global memory (blocks until
// every prerequisite grid has completed and flushed).  Both are no-ops for a normally launched kernel.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

inline bool pdl_enabled() {
  static int on = -1;
  if (on < 0) { const char* e = getenv("B2C_PDL"); on = (e && e[0] == '0') ? 0 : 1; }
  return on != 0;
}
// Kernels that prefetch loop-invariant operands BEFORE griddepcontrol.wait (attention steps) rely on those operands being
// complete when ANY kernel of the chain may start early.  Early starts cascade (every kernel signals launch_dependents
// at its top), so the caller breaks the cascade once, after the producers: the next launch_pdl call is issued as an
// ordinary, fully serialised launch.
inline bool& pdl_full_dependency_flag() { static thread_local bool f = false; return f; }
inline void pdl_full_dependency_next() { pdl_full_dependency_flag() = true; }
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = (pdl_enabled() && !pdl_full_dependency_flag()) ? 1 : 0;
  pdl_full_dependency_flag() = false;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// ------------------------------------------------------------------ PTX wrappers (mbarrier / bulk copies)
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// Bounded wait: a lost arrival (bad tensor map, wrong expect_tx) traps with a launch failure instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  for (uint32_t spins = 0; !mbar_try_wait(bar, parity); ++spins) {
    if (spins > (1u << 24)) { printf("b2c: mbarrier wait timed out (block %d,%d thread %d)\n", blockIdx.x, blockIdx.y, threadIdx.x); __trap(); }
  }
}
// 1-D bulk async copy global -> shared (TMA engine, SASS UBLKCP); size and both addresses 16-byte aligned.
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// 128-bit streaming loads/stores that do not pollute L1
__device__ __forceinline__ uint4 ld_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_na_v4(void* p, const uint4& v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ float bf16_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }
__device__ __forceinline__ float f16_lo(uint32_t u) { return __half2float(__ushort_as_half((unsigned short)(u & 0xffffu))); }
__device__ __forceinline__ float f16_hi(uint32_t u) { return __half2float(__ushort_as_half((unsigned short)(u >> 16))); }
// the two elements of a 32-bit word of a 2-byte type, widened exactly to fp32
template <typename T> __device__ __forceinline__ float lo_f(uint32_t u);
template <typename T> __device__ __forceinline__ float hi_f(uint32_t u);
template <> __device__ __forceinline__ float lo_f<bf16>(uint32_t u) { return bf16_lo(u); }
template <> __device__ __forceinline__ float hi_f<bf16>(uint32_t u) { return bf16_hi(u); }
template <> __device__ __forceinline__ float lo_f<f16>(uint32_t u) { return f16_lo(u); }
template <> __device__ __forceinline__ float hi_f<f16>(uint32_t u) { return f16_hi(u); }
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

// ------------------------------------------------------------------ 8-element (16-byte for bf16) row chunks
template <typename T> struct Vec8;
template <> struct Vec8<bf16> {
  static __device__ __forceinline__ void load(const bf16* p, float (&v)[8]) {
    const uint4 a = *reinterpret_cast<const uint4*>(p);
    v[0] = bf16_lo(a.x); v[1] = bf16_hi(a.x); v[2] = bf16_lo(a.y); v[3] = bf16_hi(a.y);
    v[4] = bf16_lo(a.z); v[5] = bf16_hi(a.z); v[6] = bf16_lo(a.w); v[7] = bf16_hi(a.w);
  }
  static __device__ __forceinline__ void store(bf16* p, const float (&v)[8]) {
    *reinterpret_cast<uint4*>(p) = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
  }
};
template <> struct Vec8<f16> {                // load only: fp16 is a teacher operand type
  static __device__ __forceinline__ void load(const f16* p, float (&v)[8]) {
    const uint4 a = *reinterpret_cast<const uint4*>(p);
    v[0] = f16_lo(a.x); v[1] = f16_hi(a.x); v[2] = f16_lo(a.y); v[3] = f16_hi(a.y);
    v[4] = f16_lo(a.z); v[5] = f16_hi(a.z); v[6] = f16_lo(a.w); v[7] = f16_hi(a.w);
  }
};
template <> struct Vec8<float> {
  static __device__ __forceinline__ void load(const float* p, float (&v)[8]) {
    const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
  static __device__ __forceinline__ void store(float* p, const float (&v)[8]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
  }
};


inline int cdiv(long a, long b) { return (int)((a + b - 1) / b); }
__host__ __device__ inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace b2c
