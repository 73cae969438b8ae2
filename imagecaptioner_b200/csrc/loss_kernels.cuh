// Kernels (3) and (4) of the hot path: the streaming token-KD + CE pass and the fused
// feature/hidden KD reduction.  Math: SURVEY.md Appendix A.3, reference
// src/distillation_utils.py:30-54 (token KD), :154 (CE), :56-94 (feature KD), :96-136 (hidden KD).
#pragma once
#include "common.cuh"

namespace b2c {

constexpr int KD_THREADS = 128;

// ---- row IO helpers: G = 8 (vectorised, 16-byte accesses) or G = 1 (any V / alignment) -------------
template <typename TS, int G> struct RowIO;
template <> struct RowIO<float, 8> {
  static __device__ __forceinline__ void load(const float* s, int base, float (&v)[8]) {
    const float4 a = *reinterpret_cast<const float4*>(s + base), b = *reinterpret_cast<const float4*>(s + base + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
  static __device__ __forceinline__ void store_s(float* s, int base, const float (&v)[8]) {
    *reinterpret_cast<float4*>(s + base) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(s + base + 4) = make_float4(v[4], v[5], v[6], v[7]);
  }
  static __device__ __forceinline__ void store_g(float* g, long base, const float (&v)[8]) {
    uint4 a = make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3]));
    uint4 b = make_uint4(__float_as_uint(v[4]), __float_as_uint(v[5]), __float_as_uint(v[6]), __float_as_uint(v[7]));
    st_na_v4(g + base, a); st_na_v4(g + base + 4, b);
  }
};
template <> struct RowIO<bf16, 8> {
  static __device__ __forceinline__ void load(const bf16* s, int base, float (&v)[8]) {
    const uint4 a = *reinterpret_cast<const uint4*>(s + base);
    v[0] = bf16_lo(a.x); v[1] = bf16_hi(a.x); v[2] = bf16_lo(a.y); v[3] = bf16_hi(a.y);
    v[4] = bf16_lo(a.z); v[5] = bf16_hi(a.z); v[6] = bf16_lo(a.w); v[7] = bf16_hi(a.w);
  }
  static __device__ __forceinline__ void store_g(bf16* g, long base, const float (&v)[8]) {
    uint4 a = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
    st_na_v4(g + base, a);
  }
};
template <typename TS> struct RowIO<TS, 1> {
  static __device__ __forceinline__ void load(const TS* s, int base, float (&v)[1]) { v[0] = to_f<TS>(s[base]); }
  static __device__ __forceinline__ void store_s(float* s, int base, const float (&v)[1]) { s[base] = v[0]; }
  static __device__ __forceinline__ void store_g(TS* g, long base, const float (&v)[1]) { g[base] = from_f<TS>(v[0]); }
};

__device__ __forceinline__ float block_reduce_sum4(float& a, float& b, float& c, float& d, float* scratch) {
  // KD_THREADS/32 warps; every thread returns with all four totals
  a = warp_sum(a); b = warp_sum(b); c = warp_sum(c); d = warp_sum(d);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) { scratch[w * 4 + 0] = a; scratch[w * 4 + 1] = b; scratch[w * 4 + 2] = c; scratch[w * 4 + 3] = d; }
  __syncthreads();
  a = b = c = d = 0.f;
#pragma unroll
  for (int i = 0; i < KD_THREADS / 32; ++i) { a += scratch[i * 4]; b += scratch[i * 4 + 1]; c += scratch[i * 4 + 2]; d += scratch[i * 4 + 3]; }
  return a;
}

// Kernel (3).  One CTA per logits row r = t*B + b (time-major, view(-1,V) of a contiguous (T,B,V)).
// The row of student logits y and teacher logits z is brought into shared memory ONCE (1-D TMA bulk
// copies when rows are 16-byte aligned) and all three passes (max, sums, gradient) run out of smem, so
// HBM traffic is exactly: read y, read z, write dy.
//   KL_r  = sum_v pT (log pT - log pS),  pS = softmax(y/Temp), pT = softmax(z/Temp)
//   CE_r  = logsumexp(y) - y[tgt]                       (tgt != PAD)
//   dy_v  = kd_coef (pS_v - pT_v) + ce_coef (softmax(y)_v - [v == tgt])
// with kd_coef = alpha*Temp/N and ce_coef = w_ce / n_valid (0 on PAD rows).
// TZ (teacher logits): float, bf16 or f16; a half-precision row is widened exactly to fp32 on its way into shared memory, so the
// arithmetic is that of the fp32 row.
template <typename TS, typename TZ, int G, bool TEMP4>
__global__ void __launch_bounds__(KD_THREADS)
kd_token_loss_kernel(const TS* __restrict__ y, const TZ* __restrict__ z, const int64_t* __restrict__ tgt,
                     int V, float inv_temp, float kd_coef, float w_ce, const int* __restrict__ n_valid_ptr,
                     TS* __restrict__ dy /* NULL: losses only (evaluation) */, float* __restrict__ row_kl, float* __restrict__ row_ce,
                     int* __restrict__ argmax_out /* NULL, or (N): argmax_v y[r, v], lowest index on ties like torch.argmax */,
                     const int* __restrict__ steps /* NULL, or the device step count of a variable-length batch */, long rows_per_step,
                     float kd_num /* alpha * Temp: kd_coef = kd_num / (*steps * rows_per_step) when steps is set */) {
  if (steps != nullptr) {
    // variable-length batch: only the first n = *steps * rows_per_step rows exist.  A row past them reads nothing and leaves zero
    // losses and a zero gradient row; the others use the KD scale of n rows.
    const long n = min((long)gridDim.x, (long)__ldg(steps) * rows_per_step);
    if ((long)blockIdx.x >= n) {
      if (dy != nullptr) for (int v = threadIdx.x; v < V; v += KD_THREADS) dy[(long)blockIdx.x * V + v] = from_f<TS>(0.f);
      if (threadIdx.x == 0) { row_kl[blockIdx.x] = 0.f; row_ce[blockIdx.x] = 0.f; }
      return;
    }
    kd_coef = kd_num / (float)n;
  }
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* zs = reinterpret_cast<float*>(smem_raw);                             // V floats
  TS* ys = reinterpret_cast<TS*>(smem_raw + align_up((size_t)V * 4, 16)); // V TS
  __shared__ __align__(8) uint64_t bar;
  __shared__ float scratch[KD_THREADS / 32 * 4];

  const int tid = threadIdx.x;
  const long r = blockIdx.x;
  const TS* yg = y + r * (long)V;
  const TZ* zg = z + r * (long)V;

  if (G == 8) {
    if (tid == 0) { mbar_init(&bar, 1); fence_barrier_init(); }
    __syncthreads();
    if constexpr (sizeof(TZ) == 4) {
      if (tid == 0) {
        mbar_arrive_expect_tx(&bar, (uint32_t)(V * 4 + V * sizeof(TS)));
        bulk_g2s(zs, zg, (uint32_t)(V * 4), &bar);
        bulk_g2s(ys, yg, (uint32_t)(V * sizeof(TS)), &bar);
      }
    } else {
      // half-precision teacher row: 16-byte loads widened into the fp32 row while the student row's bulk copy is in flight
      if (tid == 0) {
        mbar_arrive_expect_tx(&bar, (uint32_t)(V * sizeof(TS)));
        bulk_g2s(ys, yg, (uint32_t)(V * sizeof(TS)), &bar);
      }
      for (int g = tid; g < V / 8; g += KD_THREADS) { float v[8]; Vec8<TZ>::load(zg + g * 8, v); RowIO<float, 8>::store_s(zs, g * 8, v); }
      __syncthreads();
    }
    mbar_wait(&bar, 0);
  } else {
    for (int v = tid; v < V; v += KD_THREADS) { zs[v] = to_f<TZ>(zg[v]); ys[v] = yg[v]; }
    __syncthreads();
  }

  const long t64 = tgt[r];
  const bool valid = (t64 != 0) && (t64 > 0) && (t64 < V);
  const int t_idx = valid ? (int)t64 : 0;
  const float y_tgt = to_f<TS>(ys[t_idx]);
  const int groups = V / G;

  // pass 1: row maxima
  float my = -INFINITY, mz = -INFINITY;
  for (int g = tid; g < groups; g += KD_THREADS) {
    float yv[G], zv[G];
    RowIO<TS, G>::load(ys, g * G, yv);
    RowIO<float, G>::load(zs, g * G, zv);
#pragma unroll
    for (int i = 0; i < G; ++i) { my = fmaxf(my, yv[i]); mz = fmaxf(mz, zv[i]); }
  }
  my = warp_max(my); mz = warp_max(mz);
  {
    const int w = tid >> 5, l = tid & 31;
    if (l == 0) { scratch[w * 2] = my; scratch[w * 2 + 1] = mz; }
    __syncthreads();
    my = scratch[0]; mz = scratch[1];
#pragma unroll
    for (int i = 1; i < KD_THREADS / 32; ++i) { my = fmaxf(my, scratch[i * 2]); mz = fmaxf(mz, scratch[i * 2 + 1]); }
  }

  if (argmax_out != nullptr) {                 // teacher-forced prediction of this row (validate_student_model's logits.argmax(-1))
    int best = V;
    for (int v = tid; v < V; v += KD_THREADS) if (to_f<TS>(ys[v]) == my) best = min(best, v);
    for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, o));
    __shared__ int best_s[KD_THREADS / 32];
    if ((tid & 31) == 0) best_s[tid >> 5] = best;
    __syncthreads();
    if (tid == 0) { int bb = best_s[0]; for (int i = 1; i < KD_THREADS / 32; ++i) bb = min(bb, best_s[i]); argmax_out[r] = bb; }
  }

  // pass 2: partition sums; e^{z'} is written back over z (and e^{y'} over y when y is fp32)
  float sT = 0.f, sZ = 0.f, sA = 0.f, s1 = 0.f;
  for (int g = tid; g < groups; g += KD_THREADS) {
    float yv[G], zv[G];
    RowIO<TS, G>::load(ys, g * G, yv);
    RowIO<float, G>::load(zs, g * G, zv);
#pragma unroll
    for (int i = 0; i < G; ++i) {
      const float yd = yv[i] - my, zd = (zv[i] - mz) * inv_temp;
      const float ey = __expf(yd * inv_temp), ez = __expf(zd);
      float e1;
      if (TEMP4) { const float e2 = ey * ey; e1 = e2 * e2; } else { e1 = __expf(yd); }
      sT += ey; sZ += ez; sA += ez * (zd - yd * inv_temp); s1 += e1;
      zv[i] = ez; yv[i] = ey;
    }
    RowIO<float, G>::store_s(zs, g * G, zv);
    if (sizeof(TS) == 4) RowIO<float, G>::store_s(reinterpret_cast<float*>(ys), g * G, yv);
  }
  block_reduce_sum4(sT, sZ, sA, s1, scratch);

  const float inv_sT = 1.0f / sT, inv_sZ = 1.0f / sZ, inv_s1 = 1.0f / s1;
  const int n_valid = *n_valid_ptr;
  const float ce_coef = (valid && n_valid > 0) ? w_ce / (float)n_valid : 0.0f;
  if (tid == 0) {
    row_kl[r] = sA * inv_sZ - __logf(sZ) + __logf(sT);
    row_ce[r] = valid ? (__logf(s1) + my - y_tgt) : 0.0f;
  }

  // pass 3: gradient
  if (dy == nullptr) return;
  TS* dyg = dy + r * (long)V;
  const float a_s = kd_coef * inv_sT, a_t = kd_coef * inv_sZ, a_c = ce_coef * inv_s1;
  for (int g = tid; g < groups; g += KD_THREADS) {
    float yv[G], zv[G], o[G];
    RowIO<TS, G>::load(ys, g * G, yv);
    RowIO<float, G>::load(zs, g * G, zv);
#pragma unroll
    for (int i = 0; i < G; ++i) {
      float ey, e1;
      if (sizeof(TS) == 4) { ey = yv[i]; } else { ey = __expf((yv[i] - my) * inv_temp); }
      if (TEMP4) { const float e2 = ey * ey; e1 = e2 * e2; }
      else { e1 = (sizeof(TS) == 4) ? __powf(ey, 1.0f / inv_temp) : __expf(yv[i] - my); }
      float gval = a_s * ey - a_t * zv[i] + a_c * e1;
      if (g * G + i == t_idx) gval -= ce_coef;
      o[i] = gval;
    }
    RowIO<TS, G>::store_g(dyg, (long)g * G, o);
  }
}

// Merge of the per-(row, part) partials the vocabulary-head GEMM's validation epilogue leaves (gemm.cuh EvalEpi): one warp per
// logits row, lanes over the parts, fixed order.  Same outputs as the evaluation form of kd_token_loss_kernel:
//   row_kl = sA / sZ - log sZ + log sT,  row_ce = log s1 + my - y[target] (0 on PAD rows),  argmax (lowest index among equals).
__global__ void __launch_bounds__(256)
kd_eval_combine_kernel(const float* __restrict__ parts, int nparts, long N, int V, const int64_t* __restrict__ tgt, float inv_temp,
                       float* __restrict__ row_kl, float* __restrict__ row_ce, int* __restrict__ argmax_out) {
  const long r = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= N) return;
  const float4* p = reinterpret_cast<const float4*>(parts + r * (long)nparts * 8);
  float MY = -INFINITY, MZ = -INFINITY;
  for (int i = lane; i < nparts; i += 32) { const float4 a = p[2 * i]; MY = fmaxf(MY, a.x); MZ = fmaxf(MZ, a.w); }
  MY = warp_max(MY); MZ = warp_max(MZ);
  float s1 = 0.f, sT = 0.f, sZ = 0.f, sA = 0.f, ytgt = 0.f; int best = 0x7fffffff;
  for (int i = lane; i < nparts; i += 32) {
    const float4 a = p[2 * i], b = p[2 * i + 1];
    const float dy = a.x - MY, dz = (a.w - MZ) * inv_temp;          // <= 0
    const float cz = __expf(dz);
    s1 += a.y * __expf(dy); sT += a.z * __expf(dy * inv_temp); sZ += b.x * cz;
    sA += cz * (b.y + b.x * (dz - dy * inv_temp));
    ytgt += b.z;                                                    // exactly one part holds the target column, the others wrote 0
    if (a.x == MY) best = min(best, __float_as_int(b.w));
  }
  s1 = warp_sum(s1); sT = warp_sum(sT); sZ = warp_sum(sZ); sA = warp_sum(sA); ytgt = warp_sum(ytgt);
  for (int o = 16; o > 0; o >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, o));
  if (lane == 0) {
    const long t64 = tgt[r];
    const bool valid = (t64 > 0) && (t64 < V);
    row_kl[r] = sA / sZ - __logf(sZ) + __logf(sT);
    row_ce[r] = valid ? (__logf(s1) + MY - ytgt) : 0.0f;
    if (argmax_out) argmax_out[r] = best == 0x7fffffff ? 0 : best;
  }
}

// Kernel (3), default form (V % 8 == 0, V <= 16384; NCH == ceil(V/8/256) so only the last chunk can be partial): persistent CTAs (grid = SMs x resident CTAs), each looping over logits
// rows.  The NEXT row's student and teacher logits are prefetched into a double-buffered shared-memory slot by two 1-D TMA
// bulk copies on an mbarrier while the CURRENT row is processed entirely in registers: one 128-bit shared-memory read per
// 8 logits, then row maxima, partition sums and the gradient on registers (2 ex2 per logit pair), 128-bit streaming
// stores.  HBM traffic is exactly {read y, read z, write dy}; the TMA prefetch keeps ~3 rows per SM in flight.
constexpr int KDR_THREADS = 256;

template <typename TS> struct RowS;     // 8 elements from shared memory / to global memory
template <> struct RowS<bf16> {
  static __device__ __forceinline__ void load(const bf16* p, float (&v)[8]) {
    const uint4 a = *reinterpret_cast<const uint4*>(p);
    v[0] = bf16_lo(a.x); v[1] = bf16_hi(a.x); v[2] = bf16_lo(a.y); v[3] = bf16_hi(a.y);
    v[4] = bf16_lo(a.z); v[5] = bf16_hi(a.z); v[6] = bf16_lo(a.w); v[7] = bf16_hi(a.w);
  }
  static __device__ __forceinline__ void store(bf16* p, const float (&v)[8]) {
    st_na_v4(p, make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7])));
  }
};
template <> struct RowS<f16> {          // teacher rows only
  static __device__ __forceinline__ void load(const f16* p, float (&v)[8]) {
    const uint4 a = *reinterpret_cast<const uint4*>(p);
    v[0] = f16_lo(a.x); v[1] = f16_hi(a.x); v[2] = f16_lo(a.y); v[3] = f16_hi(a.y);
    v[4] = f16_lo(a.z); v[5] = f16_hi(a.z); v[6] = f16_lo(a.w); v[7] = f16_hi(a.w);
  }
};
template <> struct RowS<float> {
  static __device__ __forceinline__ void load(const float* p, float (&v)[8]) {
    const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
  static __device__ __forceinline__ void store(float* p, const float (&v)[8]) {
    st_na_v4(p, make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3])));
    st_na_v4(p + 4, make_uint4(__float_as_uint(v[4]), __float_as_uint(v[5]), __float_as_uint(v[6]), __float_as_uint(v[7])));
  }
};

constexpr int KD_SLOTS = 2;              // row slots per CTA: the TMA prefetch runs KD_SLOTS - 1 rows ahead of the math

// Unaligned rows (V % 8 != 0): row r of y / z starts anywhere inside a 16-byte word.  The bulk copy takes the enclosing
// 16-byte-aligned byte range, so element v of the row sits at slot index sh + v with sh = the row start's offset inside its
// word (0..7 bf16 / f16, 0..3 fp32).  These rebuild the 8 elements of column group g from the two (2-byte types) or three (fp32)
// 16-byte words that hold them; the shift is uniform over the CTA, so the selects below never diverge.
__device__ __forceinline__ uint32_t pick_word(const uint32_t (&u)[8], int q, int j) {      // u[q + j], q in 0..3
  return q == 0 ? u[j] : (q == 1 ? u[j + 1] : (q == 2 ? u[j + 2] : u[j + 3]));
}
template <typename T>          // bf16 or f16
__device__ __forceinline__ void load_shifted_h(const T* slot, int sh, int g, float (&v)[8]) {
  const uint4 a = reinterpret_cast<const uint4*>(slot)[g], b = reinterpret_cast<const uint4*>(slot)[g + 1];
  const uint32_t u[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  const int q = sh >> 1, bits = (sh & 1) * 16;
  uint32_t w[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) w[j] = __funnelshift_r(pick_word(u, q, j), pick_word(u, q, j + 1), bits);
#pragma unroll
  for (int j = 0; j < 4; ++j) { v[2 * j] = lo_f<T>(w[j]); v[2 * j + 1] = hi_f<T>(w[j]); }
}
__device__ __forceinline__ void load_shifted_f32(const float* slot, int sh, int g, float (&v)[8]) {
  const float4 a = reinterpret_cast<const float4*>(slot)[2 * g], b = reinterpret_cast<const float4*>(slot)[2 * g + 1],
               c = reinterpret_cast<const float4*>(slot)[2 * g + 2];
  const float f[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
#pragma unroll
  for (int k = 0; k < 8; ++k) v[k] = sh == 0 ? f[k] : (sh == 1 ? f[k + 1] : (sh == 2 ? f[k + 2] : f[k + 3]));
}
__device__ __forceinline__ void load_shifted(const bf16* slot, int sh, int g, float (&v)[8]) { load_shifted_h(slot, sh, g, v); }
__device__ __forceinline__ void load_shifted(const f16* slot, int sh, int g, float (&v)[8]) { load_shifted_h(slot, sh, g, v); }
__device__ __forceinline__ void load_shifted(const float* slot, int sh, int g, float (&v)[8]) { load_shifted_f32(slot, sh, g, v); }

// Body of kernel (3)'s default form.  UNALIGNED = false: V % 8 == 0, 16-byte aligned y / z / dy, dy pitch V (ld == V).
// UNALIGNED = true (bf16 student logits, any V): y and z keep pitch V and any alignment; each row is fetched by bulk copies of
// its enclosing 16-byte-aligned ranges, except a row whose enclosing range would reach outside [y, y + N*V) or [z, z + N*V)
// (the first / last row or two): that one is read with guarded plain loads.  Columns >= V are left out of the maxima, the
// sums and the CE term.  dy has pitch ld (ld % 8 == 0, 16-byte aligned): 16-byte stores, columns V..roundup(V,8)-1 written
// as exact zeros.
// TZ: the teacher logits' type (float, bf16 or f16).  A slot holds V * sizeof(TZ) teacher bytes; each 16-byte word of a
// half-precision row gives 8 logits, widened exactly to fp32 in registers.
template <typename TS, typename TZ, int NCH, bool TEMP4, bool UNALIGNED>
__device__ __forceinline__ void kd_token_pipe_body(const TS* __restrict__ y, const TZ* __restrict__ z, const int64_t* __restrict__ tgt,
                                                   long N, int V, long ld, float inv_temp, float temperature, float kd_coef, float w_ce,
                                                   const int* __restrict__ n_valid_ptr, TS* __restrict__ dy, float* __restrict__ row_kl,
                                                   float* __restrict__ row_ce, const int* __restrict__ steps, long rows_per_step, float kd_num) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[KD_SLOTS];
  __shared__ float scratch[KDR_THREADS / 32 * 4];
  const int Vp = (V + 7) & ~7;
  // slot bytes: both multiples of 16; the unaligned form holds the enclosing ranges plus the word the last group reads past them
  const size_t zbytes = UNALIGNED ? (size_t)(Vp + 16 / sizeof(TZ)) * sizeof(TZ) : (size_t)V * sizeof(TZ);
  const size_t ybytes = UNALIGNED ? (size_t)(Vp + 8) * sizeof(TS) : (size_t)V * sizeof(TS);
  const size_t slot = zbytes + ybytes;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int groups = UNALIGNED ? (Vp >> 3) : (V >> 3);
  const int n_valid = *n_valid_ptr;
  // variable-length batch (steps != null): rows [n, N) are past the batch.  They are never fetched (the enclosing 16-byte range of
  // row n - 1 in the unaligned form may reach into row n; those columns are replaced by the sentinel below and never used) and get
  // zero losses and a zero gradient row; the KD scale is that of n rows.
  long n = N;
  if (steps != nullptr) { n = min(N, (long)__ldg(steps) * rows_per_step); kd_coef = kd_num / (float)n; }
  const uintptr_t y_end = (uintptr_t)(y + N * (long)V), z_end = (uintptr_t)(z + N * (long)V);
  // enclosing 16-byte range [lo, hi) of row `row` of y / z, and whether both lie inside their tensors
  auto y_lo = [&](long row) { return (uintptr_t)(y + row * (long)V) & ~(uintptr_t)15; };
  auto z_lo = [&](long row) { return (uintptr_t)(z + row * (long)V) & ~(uintptr_t)15; };
  auto y_hi = [&](long row) { return ((uintptr_t)(y + (row + 1) * (long)V) + 15) & ~(uintptr_t)15; };
  auto z_hi = [&](long row) { return ((uintptr_t)(z + (row + 1) * (long)V) + 15) & ~(uintptr_t)15; };
  auto bulk_row = [&](long row) {
    return !UNALIGNED || (y_lo(row) >= (uintptr_t)y && y_hi(row) <= y_end && z_lo(row) >= (uintptr_t)z && z_hi(row) <= z_end);
  };

  auto issue = [&](long row, int sidx) {       // thread 0 only
    unsigned char* dst = smem_raw + (size_t)sidx * slot;
    if constexpr (!UNALIGNED) {
      mbar_arrive_expect_tx(&full_bar[sidx], (uint32_t)slot);
      bulk_g2s(dst, z + row * (long)V, (uint32_t)zbytes, &full_bar[sidx]);
      bulk_g2s(dst + zbytes, y + row * (long)V, (uint32_t)ybytes, &full_bar[sidx]);
    } else if (bulk_row(row)) {
      const uint32_t zb = (uint32_t)(z_hi(row) - z_lo(row)), yb = (uint32_t)(y_hi(row) - y_lo(row));
      mbar_arrive_expect_tx(&full_bar[sidx], zb + yb);
      bulk_g2s(dst, (const void*)z_lo(row), zb, &full_bar[sidx]);
      bulk_g2s(dst + zbytes, (const void*)y_lo(row), yb, &full_bar[sidx]);
    } else {
      mbar_arrive(&full_bar[sidx]);            // guarded row: nothing to copy, but the slot's phase still completes
    }
  };
  if (tid == 0) { for (int i = 0; i < KD_SLOTS; ++i) mbar_init(&full_bar[i], 1); fence_barrier_init(); }
  __syncthreads();
  const long r0 = blockIdx.x, stride = gridDim.x;
  if (tid == 0) {
    for (int i = 0; i < KD_SLOTS; ++i) if (r0 + i * stride < n) issue(r0 + i * stride, i);
  }

  int it = 0;
  for (long r = r0; r < n; r += stride, ++it) {
    const int sidx = it % KD_SLOTS; const uint32_t ph = (it / KD_SLOTS) & 1;
    const TZ* zs = reinterpret_cast<const TZ*>(smem_raw + (size_t)sidx * slot);
    const TS* ys = reinterpret_cast<const TS*>(smem_raw + (size_t)sidx * slot + zbytes);
    mbar_wait(&full_bar[sidx], ph);
    float yv[NCH][8], zv[NCH][8];
    bool bulk = true;
    int sy = 0, sz = 0;
    if constexpr (!UNALIGNED) {
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        const int g = tid + i * KDR_THREADS;
        if (i < NCH - 1 || g < groups) { RowS<TS>::load(ys + g * 8, yv[i]); RowS<TZ>::load(zs + g * 8, zv[i]); }
      }
    } else {
      const TS* yr = y + r * (long)V;
      const TZ* zr = z + r * (long)V;
      bulk = bulk_row(r);
      if (bulk) {
        sy = (int)(((uintptr_t)yr & 15) / sizeof(TS)); sz = (int)(((uintptr_t)zr & 15) / sizeof(TZ));
#pragma unroll
        for (int i = 0; i < NCH; ++i) {
          const int g = tid + i * KDR_THREADS;
          if (i < NCH - 1 || g < groups) { load_shifted(ys, sy, g, yv[i]); load_shifted(zs, sz, g, zv[i]); }
        }
      } else {
#pragma unroll
        for (int i = 0; i < NCH; ++i) {
          const int g = tid + i * KDR_THREADS;
          if (i < NCH - 1 || g < groups) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int c = g * 8 + j;
              yv[i][j] = c < V ? to_f<TS>(yr[c]) : 0.f; zv[i][j] = c < V ? to_f<TZ>(zr[c]) : 0.f;
            }
          }
        }
      }
      // columns V..Vp-1 (the last group only) hold a neighbouring row or nothing.  A finite sentinel far below any logit keeps
      // them out of the maxima and gives them e^x = 0 in every sum (and a gradient of exactly 0) without a branch per element;
      // unlike -inf it never forms inf - inf in the KL term, and (x - max) / Temp stays finite for any Temp > 1e-8.
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        const int g = tid + i * KDR_THREADS;
        if (g == groups - 1) {
#pragma unroll
          for (int j = 0; j < 8; ++j) if (g * 8 + j >= V) { yv[i][j] = -1.0e30f; zv[i][j] = -1.0e30f; }
        }
      }
    }
    const long t64 = tgt[r];
    const bool valid = (t64 > 0) && (t64 < V);
    const int t_idx = valid ? (int)t64 : -1;
    float y_tgt = 0.f, z_tgt = 0.f;
    if (valid) {
      if (bulk) { y_tgt = to_f<TS>(ys[sy + t_idx]); z_tgt = to_f<TZ>(zs[sz + t_idx]); }
      else { y_tgt = to_f<TS>(y[r * (long)V + t_idx]); z_tgt = to_f<TZ>(z[r * (long)V + t_idx]); }
    }
    __syncthreads();                           // every thread has taken its groups out of the slot ...
    if (tid == 0 && r + KD_SLOTS * stride < n) issue(r + KD_SLOTS * stride, sidx);      // ... so a later row can land in it

    // phase 1: row maxima
    float my = -INFINITY, mz = -INFINITY;
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
      if (i < NCH - 1 || tid + i * KDR_THREADS < groups) {
#pragma unroll
        for (int j = 0; j < 8; ++j) { my = fmaxf(my, yv[i][j]); mz = fmaxf(mz, zv[i][j]); }
      }
    }
    my = warp_max(my); mz = warp_max(mz);
    if (lane == 0) { scratch[warp * 2] = my; scratch[warp * 2 + 1] = mz; }
    __syncthreads();
    my = scratch[0]; mz = scratch[1];
#pragma unroll
    for (int i = 1; i < KDR_THREADS / 32; ++i) { my = fmaxf(my, scratch[i * 2]); mz = fmaxf(mz, scratch[i * 2 + 1]); }
    __syncthreads();

    // phase 2: exponentials (kept in the same registers) and the four partition sums.  Everything is in log2 units:
    // yd2 = (y - my)/Temp * log2(e) is ONE FFMA, e^x is ONE ex2.approx.ftz; the ln(2) factor of sA is applied once per row.
    const float cy = inv_temp * 1.4426950408889634f;
    const float my_c = -my * cy, mz_c = -mz * cy;
    float sT = 0.f, sZ = 0.f, sA = 0.f, s1 = 0.f;
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
      if (i < NCH - 1 || tid + i * KDR_THREADS < groups) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float yd2 = fmaf(yv[i][j], cy, my_c), zd2 = fmaf(zv[i][j], cy, mz_c);
          const float ey = ex2_ftz(yd2), ez = ex2_ftz(zd2);
          sT += ey; sZ += ez; sA = fmaf(ez, zd2 - yd2, sA);
          if (TEMP4) { const float e2 = ey * ey; s1 = fmaf(e2, e2, s1); }
          else s1 += ex2_ftz((yv[i][j] - my) * 1.4426950408889634f);
          yv[i][j] = ey; zv[i][j] = ez;
        }
      }
    }
    sT = warp_sum(sT); sZ = warp_sum(sZ); sA = warp_sum(sA); s1 = warp_sum(s1);
    if (lane == 0) { scratch[warp * 4] = sT; scratch[warp * 4 + 1] = sZ; scratch[warp * 4 + 2] = sA; scratch[warp * 4 + 3] = s1; }
    __syncthreads();
    sT = sZ = sA = s1 = 0.f;
#pragma unroll
    for (int i = 0; i < KDR_THREADS / 32; ++i) { sT += scratch[i * 4]; sZ += scratch[i * 4 + 1]; sA += scratch[i * 4 + 2]; s1 += scratch[i * 4 + 3]; }
    sA *= 0.6931471805599453f;

    const float inv_sT = 1.0f / sT, inv_sZ = 1.0f / sZ, inv_s1 = 1.0f / s1;
    const float ce_coef = (valid && n_valid > 0) ? w_ce / (float)n_valid : 0.0f;
    if (tid == 0) {
      row_kl[r] = sA * inv_sZ - __logf(sZ) + __logf(sT);
      row_ce[r] = valid ? (__logf(s1) + my - y_tgt) : 0.0f;
    }

    // phase 3: gradient, straight from registers to 128-bit streaming stores.  The one-hot term of the target logit is
    // applied by the thread that owns that logit with one scalar store after its vector store (same thread, same address).
    TS* dyg = dy + r * ld;
    const float a_s = kd_coef * inv_sT, a_t = -kd_coef * inv_sZ, a_c = ce_coef * inv_s1;
    const int t_grp = t_idx >> 3;               // -1 on PAD rows: matches no group
    float g_t = 0.f;
    if (valid) {
      const float ey_t = ex2_ftz(fmaf(y_tgt, cy, my_c)), ez_t = ex2_ftz(fmaf(z_tgt, cy, mz_c));
      float e1_t;
      if (TEMP4) { const float e2 = ey_t * ey_t; e1_t = e2 * e2; } else { e1_t = ex2_ftz((y_tgt - my) * 1.4426950408889634f); }
      g_t = fmaf(a_s, ey_t, fmaf(a_t, ez_t, a_c * e1_t)) - ce_coef;
    }
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
      const int g = tid + i * KDR_THREADS;
      if (i < NCH - 1 || g < groups) {
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float ey = yv[i][j];
          float e1;
          if (TEMP4) { const float e2 = ey * ey; e1 = e2 * e2; } else { e1 = __powf(ey, temperature); }
          o[j] = fmaf(a_s, ey, fmaf(a_t, zv[i][j], a_c * e1));
        }
        RowS<TS>::store(dyg + g * 8, o);
        if (g == t_grp) dyg[t_idx] = from_f<TS>(g_t);
      }
    }
  }
  for (long r = n + blockIdx.x; r < N; r += gridDim.x) {       // rows past a variable-length batch (none otherwise)
    const float zero[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int g = tid; g < groups; g += KDR_THREADS) RowS<TS>::store(dy + r * ld + g * 8, zero);
    if (tid == 0) { row_kl[r] = 0.f; row_ce[r] = 0.f; }
  }
}

template <typename TS, typename TZ, int NCH, bool TEMP4>
__global__ void __launch_bounds__(KDR_THREADS, (NCH <= 3 ? 3 : (NCH <= 5 ? 2 : 1)))
kd_token_loss_pipe_kernel(const TS* __restrict__ y, const TZ* __restrict__ z, const int64_t* __restrict__ tgt,
                          long N, int V, float inv_temp, float temperature, float kd_coef, float w_ce, const int* __restrict__ n_valid_ptr,
                          TS* __restrict__ dy, float* __restrict__ row_kl, float* __restrict__ row_ce,
                          const int* __restrict__ steps, long rows_per_step, float kd_num) {
  kd_token_pipe_body<TS, TZ, NCH, TEMP4, false>(y, z, tgt, N, V, V, inv_temp, temperature, kd_coef, w_ce, n_valid_ptr, dy, row_kl, row_ce,
                                            steps, rows_per_step, kd_num);
}

// The form for bf16 rows of any length (V % 8 != 0 or unaligned logits) with dlogits of pitch ld (ld % 8 == 0).
template <typename TZ, int NCH, bool TEMP4>
__global__ void __launch_bounds__(KDR_THREADS, (NCH <= 3 ? 3 : (NCH <= 5 ? 2 : 1)))
kd_token_loss_pipe_unaligned_kernel(const bf16* __restrict__ y, const TZ* __restrict__ z, const int64_t* __restrict__ tgt,
                                    long N, int V, long ld, float inv_temp, float temperature, float kd_coef, float w_ce,
                                    const int* __restrict__ n_valid_ptr, bf16* __restrict__ dy, float* __restrict__ row_kl,
                                    float* __restrict__ row_ce, const int* __restrict__ steps, long rows_per_step, float kd_num) {
  kd_token_pipe_body<bf16, TZ, NCH, TEMP4, true>(y, z, tgt, N, V, ld, inv_temp, temperature, kd_coef, w_ce, n_valid_ptr, dy, row_kl, row_ce,
                                             steps, rows_per_step, kd_num);
}

// validate_student_model's monitoring metric (reference src/distillation_utils.py:398-409, compute_bleu_score): per sample,
//   |set(pred \ {PAD,START,END}) ∩ set(target \ {PAD,START,END})| / |set(target \ {PAD,START,END})|   (0 if the target set is empty).
// Token ids stand for words (vocab.itos is injective).  One warp per sample, O(T^2) comparisons (T = caption length).
__global__ void __launch_bounds__(128)
bleu1_kernel(const int* __restrict__ pred /*(T,B)*/, const int64_t* __restrict__ tgt /*(T,B)*/, int T, int B, float* __restrict__ out /*(B)*/) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  int n_set = 0, n_hit = 0;
  for (int i = lane; i < T; i += 32) {
    const long tok = tgt[(long)i * B + b];
    if (tok == 0 || tok == 1 || tok == 2) continue;
    bool first = true;
    for (int j = 0; j < i; ++j) if (tgt[(long)j * B + b] == tok) { first = false; break; }
    if (!first) continue;
    ++n_set;
    for (int j = 0; j < T; ++j) if ((long)pred[(long)j * B + b] == tok) { ++n_hit; break; }
  }
  for (int o = 16; o > 0; o >>= 1) { n_set += __shfl_xor_sync(0xffffffffu, n_set, o); n_hit += __shfl_xor_sync(0xffffffffu, n_hit, o); }
  if (lane == 0) out[b] = n_set > 0 ? (float)n_hit / (float)n_set : 0.f;
}

__global__ void count_valid_kernel(const int64_t* __restrict__ tgt, long n, int V, int* __restrict__ out) {
  __shared__ int part[32];
  int c = 0;
  for (long i = threadIdx.x; i < n; i += blockDim.x) { const long t = tgt[i]; c += (t > 0 && t < V) ? 1 : 0; }
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) { int s = 0; for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += part[i]; *out = s; }
}
// Kernel (4).  blockIdx < n_feat_blocks : feature KD for sample b (256 threads);  above : hidden KD, one warp per
// (t,b) row.  Gradients already carry beta / gamma; loss partials go to workspace for the finalize kernel.
// TZ: the teacher hidden states' type (float, bf16 or f16), widened exactly to fp32 on load.  The teacher features ft stay fp32:
// they are the projector's output, and dft flows back into it.
template <typename TF, typename TH, typename TZ>
__global__ void __launch_bounds__(256)
aux_loss_kernel(const TF* __restrict__ fs, const float* __restrict__ ft, int n_feat_blocks /*B or 0*/, int B, int Ss, int St, int E,
                const TH* __restrict__ hs, const TZ* __restrict__ ht, int n_hid_rows /*Th*B*/, int n_all_rows /*T*B*/,
                int H, int Th, float beta, float gamma,
                float* __restrict__ dfs, float* __restrict__ dft, TH* __restrict__ dhs,
                float* __restrict__ feat_part /*B*2*/, float* __restrict__ hid_part /*n_hid_rows*2*/,
                const int* __restrict__ steps /* null, or the device step count of a variable-length batch */) {
  extern __shared__ __align__(16) float sm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = blockDim.x >> 5;
  if ((int)blockIdx.x < n_feat_blocks) {
    const int b = blockIdx.x;
    const TF* S = fs + (long)b * Ss * E;
    const float* Tp = ft + (long)b * St * E;
    float* dg = sm;                          // E    delta of global means            (the E-sized arrays first: 16-byte aligned)
    float* da = dg + E;                      // E    delta of attention-pooled
    float* part = da + E;                    // [nwarp = 8][2][E] per-warp column partials
    float* ps = part + (long)8 * 2 * E;      // Ss   softmax weights (student)
    float* pt = ps + Ss;                     // St
    float* qs = pt + St;                     // Ss
    float* qt = qs + Ss;                     // St
    __shared__ float red[16];
    // Every pass reads the two token matrices with 16-byte accesses, warp per token row, lanes over 8-column chunks (E % 8 == 0).
    // Pass 1 comes from HBM, the later ones from L2 (75 KB per sample).
    const int nch = E >> 3;
    // 1. token row sums
    for (int l = warp; l < Ss; l += nwarp) {
      float a = 0.f;
      for (int c = lane; c < nch; c += 32) { float v[8]; Vec8<TF>::load(S + (long)l * E + c * 8, v); a += ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7])); }
      a = warp_sum(a); if (lane == 0) ps[l] = a;
    }
    for (int l = warp; l < St; l += nwarp) {
      float a = 0.f;
      for (int c = lane; c < nch; c += 32) { float v[8]; Vec8<float>::load(Tp + (long)l * E + c * 8, v); a += ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7])); }
      a = warp_sum(a); if (lane == 0) pt[l] = a;
    }
    __syncthreads();
    // 2. softmax over tokens (warp 0: student, warp 1: teacher)
    if (warp < 2) {
      float* p = warp == 0 ? ps : pt; const int n = warp == 0 ? Ss : St;
      float m = -INFINITY; for (int l = lane; l < n; l += 32) m = fmaxf(m, p[l]); m = warp_max(m);
      float s = 0.f; for (int l = lane; l < n; l += 32) { const float e = expf(p[l] - m); p[l] = e; s += e; } s = warp_sum(s);
      const float inv = 1.0f / s; for (int l = lane; l < n; l += 32) p[l] *= inv;
    }
    __syncthreads();
    // 3. pooled vectors: each warp sums its rows into per-column partials (global mean and attention-pooled, student minus teacher),
    //    the partials of the 8 warps are combined through shared memory
    for (int c = lane; c < nch; c += 32) {
      float g8[8], a8[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) { g8[k] = 0.f; a8[k] = 0.f; }
      const float is = 1.0f / (float)Ss, it = 1.0f / (float)St;
      for (int l = warp; l < Ss; l += nwarp) {
        float v[8]; Vec8<TF>::load(S + (long)l * E + c * 8, v);
        const float w = ps[l];
#pragma unroll
        for (int k = 0; k < 8; ++k) { g8[k] = fmaf(v[k], is, g8[k]); a8[k] = fmaf(w, v[k], a8[k]); }
      }
      for (int l = warp; l < St; l += nwarp) {
        float v[8]; Vec8<float>::load(Tp + (long)l * E + c * 8, v);
        const float w = pt[l];
#pragma unroll
        for (int k = 0; k < 8; ++k) { g8[k] = fmaf(-v[k], it, g8[k]); a8[k] = fmaf(-w, v[k], a8[k]); }
      }
      Vec8<float>::store(part + ((long)warp * 2 + 0) * E + c * 8, g8);
      Vec8<float>::store(part + ((long)warp * 2 + 1) * E + c * 8, a8);
    }
    __syncthreads();
    float acc_g = 0.f, acc_a = 0.f;
    for (int e = tid; e < E; e += blockDim.x) {
      float d_g = 0.f, d_a = 0.f;
      for (int w = 0; w < nwarp; ++w) { d_g += part[((long)w * 2 + 0) * E + e]; d_a += part[((long)w * 2 + 1) * E + e]; }
      dg[e] = d_g; da[e] = d_a; acc_g += d_g * d_g; acc_a += d_a * d_a;
    }
    acc_g = warp_sum(acc_g); acc_a = warp_sum(acc_a);
    if (lane == 0) { red[warp * 2] = acc_g; red[warp * 2 + 1] = acc_a; }
    __syncthreads();
    if (tid == 0) { float g = 0.f, a = 0.f; for (int i = 0; i < nwarp; ++i) { g += red[i * 2]; a += red[i * 2 + 1]; } feat_part[b * 2] = g; feat_part[b * 2 + 1] = a; }
    // 4. gradients
    const float inv_be = 1.0f / ((float)B * (float)E);
    const float ca = 0.4f * 2.0f * inv_be, cg = 0.6f * 2.0f * inv_be;
    for (int l = warp; l < Ss; l += nwarp) {
      float a = 0.f;
      for (int c = lane; c < nch; c += 32) {
        float v[8], d8[8]; Vec8<TF>::load(S + (long)l * E + c * 8, v); Vec8<float>::load(da + c * 8, d8);
#pragma unroll
        for (int k = 0; k < 8; ++k) a = fmaf(d8[k], v[k], a);
      }
      a = warp_sum(a); if (lane == 0) qs[l] = ca * a;
    }
    for (int l = warp; l < St; l += nwarp) {
      float a = 0.f;
      for (int c = lane; c < nch; c += 32) {
        float v[8], d8[8]; Vec8<float>::load(Tp + (long)l * E + c * 8, v); Vec8<float>::load(da + c * 8, d8);
#pragma unroll
        for (int k = 0; k < 8; ++k) a = fmaf(d8[k], v[k], a);
      }
      a = warp_sum(a); if (lane == 0) qt[l] = ca * a;
    }
    __syncthreads();
    float qsbar = 0.f, qtbar = 0.f;
    for (int l = 0; l < Ss; ++l) qsbar += ps[l] * qs[l];
    for (int l = 0; l < St; ++l) qtbar += pt[l] * qt[l];
    const int E4 = E >> 2;
    if (dfs != nullptr) {
      float4* D = reinterpret_cast<float4*>(dfs + (long)b * Ss * E);
      for (int i = tid; i < Ss * E4; i += blockDim.x) {
        const int l = i / E4, e = (i - l * E4) * 4;
        const float4 g4 = *reinterpret_cast<const float4*>(dg + e), a4 = *reinterpret_cast<const float4*>(da + e);
        const float k1 = cg / (float)Ss, k2 = ca * ps[l], k3 = ps[l] * (qs[l] - qsbar);
        D[i] = make_float4(beta * (k1 * g4.x + k2 * a4.x + k3), beta * (k1 * g4.y + k2 * a4.y + k3), beta * (k1 * g4.z + k2 * a4.z + k3), beta * (k1 * g4.w + k2 * a4.w + k3));
      }
    }
    if (dft != nullptr) {
      float4* D = reinterpret_cast<float4*>(dft + (long)b * St * E);
      for (int i = tid; i < St * E4; i += blockDim.x) {
        const int l = i / E4, e = (i - l * E4) * 4;
        const float4 g4 = *reinterpret_cast<const float4*>(dg + e), a4 = *reinterpret_cast<const float4*>(da + e);
        const float k1 = cg / (float)St, k2 = ca * pt[l], k3 = pt[l] * (qt[l] - qtbar);
        D[i] = make_float4(-beta * (k1 * g4.x + k2 * a4.x + k3), -beta * (k1 * g4.y + k2 * a4.y + k3), -beta * (k1 * g4.z + k2 * a4.z + k3), -beta * (k1 * g4.w + k2 * a4.w + k3));
      }
    }
  } else {
    if (hs == nullptr) return;
    const long row = (long)(blockIdx.x - n_feat_blocks) * nwarp + warp;
    if (row >= n_all_rows) return;
    const TH* s = hs + row * H;
    TH* d = dhs ? dhs + row * H : nullptr;
    // variable-length batch: the teacher's list and the student's steps end at *steps; the steps past it are not read, have no
    // loss (zero partials) and a zero gradient, and the mean over steps divides by the steps that are left
    int th = Th;
    if (steps != nullptr) th = min(Th, max(__ldg(steps), 0));
    if (row >= (long)th * B) {                   // student steps beyond the teacher's list: no loss, zero grad
      if (d) for (int h = lane; h < H; h += 32) d[h] = from_f<TH>(0.f);
      if (row < n_hid_rows && lane == 0) { hid_part[row * 2] = 0.f; hid_part[row * 2 + 1] = 0.f; }
      return;
    }
    const TZ* t = ht + row * H;
    float sq = 0.f, dot = 0.f, ns = 0.f, nt = 0.f;
    constexpr int HC = 2;                                   // H <= 512: the row stays in registers between the two passes
    const bool in_regs = (H & 7) == 0 && H <= HC * 256;
    float sa[HC][8], tc[HC][8];
    if (in_regs) {
#pragma unroll
      for (int c = 0; c < HC; ++c) {
        const int ch = lane + 32 * c;
        if (ch * 8 < H) {
          Vec8<TH>::load(s + ch * 8, sa[c]); Vec8<TZ>::load(t + ch * 8, tc[c]);
#pragma unroll
          for (int k = 0; k < 8; ++k) { const float a = sa[c][k], cc = tc[c][k], df = a - cc; sq += df * df; dot += a * cc; ns += a * a; nt += cc * cc; }
        }
      }
    } else {
      for (int h = lane; h < H; h += 32) { const float a = to_f<TH>(s[h]), c = to_f<TZ>(t[h]); const float df = a - c; sq += df * df; dot += a * c; ns += a * a; nt += c * c; }
    }
    sq = warp_sum(sq); dot = warp_sum(dot); ns = warp_sum(ns); nt = warp_sum(nt);
    const float eps = 1e-12f;
    const float nse = ns + eps, nte = nt + eps;
    const float inv_norm = rsqrtf(nse * nte);
    const float cosv = dot * inv_norm;
    if (lane == 0) { hid_part[row * 2] = sq; hid_part[row * 2 + 1] = 1.0f - cosv; }
    if (d) {
      const float c_mse = gamma / (float)th * 0.7f * 2.0f / ((float)B * (float)H);
      const float c_cos = gamma / (float)th * 0.3f / (float)B;
      if (in_regs) {
        const float k_a = cosv / nse;
#pragma unroll
        for (int c = 0; c < HC; ++c) {
          const int ch = lane + 32 * c;
          if (ch * 8 < H) {
            float o8[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) o8[k] = c_mse * (sa[c][k] - tc[c][k]) - c_cos * (tc[c][k] * inv_norm - k_a * sa[c][k]);
            Vec8<TH>::store(d + ch * 8, o8);
          }
        }
      } else {
        for (int h = lane; h < H; h += 32) {
          const float a = to_f<TH>(s[h]), c = to_f<TZ>(t[h]);
          d[h] = from_f<TH>(c_mse * (a - c) - c_cos * (c * inv_norm - cosv * a / nse));
        }
      }
    }
  }
}

// Deterministic fixed-order reduction of all loss partials -> out5 = {total, ce, token_kd, feature_kd, hidden_kd}.
__global__ void __launch_bounds__(1024)
loss_finalize_kernel(const float* __restrict__ row_kl, const float* __restrict__ row_ce, long N, const int* __restrict__ n_valid_ptr,
                     const float* __restrict__ feat_part, int B, int E, int has_feat,
                     const float* __restrict__ hid_part, long n_hid_rows, int H, int Th, int has_hid,
                     float temperature, float alpha, float beta, float gamma, float w_ce, float ce_mult, float* __restrict__ out5,
                     const int* __restrict__ steps /* null, or the device step count: token KD over steps*B rows, hidden KD over min(Th, steps) steps */) {
  __shared__ double red[32][5];
  double kl = 0, ce = 0, fg = 0, fa = 0, hm = 0, hc = 0;
  for (long i = threadIdx.x; i < N; i += blockDim.x) { kl += row_kl[i]; ce += row_ce[i]; }
  if (has_feat) for (long i = threadIdx.x; i < B; i += blockDim.x) { fg += feat_part[i * 2]; fa += feat_part[i * 2 + 1]; }
  if (has_hid) for (long i = threadIdx.x; i < n_hid_rows; i += blockDim.x) { hm += hid_part[i * 2]; hc += hid_part[i * 2 + 1]; }
  double v[5] = {kl, ce, 0.6 * fg + 0.4 * fa, hm, hc};
  for (int k = 0; k < 5; ++k) for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
  if ((threadIdx.x & 31) == 0) for (int k = 0; k < 5; ++k) red[threadIdx.x >> 5][k] = v[k];
  __syncthreads();
  if (threadIdx.x == 0) {
    double s[5] = {0, 0, 0, 0, 0};
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) for (int k = 0; k < 5; ++k) s[k] += red[w][k];
    const int nv = *n_valid_ptr;
    long n = N; int th = Th;                   // the partials of rows / steps past a variable-length batch are zeros
    if (steps != nullptr) { n = min(N, (long)*steps * B); th = min(Th, *steps); }
    const double kd_l = (double)temperature * temperature * s[0] / (double)n;
    const double ce_l = s[1] * (double)ce_mult / (double)nv;                       // 0/0 -> NaN like the reference when every target is PAD
    const double ft_l = has_feat ? s[2] / ((double)B * E) : 0.0;
    const double hd_l = has_hid ? (0.7 * s[3] / ((double)B * H) + 0.3 * s[4] / (double)B) / (double)th : 0.0;
    out5[0] = (float)((double)w_ce * ce_l + (double)alpha * kd_l + (double)beta * ft_l + (double)gamma * hd_l);
    out5[1] = (float)ce_l; out5[2] = (float)kd_l; out5[3] = (float)ft_l; out5[4] = (float)hd_l;
  }
}

// y *= *scale (device scalar): applies autograd's incoming grad_output to a precomputed gradient; 16-byte accesses.
template <typename T>
__global__ void __launch_bounds__(256) scale_inplace_kernel(T* __restrict__ p, long n, const float* __restrict__ scale) {
  const float s = *scale;
  constexpr int PER = 16 / (int)sizeof(T);
  const long nvec = (((uintptr_t)p) % 16 == 0) ? n / PER : 0;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long)gridDim.x * blockDim.x) {
    uint4 v = reinterpret_cast<uint4*>(p)[i];
    if (sizeof(T) == 2) {
      v.x = pack_bf16(bf16_lo(v.x) * s, bf16_hi(v.x) * s); v.y = pack_bf16(bf16_lo(v.y) * s, bf16_hi(v.y) * s);
      v.z = pack_bf16(bf16_lo(v.z) * s, bf16_hi(v.z) * s); v.w = pack_bf16(bf16_lo(v.w) * s, bf16_hi(v.w) * s);
    } else {
      v.x = __float_as_uint(__uint_as_float(v.x) * s); v.y = __float_as_uint(__uint_as_float(v.y) * s);
      v.z = __float_as_uint(__uint_as_float(v.z) * s); v.w = __float_as_uint(__uint_as_float(v.w) * s);
    }
    reinterpret_cast<uint4*>(p)[i] = v;
  }
  for (long i = nvec * PER + (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) p[i] = from_f<T>(to_f<T>(p[i]) * s);
}

}  // namespace b2c
