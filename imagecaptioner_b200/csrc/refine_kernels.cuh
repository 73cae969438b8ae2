// Kernels for the two modules either side of the decoder (SURVEY.md §8f rows 1 and 2):
//   AttentionRefinement  (reference src/student_model.py:72-118): post-norm block  x1 = LN(x + MHA(x)),  out = LN(x1 + FFN(x1))
//   FeatureProjector     (reference src/distillation_utils.py:203-252): LN(Drop(ReLU(Linear(x)))) then AdaptiveAvgPool1d over tokens
// The dense contractions run on the tcgen05 GEMM of gemm.cuh; this file holds what sits between them.
#pragma once
#include "common.cuh"

namespace b2c {

__device__ __forceinline__ float4 ld_nc_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
// Converting copy in -> out.  TI = float (the general case), or bf16 / f16 (teacher features handed to the projector in half
// precision: 16-byte loads of 8 elements, widened exactly to fp32 and rounded to T like an fp32 input would be).
template <typename T, typename TI = float>
__global__ void __launch_bounds__(256) cast_f32_kernel(const TI* __restrict__ in, T* __restrict__ out, long n) {
  const long n8 = ((((uintptr_t)in) % 16 == 0) && (((uintptr_t)out) % 16 == 0)) ? (n >> 3) : 0;
  const long stride = (long)gridDim.x * blockDim.x;
  if constexpr (sizeof(TI) == 2) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
      float v[8];
      Vec8<TI>::load(in + i * 8, v);
      if (sizeof(T) == 2) *reinterpret_cast<uint4*>(out + i * 8) = make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]), pack_bf16(v[6], v[7]));
      else { reinterpret_cast<float4*>(out + i * 8)[0] = make_float4(v[0], v[1], v[2], v[3]); reinterpret_cast<float4*>(out + i * 8)[1] = make_float4(v[4], v[5], v[6], v[7]); }
    }
    for (long i = n8 * 8 + (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = from_f<T>(to_f<TI>(in[i]));
    return;
  }
  // two 8-element groups per thread and iteration, all four 16-byte loads issued before the stores
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += 2 * stride) {
    const long i2 = i + stride;
    const bool two = i2 < n8;
    const float4 a = ld_nc_f4(reinterpret_cast<const float4*>(in) + 2 * i), b = ld_nc_f4(reinterpret_cast<const float4*>(in) + 2 * i + 1);
    float4 c = a, d = b;
    if (two) { c = ld_nc_f4(reinterpret_cast<const float4*>(in) + 2 * i2); d = ld_nc_f4(reinterpret_cast<const float4*>(in) + 2 * i2 + 1); }
    if (sizeof(T) == 2) {
      *reinterpret_cast<uint4*>(out + i * 8) = make_uint4(pack_bf16(a.x, a.y), pack_bf16(a.z, a.w), pack_bf16(b.x, b.y), pack_bf16(b.z, b.w));
      if (two) *reinterpret_cast<uint4*>(out + i2 * 8) = make_uint4(pack_bf16(c.x, c.y), pack_bf16(c.z, c.w), pack_bf16(d.x, d.y), pack_bf16(d.z, d.w));
    } else {
      reinterpret_cast<float4*>(out + i * 8)[0] = a; reinterpret_cast<float4*>(out + i * 8)[1] = b;
      if (two) { reinterpret_cast<float4*>(out + i2 * 8)[0] = c; reinterpret_cast<float4*>(out + i2 * 8)[1] = d; }
    }
  }
  for (long i = n8 * 8 + (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) out[i] = from_f<T>(in[i]);
}
// ------------------------------------------------------------------ LayerNorm over the last dim (eps inside the sqrt, biased variance)
// One warp per row; lane owns 8-element chunks lane, lane+32 (E % 8 == 0, E <= 512): coalesced 16-byte accesses.
constexpr int LN_THREADS = 256;
constexpr int LN_MAXC = 2;          // kernels are templated on NC = ceil(E / 256) <= LN_MAXC chunks per lane

// x and res may differ in type: the residual stream of the refinement block is kept in fp32 also in bf16 mode (x = the fp32 block
// input / the fp32 copy of LN1's output, res = the bf16 branch output), like torch.autocast does (LayerNorm runs in fp32 there).
template <typename TX, typename TR, int NC>
__device__ __forceinline__ void ln_load_row(const TX* x, const TR* res, long r, int E, int nch, int lane, float (&v)[NC][8], float& sum) {
  sum = 0.f;
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int ch = lane + 32 * c;
#pragma unroll
    for (int j = 0; j < 8; ++j) v[c][j] = 0.f;
    if (ch < nch) {
      Vec8<TX>::load(x + r * E + ch * 8, v[c]);
      if (res) { float t[8]; Vec8<TR>::load(res + r * E + ch * 8, t);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[c][j] += t[j]; }
#pragma unroll
      for (int j = 0; j < 8; ++j) sum += v[c][j];
    }
  }
}
template <int NC>
__device__ __forceinline__ void ln_stats(const float (&v)[NC][8], float sum, int E, int nch, int lane, float eps, float& mu, float& rs) {
  mu = warp_sum(sum) / (float)E;
  float q = 0.f;
#pragma unroll
  for (int c = 0; c < NC; ++c) if (lane + 32 * c < nch) {
#pragma unroll
    for (int j = 0; j < 8; ++j) { const float d = v[c][j] - mu; q = fmaf(d, d, q); }
  }
  rs = rsqrtf(warp_sum(q) / (float)E + eps);
}

// y = LN(x + res) * gamma + beta   (y32: optional fp32 copy of y, the residual operand of the next LayerNorm)
template <typename TX, typename TR, typename TY, int NC>
__global__ void __launch_bounds__(LN_THREADS)
ln_fwd_kernel(const TX* __restrict__ x, const TR* __restrict__ res, const float* __restrict__ gamma, const float* __restrict__ beta,
              TY* __restrict__ y, float* __restrict__ y32, float* __restrict__ mean, float* __restrict__ rstd, long R, int E, float eps) {
  const int lane = threadIdx.x & 31, wpb = LN_THREADS / 32, nch = E >> 3;
  for (long r = (long)blockIdx.x * wpb + (threadIdx.x >> 5); r < R; r += (long)gridDim.x * wpb) {
    float v[NC][8], sum, mu, rs;
    ln_load_row<TX, TR, NC>(x, res, r, E, nch, lane, v, sum);
    ln_stats<NC>(v, sum, E, nch, lane, eps, mu, rs);
    if (lane == 0) { mean[r] = mu; rstd[r] = rs; }
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const int ch = lane + 32 * c;
      if (ch < nch) {
        float g[8], b[8], o[8];
        Vec8<float>::load(gamma + ch * 8, g); Vec8<float>::load(beta + ch * 8, b);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = fmaf((v[c][j] - mu) * rs, g[j], b[j]);
        if (y) Vec8<TY>::store(y + r * E + ch * 8, o);
        if (y32) Vec8<float>::store(y32 + r * E + ch * 8, o);
      }
    }
  }
}

// FeatureProjector tail, fused: out[b,o,:] = mean over the token window of LN(x[b,l,:]) * gamma + beta.  One warp per (b,o);
// rows shared by two windows are normalised twice (no (B,L,E) intermediate is written); mean / rstd kept per row.
template <typename TX, int NC>
__global__ void __launch_bounds__(LN_THREADS)
ln_pool_fwd_kernel(const TX* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta, float* __restrict__ out,
                   float* __restrict__ mean, float* __restrict__ rstd, int B, int L, int O, int E, float eps) {
  const int lane = threadIdx.x & 31, wpb = LN_THREADS / 32, nch = E >> 3;
  const long total = (long)B * O;
  for (long w = (long)blockIdx.x * wpb + (threadIdx.x >> 5); w < total; w += (long)gridDim.x * wpb) {
    const unsigned wu = (unsigned)w, Ou = (unsigned)O, Lu = (unsigned)L;          // 32-bit index arithmetic (B * O, L * O < 2^31)
    const long b = (long)(wu / Ou); const int o = (int)(wu - (unsigned)b * Ou);
    const int lo = (int)(((unsigned)o * Lu) / Ou), hi = (int)((((unsigned)o + 1) * Lu + Ou - 1) / Ou);
    float acc[NC][8];
#pragma unroll
    for (int c = 0; c < NC; ++c)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[c][j] = 0.f;
    for (int l = lo; l < hi; ++l) {
      const long r = b * L + l;
      float v[NC][8], sum, mu, rs;
      ln_load_row<TX, TX, NC>(x, (const TX*)nullptr, r, E, nch, lane, v, sum);
      ln_stats<NC>(v, sum, E, nch, lane, eps, mu, rs);
      if (lane == 0) { mean[r] = mu; rstd[r] = rs; }
#pragma unroll
      for (int c = 0; c < NC; ++c)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[c][j] += (v[c][j] - mu) * rs;
    }
    const float inv = 1.0f / (float)(hi - lo);
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const int ch = lane + 32 * c;
      if (ch < nch) {
        float g[8], bb[8], o8[8];
        Vec8<float>::load(gamma + ch * 8, g); Vec8<float>::load(beta + ch * 8, bb);
#pragma unroll
        for (int j = 0; j < 8; ++j) o8[j] = fmaf(acc[c][j] * inv, g[j], bb[j]);
        Vec8<float>::store(out + w * E + ch * 8, o8);
      }
    }
  }
}

// dz = rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dy * gamma,  xhat = (x + res - mean) * rstd        (dz is d/dx and d/dres)
// dy comes either from `dy` or, for the projector (POOLED), from the pooled output gradient: dy[b,l,:] = sum over windows o
// containing l of dpool[b,o,:] / len(o).  Per-CTA partial sums of dgamma = sum_r dy*xhat, dbeta = sum_r dy and (the bias
// gradient of the Linear in front) sum_r dz go to part[(blockIdx, {0,1,2}, e)].
template <typename TX, typename TR, typename TDY, typename TDZ, bool POOLED, int NC>
__global__ void __launch_bounds__(LN_THREADS, NC == 1 ? 3 : 2)
ln_bwd_kernel(const TDY* __restrict__ dy, const float* __restrict__ dpool, int L, int O,
              const TX* __restrict__ x, const TR* __restrict__ res, const float* __restrict__ mean,
              const float* __restrict__ rstd, const float* __restrict__ gamma, TDZ* __restrict__ dz, float* __restrict__ dz32,
              float* __restrict__ part, long R, int E) {
  extern __shared__ float ln_sm[];          // [wpb][3][E]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = LN_THREADS / 32, nch = E >> 3;
  float ag[NC][8], ab[NC][8], az[NC][8], gm[NC][8];
#pragma unroll
  for (int c = 0; c < NC; ++c) {
#pragma unroll
    for (int j = 0; j < 8; ++j) { ag[c][j] = 0.f; ab[c][j] = 0.f; az[c][j] = 0.f; gm[c][j] = 0.f; }
    if (lane + 32 * c < nch) Vec8<float>::load(gamma + (lane + 32 * c) * 8, gm[c]);
  }
  for (long r = (long)blockIdx.x * wpb + warp; r < R; r += (long)gridDim.x * wpb) {
    const float mu = mean[r], rs = rstd[r];
    float v[NC][8], d[NC][8], sum;
    ln_load_row<TX, TR, NC>(x, res, r, E, nch, lane, v, sum);
    int o_min = 0, o_max = -1; long bo = 0;
    if (POOLED) {
      // 32-bit index arithmetic (R, L * O < 2^31): six 64-bit divisions per row made this variant ALU-bound (129 us for 100 864 rows)
      const unsigned ru = (unsigned)r, Lu = (unsigned)L, Ou = (unsigned)O;
      const unsigned b = ru / Lu, l = ru - b * Lu;
      o_min = (int)((l * Ou) / Lu); o_max = (int)(((l + 1) * Ou + Lu - 1) / Lu) - 1; bo = (long)b * O;
    }
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const int ch = lane + 32 * c;
#pragma unroll
      for (int j = 0; j < 8; ++j) d[c][j] = 0.f;
      if (ch < nch) {
        if (POOLED) {
          for (int o = o_min; o <= o_max; ++o) {
            const int lo = (int)(((unsigned)o * (unsigned)L) / (unsigned)O), hi = (int)((((unsigned)o + 1) * (unsigned)L + (unsigned)O - 1) / (unsigned)O);
            float t[8]; Vec8<float>::load(dpool + (bo + o) * E + ch * 8, t);
            const float inv = 1.0f / (float)(hi - lo);
#pragma unroll
            for (int j = 0; j < 8; ++j) d[c][j] = fmaf(t[j], inv, d[c][j]);
          }
        } else {
          Vec8<TDY>::load(dy + r * E + ch * 8, d[c]);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float xh = (v[c][j] - mu) * rs, g = d[c][j] * gm[c][j];
          v[c][j] = xh;
          s1 += g; s2 = fmaf(g, xh, s2);
          ag[c][j] = fmaf(d[c][j], xh, ag[c][j]); ab[c][j] += d[c][j];
        }
      }
    }
    const float m1 = warp_sum(s1) / (float)E, m2 = warp_sum(s2) / (float)E;
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const int ch = lane + 32 * c;
      if (ch < nch) {
        float o8[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { o8[j] = rs * (d[c][j] * gm[c][j] - m1 - v[c][j] * m2); az[c][j] += o8[j]; }
        Vec8<TDZ>::store(dz + r * E + ch * 8, o8);
        if (dz32) Vec8<float>::store(dz32 + r * E + ch * 8, o8);
      }
    }
  }
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int ch = lane + 32 * c;
    if (ch < nch) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        ln_sm[(warp * 3 + 0) * E + ch * 8 + j] = ag[c][j]; ln_sm[(warp * 3 + 1) * E + ch * 8 + j] = ab[c][j]; ln_sm[(warp * 3 + 2) * E + ch * 8 + j] = az[c][j];
      }
    }
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < 3 * E; idx += LN_THREADS) {
    const int which = idx / E, e = idx - which * E;
    float s = 0.f;
    for (int w = 0; w < wpb; ++w) s += ln_sm[(w * 3 + which) * E + e];
    part[((long)blockIdx.x * 3 + which) * E + e] = s;
  }
}
// dgamma / dbeta / (optional) dbias_prev [e] = sum over blocks of part[b, {0,1,2}, e]   (fixed order: deterministic)
// grid (ceil(E/32), 3): 32 columns x 8 row lanes per block
__global__ void __launch_bounds__(256) ln_param_grad_kernel(const float* __restrict__ part, int nblk, int E, float* __restrict__ dgamma,
                                                            float* __restrict__ dbeta, float* __restrict__ dbias_prev) {
  __shared__ float red[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5, e = blockIdx.x * 32 + tx, which = blockIdx.y;
  float* dst = which == 0 ? dgamma : (which == 1 ? dbeta : dbias_prev);
  if (!dst) return;
  float s = 0.f;
  if (e < E) {
    // four independent partial sums: the loads of a thread are in flight together instead of one L2 round trip per addend
    // (this kernel sits twice on the refinement backward's chain)
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    int b = ty;
    for (; b + 24 < nblk; b += 32) {
      s0 += part[((long)b * 3 + which) * E + e]; s1 += part[((long)(b + 8) * 3 + which) * E + e];
      s2 += part[((long)(b + 16) * 3 + which) * E + e]; s3 += part[((long)(b + 24) * 3 + which) * E + e];
    }
    for (; b < nblk; b += 8) s0 += part[((long)b * 3 + which) * E + e];
    s = (s0 + s1) + (s2 + s3);
  }
  red[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && e < E) { float t = 0.f; for (int i = 0; i < 8; ++i) t += red[i][tx]; dst[e] = t; }
}

// ------------------------------------------------------------------ column sums (bias gradients), optionally fused with the ReLU backward
// A is (rows, cols) with pitch ld, ld % 8 == 0 and cols <= ld; nch = ceil(cols / 8).  Block = 32 chunk lanes x 8 row lanes: a warp
// reads 32 consecutive 8-element chunks of one row.  Columns cols..8*nch-1 of the last chunk are read (they lie inside the pitch)
// and summed, but never written to `partial`.
// RELU_BWD: d <- act > 0 ? d * inv_keep : 0 is applied in place first (act = the saved post-ReLU / post-dropout activation).
template <typename T, bool RELU_BWD>
__device__ __forceinline__ void colsum_vec_body(T* __restrict__ A, const T* __restrict__ act, long rows, int cols, long ld, int nch,
                                                float inv_keep, float* __restrict__ partial) {
  __shared__ float red[8][32 * 8 + 8];
  const int lane = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int ch = blockIdx.x * 32 + lane;
  const long per = (rows + gridDim.y - 1) / gridDim.y;
  const long r0 = (long)blockIdx.y * per, r1 = (r0 + per < rows) ? r0 + per : rows;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  if (ch < nch) {
    long r = r0 + ry;
    // four independent 16-byte row loads in flight per thread (the one-row-at-a-time loop was a chain of L2 / HBM round trips:
    // 68 us for the 42 MB gate-gradient matrix = 0.6 TB/s, on the branch that ends the step; profiles/README.md round 2)
    for (; r + 24 < r1; r += 32) {
      float v[4][8];
#pragma unroll
      for (int u = 0; u < 4; ++u) Vec8<T>::load(A + (r + 8 * u) * ld + ch * 8, v[u]);
      if (RELU_BWD) {
        float a[4][8];
#pragma unroll
        for (int u = 0; u < 4; ++u) Vec8<T>::load(act + (r + 8 * u) * ld + ch * 8, a[u]);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
#pragma unroll
          for (int j = 0; j < 8; ++j) v[u][j] = a[u][j] > 0.f ? v[u][j] * inv_keep : 0.f;
          Vec8<T>::store(A + (r + 8 * u) * ld + ch * 8, v[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += v[u][j];
    }
    for (; r < r1; r += 8) {
      float v[8];
      Vec8<T>::load(A + r * ld + ch * 8, v);
      if (RELU_BWD) {
        float a[8]; Vec8<T>::load(act + r * ld + ch * 8, a);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = a[j] > 0.f ? v[j] * inv_keep : 0.f;
        Vec8<T>::store(A + r * ld + ch * 8, v);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += v[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[ry][lane * 8 + j] = acc[j];
  __syncthreads();
  const int t = threadIdx.x;                       // 256 threads = 32 chunks x 8 columns
  const int col = blockIdx.x * 256 + t;
  if (col < cols) {
    float sres = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) sres += red[i][t];
    partial[(long)blockIdx.y * cols + col] = sres;
  }
}
template <typename T, bool RELU_BWD>
__global__ void __launch_bounds__(256)
colsum_vec_kernel(T* __restrict__ A, const T* __restrict__ act, long rows, int cols, float inv_keep, float* __restrict__ partial) {
  colsum_vec_body<T, RELU_BWD>(A, act, rows, cols, cols, cols >> 3, inv_keep, partial);     // contiguous, cols % 8 == 0
}
// column sums of a pitched matrix (e.g. the logits gradient with its row pitch rounded up to 8 elements)
template <typename T>
__global__ void __launch_bounds__(256)
colsum_vec_pitched_kernel(const T* __restrict__ A, long rows, int cols, long ld, float* __restrict__ partial) {
  colsum_vec_body<T, false>(const_cast<T*>(A), (const T*)nullptr, rows, cols, ld, (cols + 7) >> 3, 1.f, partial);
}

// ------------------------------------------------------------------ multi-head self-attention core over S tokens (S = 49), one CTA per (sample, head)
// qkv (B*S, 3E) -> out (B*S, E);  probabilities BEFORE dropout are kept (B, heads, S, S) for the backward.
// All products are 4x4 register tiles over shared-memory operands read with 16-byte loads (row pitches are multiples of 4 floats
// and odd multiples of 16 bytes, so the quarter-warp accesses are conflict free).
constexpr int MHA_THREADS = 256;
constexpr uint32_t MHA_DROP_SITE = 200u;

// C[i][j] = sum_k A[i][k] * B[j][k]          (A: Mi x K, B: Nj x K, both with pitch pk)
// A thread owns the STRIDED 4x4 tile rows {it + a*ti} x {jt + b*tj}: the threads of a quarter warp then read CONSECUTIVE rows
// (pitch = odd multiple of 16 bytes -> conflict free); contiguous 4-row blocks would put them 4 rows apart (7-way conflicts).
template <typename F>
__device__ __forceinline__ void mha_tile_nt(const float* A, const float* Bm, int Mi, int Nj, int K, int pk, F&& emit) {
  const int ti = (Mi + 3) >> 2, tj = (Nj + 3) >> 2;
  for (int t = threadIdx.x; t < ti * tj; t += MHA_THREADS) {
    const int it = t / tj, jt = t - it * tj;
    float acc[4][4] = {};
    const float* ar[4]; const float* br[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) { ar[a] = A + min(it + a * ti, Mi - 1) * pk; br[a] = Bm + min(jt + a * tj, Nj - 1) * pk; }
    for (int k = 0; k < K; k += 4) {
      float4 av[4], bv[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) { av[a] = *reinterpret_cast<const float4*>(ar[a] + k); bv[a] = *reinterpret_cast<const float4*>(br[a] + k); }
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b)
          acc[a][b] = fmaf(av[a].x, bv[b].x, fmaf(av[a].y, bv[b].y, fmaf(av[a].z, bv[b].z, fmaf(av[a].w, bv[b].w, acc[a][b]))));
    }
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) if (it + a * ti < Mi && jt + b * tj < Nj) emit(it + a * ti, jt + b * tj, acc[a][b]);
  }
}
// C[i][d] = sum_j P[i][j] * V[j][d]          (P: Mi x J pitch pp; V: J x D pitch pd)
template <typename F>
__device__ __forceinline__ void mha_tile_nn(const float* P, const float* V, int Mi, int J, int D, int pp, int pd, F&& emit) {
  const int ti = (Mi + 3) >> 2, td = D >> 2;
  for (int t = threadIdx.x; t < ti * td; t += MHA_THREADS) {
    const int i0 = (t / td) * 4, d0 = (t % td) * 4;
    float acc[4][4] = {};
    const float* pr[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) pr[a] = P + min(i0 + a, Mi - 1) * pp;
    for (int j = 0; j < J; ++j) {
      const float4 v = *reinterpret_cast<const float4*>(V + j * pd + d0);
#pragma unroll
      for (int a = 0; a < 4; ++a) { const float pv = pr[a][j]; acc[a][0] = fmaf(pv, v.x, acc[a][0]); acc[a][1] = fmaf(pv, v.y, acc[a][1]); acc[a][2] = fmaf(pv, v.z, acc[a][2]); acc[a][3] = fmaf(pv, v.w, acc[a][3]); }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) if (i0 + a < Mi) {
#pragma unroll
      for (int b = 0; b < 4; ++b) emit(i0 + a, d0 + b, acc[a][b]);
    }
  }
}
// C[j][d] = sum_i P[i][j] * Dm[i][d]         (P: I x Nj pitch pp (multiple of 4); Dm: I x D pitch pd)
template <typename F>
__device__ __forceinline__ void mha_tile_tn(const float* P, const float* Dm, int I, int Nj, int D, int pp, int pd, F&& emit) {
  const int tj = (Nj + 3) >> 2, td = D >> 2;
  for (int t = threadIdx.x; t < tj * td; t += MHA_THREADS) {
    const int j0 = (t / td) * 4, d0 = (t % td) * 4;
    float acc[4][4] = {};
    for (int i = 0; i < I; ++i) {
      const float4 p = *reinterpret_cast<const float4*>(P + i * pp + j0);      // columns beyond Nj are zero padding
      const float4 v = *reinterpret_cast<const float4*>(Dm + i * pd + d0);
      const float pa[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
      for (int a = 0; a < 4; ++a) { acc[a][0] = fmaf(pa[a], v.x, acc[a][0]); acc[a][1] = fmaf(pa[a], v.y, acc[a][1]); acc[a][2] = fmaf(pa[a], v.z, acc[a][2]); acc[a][3] = fmaf(pa[a], v.w, acc[a][3]); }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) if (j0 + a < Nj) {
#pragma unroll
      for (int b = 0; b < 4; ++b) emit(j0 + a, d0 + b, acc[a][b]);
    }
  }
}
__host__ __device__ __forceinline__ int mha_pitch(int n) { int p = (n + 3) & ~3; if (((p >> 2) & 1) == 0) p += 4; return p; }   // odd multiple of 16 bytes

template <typename T>
__device__ __forceinline__ void mha_load_heads(const T* qkv, int b, int h, int S, int E, int hd, int ph, float* Qs, float* Ks, float* Vs) {
  if (hd & 7) {                                // head_dim % 4 == 0 only: scalar loads
    for (int idx = threadIdx.x; idx < S * hd; idx += MHA_THREADS) {
      const int i = idx / hd, d = idx - i * hd;
      const T* row = qkv + (long)(b * S + i) * 3 * E + h * hd + d;
      Qs[i * ph + d] = to_f<T>(row[0]); Ks[i * ph + d] = to_f<T>(row[E]); Vs[i * ph + d] = to_f<T>(row[2 * E]);
    }
    return;
  }
  const int v8 = hd >> 3;
  for (int idx = threadIdx.x; idx < S * v8; idx += MHA_THREADS) {
    const int i = idx / v8, c = idx - i * v8;
    const T* row = qkv + (long)(b * S + i) * 3 * E + h * hd + c * 8;
    float t[8];
    Vec8<T>::load(row, t);         Vec8<float>::store(Qs + i * ph + c * 8, t);
    Vec8<T>::load(row + E, t);     Vec8<float>::store(Ks + i * ph + c * 8, t);
    Vec8<T>::load(row + 2 * E, t); Vec8<float>::store(Vs + i * ph + c * 8, t);
  }
}

template <typename T>
__global__ void __launch_bounds__(MHA_THREADS)
mha_fwd_kernel(const T* __restrict__ qkv, T* __restrict__ out, T* __restrict__ probs, int S, int E, int heads, float scale,
               float drop_p, uint64_t seed, const unsigned long long* __restrict__ seed_dev) {
  extern __shared__ __align__(16) float mh_sm[];
  if (drop_p > 0.f) seed = drop_seed(seed, seed_dev);
  const int hd = E / heads, ph = mha_pitch(hd), ps = mha_pitch(S);
  float* Qs = mh_sm; float* Ks = Qs + S * ph; float* Vs = Ks + S * ph; float* sc = Vs + S * ph;    // sc: S x ps
  const int b = blockIdx.x, h = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  mha_load_heads<T>(qkv, b, h, S, E, hd, ph, Qs, Ks, Vs);
  __syncthreads();
  mha_tile_nt(Qs, Ks, S, S, hd, ph, [&](int i, int j, float v) { sc[i * ps + j] = v * scale; });
  __syncthreads();
  const float inv_keep = drop_p > 0.f ? 1.0f / (1.0f - drop_p) : 1.0f;
  for (int i = warp; i < S; i += MHA_THREADS / 32) {
    float m = -INFINITY;
    for (int j = lane; j < S; j += 32) m = fmaxf(m, sc[i * ps + j]);
    m = warp_max(m);
    float s = 0.f;
    for (int j = lane; j < S; j += 32) { const float e = Math<T>::exp_(sc[i * ps + j] - m); sc[i * ps + j] = e; s += e; }
    s = warp_sum(s);
    const float inv = 1.0f / s;
    const long pbase = ((long)(b * heads + h) * S + i) * S;
    for (int j = lane; j < S; j += 32) {
      const float p = sc[i * ps + j] * inv;
      probs[pbase + j] = from_f<T>(p);
      sc[i * ps + j] = drop_p > 0.f ? p * dropout_scale(seed, MHA_DROP_SITE, (uint64_t)(pbase + j), drop_p, inv_keep) : p;
    }
  }
  __syncthreads();
  mha_tile_nn(sc, Vs, S, S, hd, ps, ph, [&](int i, int d, float v) { out[(long)(b * S + i) * E + h * hd + d] = from_f<T>(v); });
}

template <typename T>
__global__ void __launch_bounds__(MHA_THREADS)
mha_bwd_kernel(const T* __restrict__ qkv, const T* __restrict__ probs, const T* __restrict__ dout, T* __restrict__ dqkv,
               int S, int E, int heads, float scale, float drop_p, uint64_t seed, const unsigned long long* __restrict__ seed_dev) {
  extern __shared__ __align__(16) float mh_sm[];
  if (drop_p > 0.f) seed = drop_seed(seed, seed_dev);
  const int hd = E / heads, ph = mha_pitch(hd), ps = mha_pitch(S);
  float* Qs = mh_sm; float* Ks = Qs + S * ph; float* Vs = Ks + S * ph; float* dOs = Vs + S * ph;
  float* Ps = dOs + S * ph; float* dS = Ps + S * ps; float* Pd = drop_p > 0.f ? dS + S * ps : Ps;     // S x ps each; Pd aliases Ps without dropout
  const int b = blockIdx.x, h = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float inv_keep = drop_p > 0.f ? 1.0f / (1.0f - drop_p) : 1.0f;
  mha_load_heads<T>(qkv, b, h, S, E, hd, ph, Qs, Ks, Vs);
  for (int idx = tid; idx < S * hd; idx += MHA_THREADS) {
    const int i = idx / hd, d = idx - i * hd;
    dOs[i * ph + d] = to_f<T>(dout[(long)(b * S + i) * E + h * hd + d]);
  }
  const long pb = (long)(b * heads + h) * S * S;
  for (int idx = tid; idx < S * ps; idx += MHA_THREADS) {
    const int i = idx / ps, j = idx - i * ps;
    float p = 0.f, m = 1.f;
    if (j < S) { p = to_f<T>(probs[pb + i * S + j]); if (drop_p > 0.f) m = dropout_scale(seed, MHA_DROP_SITE, (uint64_t)(pb + i * S + j), drop_p, inv_keep); }
    Ps[idx] = p; if (drop_p > 0.f) Pd[idx] = p * m; dS[idx] = m;        // dS holds the mask until dP overwrites it
  }
  __syncthreads();
  // dV = Pd^T dO
  mha_tile_tn(Pd, dOs, S, S, hd, ps, ph, [&](int j, int d, float v) { dqkv[(long)(b * S + j) * 3 * E + 2 * E + h * hd + d] = from_f<T>(v); });
  // dP = (dO V^T) * mask
  mha_tile_nt(dOs, Vs, S, S, hd, ph, [&](int i, int j, float v) { dS[i * ps + j] = v * dS[i * ps + j]; });
  __syncthreads();
  // softmax backward per row: dS = P * (dP - sum_j dP * P) * scale
  for (int i = warp; i < S; i += MHA_THREADS / 32) {
    float dot = 0.f;
    for (int j = lane; j < S; j += 32) dot = fmaf(dS[i * ps + j], Ps[i * ps + j], dot);
    dot = warp_sum(dot);
    for (int j = lane; j < S; j += 32) dS[i * ps + j] = Ps[i * ps + j] * (dS[i * ps + j] - dot) * scale;
    for (int j = S + lane; j < ps; j += 32) dS[i * ps + j] = 0.f;
  }
  __syncthreads();
  // dQ = dS K,  dK = dS^T Q
  mha_tile_nn(dS, Ks, S, S, hd, ps, ph, [&](int i, int d, float v) { dqkv[(long)(b * S + i) * 3 * E + h * hd + d] = from_f<T>(v); });
  mha_tile_tn(dS, Qs, S, S, hd, ps, ph, [&](int j, int d, float v) { dqkv[(long)(b * S + j) * 3 * E + E + h * hd + d] = from_f<T>(v); });
}

// ------------------------------------------------------------------ AdaptiveAvgPool1d over the token axis: window o = [floor(o*L/O), ceil((o+1)*L/O))
template <typename T>
__global__ void __launch_bounds__(256) pool_fwd_kernel(const T* __restrict__ y, float* __restrict__ out, int B, int L, int O, int E) {
  const long total = (long)B * O * E;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int e = (int)(idx % E); const long bo = idx / E; const int o = (int)(bo % O); const long b = bo / O;
    const int lo = (int)(((long)o * L) / O), hi = (int)(((long)(o + 1) * L + O - 1) / O);
    float a = 0.f;
    for (int l = lo; l < hi; ++l) a += to_f<T>(y[(b * L + l) * E + e]);
    out[idx] = a / (float)(hi - lo);
  }
}
}  // namespace b2c
