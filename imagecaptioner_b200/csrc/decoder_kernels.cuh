// Kernels (1) and the pointwise glue of the decoder hot path.  Math: SURVEY.md Appendix A.1/A.2,
// reference src/student_model.py:173-203 (attention), :232-251 (step), :339-381 (greedy loop).
#pragma once
#include "common.cuh"

namespace b2c {

// ======================================================================================
// Parameter packing: fp32 master weights -> compute-type operand buffers, one launch.
// ======================================================================================
// row / column of a linear index: 32-bit division when the index fits (a 64-bit integer division is ~100 instructions; two of them per
// thread in lstm_pointwise_bwd cost 0.7 us per launch, 28 us per KD step)
__device__ __forceinline__ void divmod_idx(long i, int d, long& q, int& r) {
  if (i < 0x7fffffffL) { const unsigned qi = (unsigned)i / (unsigned)d; q = (long)qi; r = (int)((unsigned)i - qi * (unsigned)d); }
  else { q = i / d; r = (int)(i - q * d); }
}
struct PackSeg {
  const float* src; void* dst;
  const float* src2;        // optional: dst = src + src2 (bias_ih + bias_hh)
  int rows, cols; long lds, ldd;
  int as_float;             // 1: dst is fp32 regardless of T (bias vectors)
  int perm_h;               // != 0 (= H): gate-interleave the rows, dst row r <- src row (r & 3) * H + (r >> 2)
};
constexpr int PACK_MAX_SEGS = 20;
struct PackTable { PackSeg seg[PACK_MAX_SEGS]; int n; };

template <typename T>
__global__ void __launch_bounds__(256) pack_params_kernel(const __grid_constant__ PackTable tab) {
  const PackSeg& s = tab.seg[blockIdx.y];
  const long total = (long)s.rows * s.cols;
  // fast path: whole 4-element groups of a row with 16-byte source / 8- or 16-byte destination accesses, two groups in flight per
  // thread (the scalar loop below was a chain of dependent round trips: 53 us for the decoder's 29 MB of fp32 masters, at the head of
  // the step's critical path)
  if (!s.src2 && !s.as_float && (s.cols & 3) == 0 && (s.lds & 3) == 0 && (s.ldd & 3) == 0 && (((uintptr_t)s.src) & 15) == 0 &&
      (((uintptr_t)s.dst) & 15) == 0) {
    const int c4n = s.cols >> 2;
    const long groups = (long)s.rows * c4n, stride = (long)gridDim.x * blockDim.x;
    for (long g0 = (long)blockIdx.x * blockDim.x + threadIdx.x; g0 < groups; g0 += 2 * stride) {
      const long g1 = g0 + stride;
      long r0, r1; int c0, c1;
      divmod_idx(g0, c4n, r0, c0); divmod_idx(g1, c4n, r1, c1);
      c0 *= 4; c1 *= 4;
      const long rs0 = s.perm_h ? (long)(r0 & 3) * s.perm_h + (r0 >> 2) : r0, rs1 = s.perm_h ? (long)(r1 & 3) * s.perm_h + (r1 >> 2) : r1;
      const float4 v0 = *reinterpret_cast<const float4*>(s.src + rs0 * s.lds + c0);
      float4 v1 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (g1 < groups) v1 = *reinterpret_cast<const float4*>(s.src + rs1 * s.lds + c1);
      if (sizeof(T) == 2) {
        *reinterpret_cast<uint2*>(reinterpret_cast<T*>(s.dst) + r0 * s.ldd + c0) = make_uint2(pack_bf16(v0.x, v0.y), pack_bf16(v0.z, v0.w));
        if (g1 < groups) *reinterpret_cast<uint2*>(reinterpret_cast<T*>(s.dst) + r1 * s.ldd + c1) = make_uint2(pack_bf16(v1.x, v1.y), pack_bf16(v1.z, v1.w));
      } else {
        *reinterpret_cast<float4*>(reinterpret_cast<float*>(s.dst) + r0 * s.ldd + c0) = v0;
        if (g1 < groups) *reinterpret_cast<float4*>(reinterpret_cast<float*>(s.dst) + r1 * s.ldd + c1) = v1;
      }
    }
    return;
  }
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const long r = i / s.cols; const int c = (int)(i - r * s.cols);
    const long rs = s.perm_h ? (long)(r & 3) * s.perm_h + (r >> 2) : r;
    float v = s.src[rs * s.lds + c];
    if (s.src2) v += s.src2[rs * s.lds + c];
    if (s.as_float) reinterpret_cast<float*>(s.dst)[r * s.ldd + c] = v;
    else reinterpret_cast<T*>(s.dst)[r * s.ldd + c] = from_f<T>(v);
  }
}

// emb[r,:] = table[ids[r],:]   (ids out of range -> row 0, like a clamped lookup; the host validates nothing here)
template <typename T>
__global__ void __launch_bounds__(256) embedding_gather_kernel(const float* __restrict__ table, const int64_t* __restrict__ ids,
                                                               long rows, int E, int V, T* __restrict__ out, long ldo) {
  const int per = E / 4;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < rows * per; i += (long)gridDim.x * blockDim.x) {
    long r; int c; divmod_idx(i, per, r, c); c *= 4;
    long id = ids[r]; if (id < 0 || id >= V) id = 0;
    const float4 v = *reinterpret_cast<const float4*>(table + id * E + c);
    T* o = out + r * ldo + c;
    o[0] = from_f<T>(v.x); o[1] = from_f<T>(v.y); o[2] = from_f<T>(v.z); o[3] = from_f<T>(v.w);
  }
}

// dtable[ids[r],:] += drows[r,:]
__global__ void __launch_bounds__(256) embedding_scatter_add_kernel(const float* __restrict__ drows, const int64_t* __restrict__ ids,
                                                                    long rows, int E, int V, float* __restrict__ dtable) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < rows * E; i += (long)gridDim.x * blockDim.x) {
    long r; int c; divmod_idx(i, E, r, c);
    long id = ids[r]; if (id < 0 || id >= V) id = 0;
    atomicAdd(dtable + id * E + c, drows[i]);
  }
}

// caller-supplied initial LSTM state of one layer (reference src/student_model.py:205 `hidden`): h0 (B,H) fp32 -> the recurrent half of
// the layer's step-0 operand rows (pitch ld), c0 (B,H) fp32 -> slot 0 of the cell buffer
template <typename T>
__global__ void __launch_bounds__(256) initial_state_kernel(const float* __restrict__ h0, const float* __restrict__ c0, int B, int H,
                                                            T* __restrict__ h_rec, long ld, float* __restrict__ c_slot0) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < (long)B * H; i += (long)gridDim.x * blockDim.x) {
    const long b = i / H; const int j = (int)(i - b * H);
    h_rec[b * ld + j] = from_f<T>(h0[i]);
    c_slot0[i] = c0[i];
  }
}

// ======================================================================================
// Kernel (1): one decode step of spatial attention for one sample per CTA.
//   s_l = sum_e tanh(P[l,e] + u[e]);  w = softmax_l(s);  ctx[e] = sum_l w_l F[l,e]
// P_b and F_b (S x E each, contiguous) are staged in shared memory by two 1-D TMA bulk copies.
// ======================================================================================
constexpr int ATT_THREADS = 256;
constexpr int ATT_MAXTOK = 7;     // tokens per warp held in registers (S <= 56 with 8 warps)

// F_b (the S x E feature tokens of one sample, compute type) is staged in shared memory by one 1-D TMA bulk copy on an
// mbarrier.  P_b (the hoisted projection, fp32 in both modes because the score sums E tanh terms) is used exactly once per
// step, so it is streamed from L2 with coalesced 128-bit loads into registers instead of taking shared memory:
// 26 KB per CTA at E=256 bf16, so all B CTAs of a step are co-resident.
//
// Latency structure (ncu: no pipe above 35 %, the kernels are a chain of L2 round trips): P, F (and in the backward also the
// saved u and attention weights) are LOOP INVARIANTS, so their loads are issued BEFORE griddepcontrol.wait and overlap the
// tail of the preceding kernel; only u (forward) / d ctx (backward) wait for it.  Callers break the early-start cascade once
// after the producers of the invariants (pdl_full_dependency_next in common.cuh).
template <typename T, int NQ, int KA>  // NQ = float4 per lane per token (ceil(E/128)); 0 = generic loop.  KA = tokens per warp fetched in the prologue
__global__ void __launch_bounds__(ATT_THREADS, KA >= ATT_MAXTOK ? 1 : 4)
attn_step_fwd_kernel(const float* __restrict__ P, const T* __restrict__ F, const float* __restrict__ u, long ldu,
                     int S, int E, T* __restrict__ ctx, long ldctx, float* __restrict__ attw /* (B,S) or null */,
                     float* __restrict__ u_save /* (B,E) or null: dense copy of u (a forward save when u sits inside a wider row) */,
                     const int* __restrict__ steps /* null, or the device step count: step `step` >= *steps does nothing */, int step) {
  extern __shared__ __align__(128) unsigned char att_smem[];
  const int SE = S * E;
  T* Fs = reinterpret_cast<T*>(att_smem);
  float* us = reinterpret_cast<float*>(Fs + SE);
  float* sc = us + E;
  __shared__ __align__(8) uint64_t bar;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = ATT_THREADS / 32;
  const int b = blockIdx.x;
  pdl_launch_dependents();
  if (steps != nullptr && step >= __ldg(steps)) { pdl_wait(); return; }      // past the batch's length (invariant I1, api.cu)
  // ---- prologue: independent of the preceding kernel
  if (tid == 0) { mbar_init(&bar, 1); fence_barrier_init(); }
  const float4* Pb = reinterpret_cast<const float4*>(P + (long)b * SE);
  const int E4 = E >> 2;
  constexpr int NQR = NQ > 0 ? NQ : 1;
  constexpr int KB = ATT_MAXTOK - KA > 0 ? ATT_MAXTOK - KA : 1;
  // NQ > 0 instantiations are launched only when every token fits a warp's register rows (S <= ATT_MAXTOK * nwarp, checked by the
  // host): the generic loop is then not even compiled in (a third of this kernel's code; it runs 20 times per step from a cold I-cache)
  constexpr bool fast = NQ > 0;
  float4 pa[KA][NQR];
  if constexpr (fast) {
#pragma unroll
    for (int k = 0; k < KA; ++k) {
      const int l = warp + k * nwarp;
#pragma unroll
      for (int j = 0; j < NQR; ++j) {
        const int q = lane + j * 32;
        if (l < S && q < E4) pa[k][j] = __ldg(Pb + l * E4 + q);
      }
    }
  }
  __syncthreads();
  if (tid == 0) {
    const uint32_t fb = (uint32_t)(SE * sizeof(T));
    mbar_arrive_expect_tx(&bar, fb);
    bulk_g2s(Fs, F + (long)b * SE, fb, &bar);
  }
  pdl_wait();
  // u is the only operand produced by the preceding kernel
  for (int e = tid; e < E; e += ATT_THREADS) { const float uv = __ldcg(u + (long)b * ldu + e); us[e] = uv; if (u_save) u_save[(long)b * E + e] = uv; }
  __syncthreads();
  // scores: warp per token, lanes over E in float4 units
  auto score = [&](const float4 (&pv)[NQR], int l) {
    float a = 0.f;
#pragma unroll
    for (int j = 0; j < NQR; ++j) {
      const int q = lane + j * 32;
      if (q < E4) {
        const float4 p = pv[j];
        const float4 uu = *reinterpret_cast<const float4*>(us + q * 4);
        a += Math<T>::tanh_(p.x + uu.x) + Math<T>::tanh_(p.y + uu.y) + Math<T>::tanh_(p.z + uu.z) + Math<T>::tanh_(p.w + uu.w);
      }
    }
    a = warp_sum(a);
    if (lane == 0) sc[l] = a;
  };
  if constexpr (fast) {
    float4 pb[KB][NQR];
    if (KA < ATT_MAXTOK) {
#pragma unroll
      for (int k = 0; k < KB; ++k) {
        const int l = warp + (KA + k) * nwarp;
#pragma unroll
        for (int j = 0; j < NQR; ++j) {
          const int q = lane + j * 32;
          if (l < S && q < E4) pb[k][j] = __ldg(Pb + l * E4 + q);
        }
      }
    }
#pragma unroll
    for (int k = 0; k < KA; ++k) { const int l = warp + k * nwarp; if (l < S) score(pa[k], l); }
    if (KA < ATT_MAXTOK) {
#pragma unroll
      for (int k = 0; k < KB; ++k) { const int l = warp + (KA + k) * nwarp; if (l < S) score(pb[k], l); }
    }
  } else if constexpr (!fast) {
    for (int l = warp; l < S; l += nwarp) {
      float a = 0.f;
      for (int q = lane; q < E4; q += 32) {
        const float4 p = __ldg(Pb + l * E4 + q);
        const float4 uu = *reinterpret_cast<const float4*>(us + q * 4);
        a += Math<T>::tanh_(p.x + uu.x) + Math<T>::tanh_(p.y + uu.y) + Math<T>::tanh_(p.z + uu.z) + Math<T>::tanh_(p.w + uu.w);
      }
      a = warp_sum(a);
      if (lane == 0) sc[l] = a;
    }
  }
  __syncthreads();
  if (warp == 0) {
    float m = -INFINITY;
    for (int l = lane; l < S; l += 32) m = fmaxf(m, sc[l]);
    m = warp_max(m);
    float s = 0.f;
    for (int l = lane; l < S; l += 32) { const float e = Math<T>::exp_(sc[l] - m); sc[l] = e; s += e; }
    s = warp_sum(s);
    const float inv = 1.0f / s;
    for (int l = lane; l < S; l += 32) { const float wv = sc[l] * inv; sc[l] = wv; if (attw) attw[(long)b * S + l] = wv; }
  }
  __syncthreads();
  mbar_wait(&bar, 0);                          // the feature tokens have landed (their copy overlapped everything above)
  for (int e = tid; e < E; e += ATT_THREADS) {
    float a = 0.f;
    for (int l = 0; l < S; ++l) a = fmaf(sc[l], to_f<T>(Fs[l * E + e]), a);
    ctx[(long)b * ldctx + e] = from_f<T>(a);
  }
}

// Backward of one attention step (inside the reverse time loop): ds (B,S) and du (B,E).
//   dw_l = sum_e dctx_e F[l,e];  ds_l = w_l (dw_l - sum_j w_j dw_j);  du_e = sum_l ds_l (1 - tanh^2(P[l,e]+u_e))
// Shared memory: Fs (S*E) | dcs (E) | dw (S) | ws (S).  The du phase walks P in batches of PB rows, the next batch in flight
// while the current one goes through the MUFU (the unbatched loop was 49 serialised L2 round trips: 58 % of all stall samples).
template <typename T, int PB, bool E256 = false>       // E256: E <= 256 known at compile time (one 8-element chunk per lane; the wide loop is not compiled in)
__global__ void __launch_bounds__(ATT_THREADS, 4)
attn_step_bwd_kernel(const float* __restrict__ P, const T* __restrict__ F, const float* __restrict__ u, long ldu,
                     const float* __restrict__ attw, const float* __restrict__ dctx, long lddctx,
                     int S, int E, float* __restrict__ ds_out, T* __restrict__ du, long lddu,
                     const int* __restrict__ steps /* null, or the device step count: step `step` >= *steps does nothing */, int step) {
  extern __shared__ __align__(128) unsigned char att_smem[];
  const int SE = S * E;
  T* Fs = reinterpret_cast<T*>(att_smem);
  float* dcs = reinterpret_cast<float*>(Fs + SE);
  float* dw = dcs + E;
  float* ws = dw + S;
  __shared__ __align__(8) uint64_t bar;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = ATT_THREADS / 32;
  const int b = blockIdx.x;
  const float* Pb = P + (long)b * SE;
  pdl_launch_dependents();
  if (steps != nullptr && step >= __ldg(steps)) { pdl_wait(); return; }      // past the batch's length (invariant I1, api.cu)
  // ---- prologue: F, P, u and the attention weights were written by the forward pass
  if (tid == 0) { mbar_init(&bar, 1); fence_barrier_init(); }
  for (int l = tid; l < S; l += ATT_THREADS) ws[l] = attw[(long)b * S + l];
  float cur[PB];
  float ue0 = 0.f;
  if (tid < E) {
    ue0 = u[(long)b * ldu + tid];
#pragma unroll
    for (int i = 0; i < PB; ++i) if (i < S) cur[i] = __ldg(Pb + (long)i * E + tid);
  }
  __syncthreads();
  if (tid == 0) {
    const uint32_t fb = (uint32_t)(SE * sizeof(T));
    mbar_arrive_expect_tx(&bar, fb);
    bulk_g2s(Fs, F + (long)b * SE, fb, &bar);
  }
  pdl_wait();
  for (int e = tid; e < E; e += ATT_THREADS) dcs[e] = __ldcg(dctx + (long)b * lddctx + e);
  __syncthreads();
  mbar_wait(&bar, 0);
  // dw: warp per token, each lane owns 8-element chunks (one 16-byte shared load per token in bf16)
  if (E256 || E <= 256) {
    float d[8];
    const int c = lane * 8;
    const bool on = c < E;
    if (on) Vec8<float>::load(dcs + c, d);
    for (int l = warp; l < S; l += nwarp) {
      float a = 0.f;
      if (on) {
        float f[8];
        Vec8<T>::load(Fs + l * E + c, f);
#pragma unroll
        for (int i = 0; i < 8; ++i) a = fmaf(d[i], f[i], a);
      }
      a = warp_sum(a);
      if (lane == 0) dw[l] = a;
    }
  } else if constexpr (!E256) {
    for (int l = warp; l < S; l += nwarp) {
      float a = 0.f;
      for (int c = lane * 8; c < E; c += 256) {
        float f[8], d[8];
        Vec8<T>::load(Fs + l * E + c, f);
        Vec8<float>::load(dcs + c, d);
#pragma unroll
        for (int i = 0; i < 8; ++i) a = fmaf(d[i], f[i], a);
      }
      a = warp_sum(a);
      if (lane == 0) dw[l] = a;
    }
  }
  __syncthreads();
  if (warp == 0) {
    float dot = 0.f;
    for (int l = lane; l < S; l += 32) dot = fmaf(ws[l], dw[l], dot);
    dot = warp_sum(dot);
    for (int l = lane; l < S; l += 32) { const float v = ws[l] * (dw[l] - dot); dw[l] = v; ds_out[(long)b * S + l] = v; }
  }
  __syncthreads();
  for (int e = tid; e < E; e += ATT_THREADS) {
    float ue = ue0;
    if (e != tid) {
      ue = u[(long)b * ldu + e];
#pragma unroll
      for (int i = 0; i < PB; ++i) if (i < S) cur[i] = __ldg(Pb + (long)i * E + e);
    }
    float a = 0.f;
    for (int l0 = 0; l0 < S; l0 += PB) {
      float nxt[PB];
      if (l0 + PB < S) {
#pragma unroll
        for (int i = 0; i < PB; ++i) if (l0 + PB + i < S) nxt[i] = __ldg(Pb + (long)(l0 + PB + i) * E + e);
      }
#pragma unroll
      for (int i = 0; i < PB; ++i) {
        if (l0 + i < S) a = fmaf(dw[l0 + i], Math<T>::dtanh_(cur[i] + ue), a);
      }
#pragma unroll
      for (int i = 0; i < PB; ++i) cur[i] = nxt[i];
    }
    du[(long)b * lddu + e] = from_f<T>(a);
  }
}

// After the reverse loop, one pass per sample over all steps:
//   dP[l,e]      = sum_t ds[t,l] (1 - tanh^2(P[l,e] + u[t,e]))
//   dF_attn[l,e] = sum_t w[t,l] dctx[t,e]
// u/dctx/w/ds for all T steps of this sample sit in shared memory (T*(2E+2S) floats).
template <typename T>
__global__ void __launch_bounds__(ATT_THREADS)
attn_post_kernel(const float* __restrict__ P, const float* __restrict__ u /*(T,B,E)*/, const float* __restrict__ dctx /*(T,B,.) pitch lddctx*/, long lddctx,
                 const float* __restrict__ attw /*(T,B,S)*/, const float* __restrict__ ds /*(T,B,S)*/,
                 int Tn, int B, int S, int E, T* __restrict__ dP, float* __restrict__ dF) {
  extern __shared__ __align__(128) unsigned char att_smem[];
  float* us = reinterpret_cast<float*>(att_smem);     // Tn*E
  float* dcs = us + (long)Tn * E;                      // Tn*E
  float* ws = dcs + (long)Tn * E;                      // Tn*S
  float* dss = ws + (long)Tn * S;                      // Tn*S
  const int tid = threadIdx.x, b = blockIdx.x;
  for (int i = tid; i < Tn * E; i += ATT_THREADS) { const int t = i / E, e = i - t * E; us[i] = u[((long)t * B + b) * E + e]; dcs[i] = dctx[((long)t * B + b) * lddctx + e]; }
  for (int i = tid; i < Tn * S; i += ATT_THREADS) { const int t = i / S, l = i - t * S; ws[i] = attw[((long)t * B + b) * S + l]; dss[i] = ds[((long)t * B + b) * S + l]; }
  __syncthreads();
  const long base = (long)b * S * E;
  for (int idx = tid; idx < S * E; idx += ATT_THREADS) {
    const int l = idx / E, e = idx - l * E;
    const float p = P[base + idx];
    float aP = 0.f, aF = 0.f;
    for (int t = 0; t < Tn; ++t) {
      aP = fmaf(dss[t * S + l], Math<T>::dtanh_(p + us[t * E + e]), aP);
      aF = fmaf(ws[t * S + l], dcs[t * E + e], aF);
    }
    dP[base + idx] = from_f<T>(aP);
    dF[base + idx] = aF;
  }
}

// Register version of the pass above for Tn <= TMAX: a thread owns one column e and keeps u[t,e] and dctx[t,e] of ALL steps in
// registers (they do not depend on the token), so the inner loop over steps is two broadcast 16-byte shared loads (ds, w,
// stored [token][step]) per four steps plus the MUFU math: ~10 instructions per (token, column, step) instead of ~24 with
// the operands in shared memory.  grid (B, token splits): blockIdx.y owns a contiguous range of tokens.
template <typename T, int TMAX>
__global__ void __launch_bounds__(ATT_THREADS, TMAX <= 20 ? 4 : 2)
attn_post_reg_kernel(const float* __restrict__ P, const float* __restrict__ u /*(T,B,E)*/, const float* __restrict__ dctx /*(T,B,.) pitch lddctx*/, long lddctx,
                     const float* __restrict__ attw /*(T,B,S)*/, const float* __restrict__ ds /*(T,B,S)*/,
                     int Tn, int B, int S, int E, T* __restrict__ dP, float* __restrict__ dF) {
  extern __shared__ __align__(128) unsigned char att_smem[];
  const int tid = threadIdx.x, b = blockIdx.x;
  const int per = (S + gridDim.y - 1) / gridDim.y, l0 = blockIdx.y * per, l1 = min(S, l0 + per), nl = l1 - l0;
  if (nl <= 0) return;
  const int TP = (Tn + 3) & ~3;
  float* dsT = reinterpret_cast<float*>(att_smem);      // [nl][TP]
  float* wT = dsT + per * TP;                           // [nl][TP]
  for (int i = tid; i < nl * TP; i += ATT_THREADS) {
    const int ll = i / TP, t = i - ll * TP;
    const long g = ((long)t * B + b) * S + l0 + ll;
    dsT[i] = t < Tn ? ds[g] : 0.f;
    wT[i] = t < Tn ? attw[g] : 0.f;
  }
  __syncthreads();
  const long base = (long)b * S * E;
  for (int e = tid; e < E; e += ATT_THREADS) {
    float ur[TMAX], dcr[TMAX];
#pragma unroll
    for (int t = 0; t < TMAX; ++t) {
      ur[t] = t < Tn ? u[((long)t * B + b) * E + e] : 0.f;
      dcr[t] = t < Tn ? dctx[((long)t * B + b) * lddctx + e] : 0.f;
    }
    float p_next = P[base + (long)l0 * E + e];
#pragma unroll 1
    for (int l = l0; l < l1; ++l) {
      const float p = p_next;
      if (l + 1 < l1) p_next = P[base + (long)(l + 1) * E + e];      // next token's row is in flight under this one's MUFU work
      const float4* d4p = reinterpret_cast<const float4*>(dsT + (l - l0) * TP);
      const float4* w4p = reinterpret_cast<const float4*>(wT + (l - l0) * TP);
      float aP = 0.f, aF = 0.f;
#pragma unroll
      for (int t4 = 0; t4 < TMAX; t4 += 4) {
        if (t4 < TP) {
          const float4 d4 = d4p[t4 >> 2], w4 = w4p[t4 >> 2];
          const float dd[4] = {d4.x, d4.y, d4.z, d4.w}, ww[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            aP = fmaf(dd[j], Math<T>::dtanh_(p + ur[t4 + j]), aP);
            aF = fmaf(ww[j], dcr[t4 + j], aF);
          }
        }
      }
      dP[base + (long)l * E + e] = from_f<T>(aP);
      dF[base + (long)l * E + e] = aF;
    }
  }
}

// ======================================================================================
// attention_combine folded into layer 0 (oracle/manual_backward.py v2):  b_x = W_ih0 b_c + b_ih0 + b_hh0  (interleaved rows),
// and the pieces of its adjoint that are not contractions:  db_c = W_ih0^T db_x,  dW_ih0 += db_x (x) b_c   (natural row order)
// ======================================================================================
__global__ void __launch_bounds__(256)
bias_fold_kernel(const float* __restrict__ w_ih0, const float* __restrict__ b_c, const float* __restrict__ b_ih, const float* __restrict__ b_hh,
                 int H, int E, float* __restrict__ bx) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= 4 * H) return;
  const int src = (warp & 3) * H + (warp >> 2);           // interleaved row `warp` <- gate-major row `src`
  float a = 0.f;
  for (int e = lane; e < E; e += 32) a = fmaf(w_ih0[(long)src * E + e], b_c[e], a);
  a = warp_sum(a);
  if (lane == 0) bx[warp] = a + b_ih[src] + b_hh[src];
}
// db_c[e] = sum_n W_ih0[n,e] dbx[n]:  grid (ceil(E/32), row splits), 8 row lanes per block, partial sums added atomically
// into a zeroed db_c (E floats)
__global__ void __launch_bounds__(256)
bias_fold_bwd_kernel(const float* __restrict__ w_ih0, const float* __restrict__ dbx, int H4, int E, float* __restrict__ db_c) {
  __shared__ float red[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5, e = blockIdx.x * 32 + tx;
  const int per = (H4 + gridDim.y - 1) / gridDim.y, n0 = blockIdx.y * per, n1 = min(H4, n0 + per);
  float a = 0.f;
  if (e < E) for (int n = n0 + ty; n < n1; n += 8) a = fmaf(w_ih0[(long)n * E + e], dbx[n], a);
  red[ty][tx] = a;
  __syncthreads();
  if (ty == 0 && e < E) { float s = 0.f; for (int i = 0; i < 8; ++i) s += red[i][tx]; atomicAdd(db_c + e, s); }
}
// dW[n,e] += dbx[n] * b_c[e]
__global__ void __launch_bounds__(256)
rank1_add_kernel(float* __restrict__ dW, const float* __restrict__ dbx, const float* __restrict__ b_c, long rows, int E) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < rows * E; i += (long)gridDim.x * blockDim.x) {
    long n; int e; divmod_idx(i, E, n, e);
    dW[i] = fmaf(dbx[n], b_c[e], dW[i]);
  }
}

// ======================================================================================
// LSTM cell adjoint.  Gate storage is INTERLEAVED: element (b, 4j+g) is gate g (i,f,g,o) of hidden unit j.
// (The forward cell is the epilogue of the gate GEMM: gemm.cuh LstmEpi.)
// ======================================================================================
// dh = [carry] + [dh_b * mask] + [dh_ext] + [dh_hid] + [dh_q]; then the cell adjoint; dc is updated in place.
// The forward's saves (gates, c), dh_ext and dh_hid are complete before the reverse recurrence starts, so they are loaded (and
// tanh(c) evaluated) BEFORE griddepcontrol.wait; only the carried gradients (carry, above, dq, dc) wait for the previous kernel.
template <typename T> struct Gate4;
template <> struct Gate4<bf16> {
  static __device__ __forceinline__ void load(const bf16* p, float (&v)[4]) {
    const uint2 a = *reinterpret_cast<const uint2*>(p);
    v[0] = bf16_lo(a.x); v[1] = bf16_hi(a.x); v[2] = bf16_lo(a.y); v[3] = bf16_hi(a.y);
  }
  static __device__ __forceinline__ void store(bf16* p, const float (&v)[4]) {
    *reinterpret_cast<uint2*>(p) = make_uint2(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]));
  }
};
template <> struct Gate4<float> {
  static __device__ __forceinline__ void load(const float* p, float (&v)[4]) {
    const float4 a = *reinterpret_cast<const float4*>(p); v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
  }
  static __device__ __forceinline__ void store(float* p, const float (&v)[4]) { *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]); }
};

template <typename T>
__global__ void __launch_bounds__(256)
lstm_pointwise_bwd_kernel(const T* __restrict__ gates, const float* __restrict__ c_prev, const float* __restrict__ c_cur,
                          float* __restrict__ dc, int dc_is_zero,
                          const float* __restrict__ dh_carry, long ld_carry, const float* __restrict__ dh_above, long ld_above,
                          const float* __restrict__ dh_ext, const T* __restrict__ dh_hid, const T* __restrict__ dh_q, long ld_q,
                          T* __restrict__ dgates, int B, int H, float drop_p, uint64_t seed, uint32_t site, long row_base,
                          const unsigned long long* __restrict__ seed_dev, const int* __restrict__ steps, int step) {
  pdl_launch_dependents();
  if (steps != nullptr) {                      // variable-length batch (api.cu, invariants I1 and I4)
    const int n = __ldg(steps);
    if (step >= n) { pdl_wait(); return; }
    if (step == n - 1) { dc_is_zero = 1; dh_carry = nullptr; dh_q = nullptr; }   // the batch's last step: nothing flows back into it
  }
  if (drop_p > 0.f) seed = drop_seed(seed, seed_dev);
  const long total = (long)B * H;
  const float inv_keep = drop_p > 0.f ? 1.0f / (1.0f - drop_p) : 1.0f;
  struct Saved { float gt[4]; float tc, cp, dh_fixed, mask; };
  auto load_saved = [&](long idx, Saved& sv) {
    const long b = (long)((unsigned)idx / (unsigned)H); const int j = (int)(idx - b * H);      // B * H < 2^31: 32-bit division
    Gate4<T>::load(gates + b * 4 * H + 4 * j, sv.gt);
    sv.tc = Math<T>::tanh_(c_cur[idx]);
    sv.cp = c_prev[idx];
    float d = 0.f;
    if (dh_ext) d += dh_ext[idx];
    if (dh_hid) d += to_f<T>(dh_hid[idx]);
    sv.dh_fixed = d;
    sv.mask = (dh_above && drop_p > 0.f) ? dropout_scale(seed, site, (uint64_t)((row_base + b) * H + j), drop_p, inv_keep) : 1.0f;
  };
  const long idx0 = (long)blockIdx.x * blockDim.x + threadIdx.x;
  Saved sv;
  if (idx0 < total) load_saved(idx0, sv);
  pdl_wait();
  for (long idx = idx0; idx < total; idx += (long)gridDim.x * blockDim.x) {
    if (idx != idx0) load_saved(idx, sv);
    const long b = (long)((unsigned)idx / (unsigned)H); const int j = (int)(idx - b * H);
    float dh = sv.dh_fixed;
    if (dh_carry) dh += __ldcg(dh_carry + b * ld_carry + j);
    if (dh_above) dh += __ldcg(dh_above + b * ld_above + j) * sv.mask;
    if (dh_q) dh += to_f<T>(dh_q[b * ld_q + j]);
    const float i = sv.gt[0], f = sv.gt[1], g = sv.gt[2], o = sv.gt[3], tc = sv.tc;
    const float dcc = (dc_is_zero ? 0.f : __ldcg(dc + idx)) + dh * o * (1.0f - tc * tc);
    const float dg[4] = {dcc * g * i * (1.0f - i), dcc * sv.cp * f * (1.0f - f), dcc * i * (1.0f - g * g), dh * tc * o * (1.0f - o)};
    Gate4<T>::store(dgates + b * 4 * H + 4 * j, dg);
    dc[idx] = dcc * f;
  }
}

// ======================================================================================
// Variable-length batches (b2c.h *_steps entry points): the rows of the steps at and past the device step count, in several
// (steps, B, .) buffers, set to zero by one launch.  Segment y of the grid: step_words 4-byte words per step, n_steps steps.
// ======================================================================================
struct TailSeg { void* base; long step_words; int n_steps; };
constexpr int TAIL_MAX_SEGS = 8;
struct TailTable { TailSeg seg[TAIL_MAX_SEGS]; int n; };
__global__ void __launch_bounds__(256) tail_zero_kernel(const __grid_constant__ TailTable tab, const int* __restrict__ steps) {
  const TailSeg& s = tab.seg[blockIdx.y];
  const int n = min(max(__ldg(steps), 0), s.n_steps);
  uint32_t* p = reinterpret_cast<uint32_t*>(s.base);
  const long w0 = (long)n * s.step_words, w1 = (long)s.n_steps * s.step_words;
  // scalar words up to the first 16-byte boundary, 16-byte stores over the rest, scalar words after the last boundary
  long v0 = w0 + (long)((16 - ((uintptr_t)(p + w0) & 15)) & 15) / 4;
  if (v0 > w1) v0 = w1;
  const long nv = (w1 - v0) / 4;
  const long i0 = (long)blockIdx.x * blockDim.x + threadIdx.x, stride = (long)gridDim.x * blockDim.x;
  for (long i = w0 + i0; i < v0; i += stride) p[i] = 0u;
  uint4* q = reinterpret_cast<uint4*>(p + v0);
  for (long i = i0; i < nv; i += stride) q[i] = make_uint4(0u, 0u, 0u, 0u);
  for (long i = v0 + nv * 4 + i0; i < w1; i += stride) p[i] = 0u;
}

// ======================================================================================
// small glue
// ======================================================================================
// output_projection dropout (training only): o1 *= keep-mask/(1-p)
template <typename T>
__global__ void __launch_bounds__(256) dropout_inplace_kernel(T* __restrict__ x, long n, float p, uint64_t seed, uint32_t site,
                                                              const unsigned long long* __restrict__ seed_dev) {
  seed = drop_seed(seed, seed_dev);
  const float inv_keep = 1.0f / (1.0f - p);
  // 8 elements (16 bytes in bf16) per thread and iteration, the same per-element mask as the scalar form
  const long n8 = (((uintptr_t)x) & 15) == 0 ? (n >> 3) : 0;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long)gridDim.x * blockDim.x) {
    float v[8];
    Vec8<T>::load(x + i * 8, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] *= dropout_scale(seed, site, (uint64_t)(i * 8 + j), p, inv_keep);
    Vec8<T>::store(x + i * 8, v);
  }
  for (long i = n8 * 8 + (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    x[i] = from_f<T>(to_f<T>(x[i]) * dropout_scale(seed, site, (uint64_t)i, p, inv_keep));
}
// d(pre-ReLU, pre-dropout) = d(o1) * [o1 > 0] / (1-p)      (o1 is the saved post-ReLU, post-dropout activation)
template <typename T>
__global__ void __launch_bounds__(256) relu_bwd_inplace_kernel(T* __restrict__ d, const T* __restrict__ act, long n, float inv_keep) {
  // 8 elements (16 bytes in bf16) per thread and iteration; it sits on the main chain between the head's two backward GEMMs
  // (22 us with one 2-byte element per thread and iteration)
  const long n8 = ((((uintptr_t)d) & 15) == 0 && (((uintptr_t)act) & 15) == 0) ? (n >> 3) : 0;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long)gridDim.x * blockDim.x) {
    float dv[8], av[8];
    Vec8<T>::load(d + i * 8, dv); Vec8<T>::load(act + i * 8, av);
#pragma unroll
    for (int j = 0; j < 8; ++j) dv[j] = av[j] > 0.f ? dv[j] * inv_keep : 0.f;
    Vec8<T>::store(d + i * 8, dv);
  }
  for (long i = n8 * 8 + (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    d[i] = from_f<T>(to_f<T>(act[i]) > 0.f ? to_f<T>(d[i]) * inv_keep : 0.f);
}

// column sums of a (rows, cols) matrix with pitch ld: grid (ceil(cols/32), RS); partial[(rs, col)]
template <typename T>
__global__ void __launch_bounds__(256) colsum_partial_kernel(const T* __restrict__ A, long rows, int cols, long ld, float* __restrict__ partial) {
  __shared__ float red[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + tx;
  const long per = (rows + gridDim.y - 1) / gridDim.y;
  const long r0 = (long)blockIdx.y * per, r1 = (r0 + per < rows) ? r0 + per : rows;
  float a = 0.f;
  if (col < cols) for (long r = r0 + ty; r < r1; r += 8) a += to_f<T>(A[r * ld + col]);
  red[ty][tx] = a;
  __syncthreads();
  if (ty == 0 && col < cols) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += red[i][tx];
    partial[(long)blockIdx.y * cols + col] = s;
  }
}
__global__ void __launch_bounds__(256) colsum_final_kernel(const float* __restrict__ partial, int RS, int cols, float* __restrict__ out, float* __restrict__ out2,
                                                           int unperm_h = 0) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= cols) return;
  float s = 0.f;
  for (int r = 0; r < RS; ++r) s += partial[(long)r * cols + col];
  const int oc = unperm_h ? (col & 3) * unperm_h + (col >> 2) : col;      // interleaved gate column -> gate-major index
  out[oc] = s;
  if (out2) out2[oc] = s;
}

// Greedy feedback: tok[b] = argmax_v logits[b,v] (lowest index on ties, like torch.argmax); records the step's
// tokens and the caption length (first <END>) without leaving the device.
__global__ void __launch_bounds__(256)
argmax_feedback_kernel(const float* __restrict__ logits, int V, long ld, int64_t end_id, int t,
                       int64_t* __restrict__ cur_tok, int64_t* __restrict__ tokens_t, int32_t* __restrict__ lengths, int32_t* __restrict__ done) {
  __shared__ float bv[8]; __shared__ int bi[8];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* row = logits + (long)b * ld;
  float best = -INFINITY; int besti = 0x7fffffff;
  for (int v = tid; v < V; v += 256) { const float x = row[v]; if (x > best || (x == best && v < besti)) { best = x; besti = v; } }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o); const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
    if (ob > best || (ob == best && oi < besti)) { best = ob; besti = oi; }
  }
  if (lane == 0) { bv[warp] = best; bi[warp] = besti; }
  __syncthreads();
  if (tid == 0) {
    for (int i = 1; i < 8; ++i) if (bv[i] > best || (bv[i] == best && bi[i] < besti)) { best = bv[i]; besti = bi[i]; }
    if (besti == 0x7fffffff) besti = 0;      // all-NaN row
    cur_tok[b] = besti; tokens_t[b] = besti;
    if (t == 0) { done[b] = 0; lengths[b] = -1; }
    if (besti == end_id && !done[b]) { done[b] = 1; lengths[b] = t; }
  }
}
// Same feedback from the per-row partial (max, index) pairs the vocabulary-head GEMM's argmax epilogue leaves (gemm.cuh ArgmaxEpi):
// one warp per sample reduces its `nparts` partials with the same ordering (larger value, then lower index).
__global__ void __launch_bounds__(256)
argmax_parts_feedback_kernel(const float* __restrict__ pmax, const int* __restrict__ pidx, int nparts, int B, int64_t end_id, int t,
                             int64_t* __restrict__ cur_tok, int64_t* __restrict__ tokens_t, int32_t* __restrict__ lengths, int32_t* __restrict__ done) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  float best = -INFINITY; int besti = 0x7fffffff;
  for (int p = lane; p < nparts; p += 32) {
    const float x = pmax[(long)b * nparts + p]; const int i = pidx[(long)b * nparts + p];
    if (x > best || (x == best && i < besti)) { best = x; besti = i; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o); const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
    if (ob > best || (ob == best && oi < besti)) { best = ob; besti = oi; }
  }
  if (lane == 0) {
    if (besti == 0x7fffffff) besti = 0;      // all-NaN row
    cur_tok[b] = besti; tokens_t[b] = besti;
    if (t == 0) { done[b] = 0; lengths[b] = -1; }
    if (besti == end_id && !done[b]) { done[b] = 1; lengths[b] = t; }
  }
}
__global__ void bump_counter_kernel(unsigned long long* c) { *c += 1ull; }
__global__ void fill_i64_kernel(int64_t* p, long n, int64_t v) { for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) p[i] = v; }
__global__ void finish_lengths_kernel(int32_t* lengths, int B, int T) { const int b = blockIdx.x * blockDim.x + threadIdx.x; if (b < B && lengths[b] < 0) lengths[b] = T; }

}  // namespace b2c
