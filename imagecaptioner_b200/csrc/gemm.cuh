// Dense contractions of the hot path (kernel (2) of the north star).
//
//   C[m,n] = act( alpha * sum_k A(m,k) * B(n,k) + bias[n] ) + beta * C[m,n]
//
// Operand "majorness" (row-major storage everywhere):
//   A K-major : A(m,k) = A[m*lda + k]      A MN-major: A(m,k) = A[k*lda + m]
//   B K-major : B(n,k) = B[n*ldb + k]      B MN-major: B(n,k) = B[k*ldb + n]
// so  forward linear  y = x W^T        -> (A K, B K)
//     data gradient   dx = dy W        -> (A K, B MN)
//     weight gradient dW = dy^T x      -> (A MN, B MN)
//
// Two implementations, both sm_100a CUDA, chosen by the precision mode (not by backend):
//   * gemm_simt_kernel  — fp32 FFMA tiles; the fp32 parity mode (1e-4 / exact argmax) and any shape
//                         TMA cannot describe (row pitch not a multiple of 16 bytes).
//   * gemm_tc_kernel    — bf16 operands staged by TMA (SWIZZLE_128B) into a 4-stage mbarrier ring,
//                         tcgen05.mma (cta_group::1, M=128, N=64/128/256, K=16) accumulating fp32 in TMEM,
//                         tcgen05.ld epilogue with fused alpha / bias / ReLU / beta.
#pragma once
#include <type_traits>
#include "common.cuh"

namespace b2c {

// ======================================================================================
// Fused LSTM-cell epilogue.  With the gate rows of W_cat interleaved (row 4j+g = gate g of hidden unit j) four consecutive
// output columns of the gate contraction are the i,f,g,o pre-activations of ONE unit, so the epilogue that already holds
// them in registers finishes the cell: adds bias / the time-batched embedding addend, applies the gates, updates c in fp32
// and scatters h to the recurrent slot, the next layer's input (inter-layer dropout) and the top-layer output.
// ======================================================================================
struct LstmEpi {
  int enabled, H;
  const void* addend;          // (rows, 4H) operand type, interleaved columns, or null
  const float* bias;           // (4H) interleaved, or null
  const float* c_prev; float* c_out;
  void* gates_out;             // (rows, 4H) post-activation gates, interleaved (null in decode)
  void* h_rec; long ld_rec; void* h_next; long ld_next; void* h_top; long ld_top;
  float drop_p; unsigned long long seed; unsigned int site; long row_base;
  const unsigned long long* seed_dev;   // optional device step counter mixed into the seed (CUDA-graph replays)
  const float* addend32; long ld_addend32;   // optional fp32 addend (rows, >= 4H) with its own pitch: the recurrent half W_hh h_{t-1} of the
                                        // pre-activations when it was contracted ahead of time (tcgen05 path only)
  const int* steps; int step;           // variable-length recurrences: the launch does nothing when step >= *steps (any flavour; steps
                                        // null = always run).  Set from GemmArgs, see GemmStepScope.
};

// Validation (validate_student_model, reference src/train_student_kd.py:29-86) needs, per logits row, only the token-KD term, the CE
// term and the argmax.  The vocabulary-head GEMM can reduce every accumulator tile in its epilogue to per-row PARTIALS of those
// (online-softmax form) against the teacher logits it streams alongside, instead of writing the (T,B,V) logits that a second
// kernel would read back: 8 floats per (row, part), a part being the run of `cols_per_part` columns one epilogue thread drains.
//   my, s1 = sum e^{y-my}, sT = sum e^{(y-my)/Temp};  mz, sZ = sum e^{(z-mz)/Temp}, sA = sum e^{(z-mz)/Temp} ((z-mz) - (y-my))/Temp;
//   y[target] if the target column lies in the part; the part's argmax column (lowest index among equals).
// kd_eval_combine_kernel (loss_kernels.cuh) merges the parts of a row.  The descriptor travels in the LstmEpi slot: enabled == 3.
// The teacher logits are fp32 (epilogue flavour 3), bf16 (6) or f16 (7), each its own instantiation (see gemm_tc_kernel).
constexpr int EVAL_PART_FLOATS = 8;
struct EvalEpi { const void* teacher; const int64_t* targets; float* parts; float inv_temp; int nparts; int cols_per_part; int teacher_dtype; };

// Greedy decoding needs argmax_n C[m, n] only: the vocabulary-head GEMM can reduce every accumulator tile to per-row partial
// (max, index) pairs in its epilogue instead of writing the logits (41 MB per step at B = 2048, V = 5000, read again by the argmax
// kernel).  One partial per (row, part): a part is the run of `cols_per_part` columns one epilogue warp drains of one tile.
// The descriptor travels in the (otherwise unused) LstmEpi slot of the general instantiation: enabled == 2.
struct ArgmaxEpi { float* pmax; int* pidx; int nparts; int cols_per_part; };
inline LstmEpi pack_argmax(const ArgmaxEpi& a) {
  LstmEpi le{};
  le.enabled = 2; le.H = a.nparts; le.c_out = a.pmax; le.gates_out = a.pidx; le.ld_rec = a.cols_per_part;
  return le;
}
inline LstmEpi pack_eval(const EvalEpi& e) {
  LstmEpi le{};
  le.enabled = 3; le.H = e.nparts; le.c_out = e.parts; le.addend = e.teacher; le.h_rec = const_cast<int64_t*>(e.targets);
  le.ld_rec = e.cols_per_part; le.drop_p = e.inv_temp;
  return le;
}

// one hidden unit: pre[4] = i,f,g,o pre-activations (bias/addend already added) -> act[4], c, h
template <typename TL>
__device__ __forceinline__ void lstm_cell_unit(const float (&pre)[4], float c_prev, float (&act)[4], float& c, float& h) {
  act[0] = Math<TL>::sigmoid_(pre[0]); act[1] = Math<TL>::sigmoid_(pre[1]);
  act[2] = Math<TL>::tanh_(pre[2]);    act[3] = Math<TL>::sigmoid_(pre[3]);
  c = fmaf(act[1], c_prev, act[0] * act[2]);
  h = act[3] * Math<TL>::tanh_(c);
}

// ======================================================================================
// SIMT fp32-accumulate GEMM (any operand type, any majorness)
// ======================================================================================
constexpr int SG_BM = 64, SG_BN = 64, SG_BK = 16;

template <typename TA, typename TB, typename TC>
__global__ void __launch_bounds__(256)
gemm_simt_kernel(int M, int N, int K, float alpha, const TA* __restrict__ A, long lda, int a_mn,
                 const TB* __restrict__ B, long ldb, int b_mn, float beta, TC* __restrict__ C, long ldc,
                 const float* __restrict__ bias, int relu, int row_unperm_h, const __grid_constant__ LstmEpi le) {
  __shared__ float As[SG_BK][SG_BM + 4];
  __shared__ float Bs[SG_BK][SG_BN + 4];
  pdl_launch_dependents();
  pdl_wait();
  if (le.steps != nullptr && le.step >= __ldg(le.steps)) return;      // a step past the batch's length (after the wait: invariant I1, api.cu)
  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * SG_BM, n0 = blockIdx.x * SG_BN;
  const int tx = tid & 15, ty = tid >> 4;      // 16 x 16 threads, 4x4 outputs each
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < K; k0 += SG_BK) {
#pragma unroll
    for (int it = 0; it < (SG_BM * SG_BK) / 256; ++it) {
      const int idx = tid + it * 256;
      int mm, kk;
      if (a_mn) { kk = idx / SG_BM; mm = idx % SG_BM; } else { mm = idx / SG_BK; kk = idx % SG_BK; }
      const int gm = m0 + mm, gk = k0 + kk;
      float v = 0.f;
      if (gm < M && gk < K) v = to_f<TA>(a_mn ? A[(long)gk * lda + gm] : A[(long)gm * lda + gk]);
      As[kk][mm] = v;
    }
#pragma unroll
    for (int it = 0; it < (SG_BN * SG_BK) / 256; ++it) {
      const int idx = tid + it * 256;
      int nn, kk;
      if (b_mn) { kk = idx / SG_BN; nn = idx % SG_BN; } else { nn = idx / SG_BK; kk = idx % SG_BK; }
      const int gn = n0 + nn, gk = k0 + kk;
      float v = 0.f;
      if (gn < N && gk < K) v = to_f<TB>(b_mn ? B[(long)gk * ldb + gn] : B[(long)gn * ldb + gk]);
      Bs[kk][nn] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < SG_BK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  if (le.enabled) {                          // this thread's 4 columns are the 4 gates of hidden unit `unit` (N = 4H, N % 4 == 0)
    const int gn = n0 + tx * 4, unit = gn >> 2, H = le.H;
    if (gn >= N) return;
    const float inv_keep = le.drop_p > 0.f ? 1.0f / (1.0f - le.drop_p) : 1.0f;
    const uint64_t dseed = le.drop_p > 0.f ? drop_seed(le.seed, le.seed_dev) : 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int gm = m0 + ty * 4 + i;
      if (gm >= M) continue;
      float pre[4], act[4], c, h;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        pre[j] = acc[i][j];
        if (le.bias) pre[j] += le.bias[gn + j];
        if (le.addend) pre[j] += to_f<TA>(reinterpret_cast<const TA*>(le.addend)[(long)gm * N + gn + j]);
      }
      lstm_cell_unit<TA>(pre, le.c_prev[(long)gm * H + unit], act, c, h);
      le.c_out[(long)gm * H + unit] = c;
      if (le.gates_out) {
#pragma unroll
        for (int j = 0; j < 4; ++j) reinterpret_cast<TA*>(le.gates_out)[(long)gm * N + gn + j] = from_f<TA>(act[j]);
      }
      if (le.h_rec) reinterpret_cast<TA*>(le.h_rec)[(long)gm * le.ld_rec + unit] = from_f<TA>(h);
      if (le.h_next) {
        const float m = le.drop_p > 0.f ? dropout_scale(dseed, le.site, (uint64_t)((le.row_base + gm) * H + unit), le.drop_p, inv_keep) : 1.0f;
        reinterpret_cast<TA*>(le.h_next)[(long)gm * le.ld_next + unit] = from_f<TA>(h * m);
      }
      if (le.h_top) reinterpret_cast<TA*>(le.h_top)[(long)gm * le.ld_top + unit] = from_f<TA>(h);
    }
    return;
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gm = m0 + ty * 4 + i;
    if (gm >= M) continue;
    const long orow = row_unperm_h ? (long)(gm & 3) * row_unperm_h + (gm >> 2) : (long)gm;     // interleaved row -> gate-major row
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gn = n0 + tx * 4 + j;
      if (gn >= N) continue;
      float v = alpha * acc[i][j];
      if (bias) v += bias[gn];
      if (relu) v = fmaxf(v, 0.f);
      if (beta != 0.f) v += beta * to_f<TC>(C[orow * ldc + gn]);
      C[orow * ldc + gn] = from_f<TC>(v);
    }
  }
}

// ======================================================================================
// tcgen05 / TMEM / TMA bf16 GEMM
// ======================================================================================
constexpr int TC_BM = 128, TC_BK = 64, TC_THREADS = 320;     // warp 0 TMA, warp 1 MMA, warps 2-9 epilogue (two per TMEM lane quarter)
constexpr uint32_t TC_A_BYTES = TC_BM * TC_BK * 2;     // 16 KiB per stage

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               :: "r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" :: "l"(map) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// Shared-memory matrix descriptor (SM100 UMMA), SWIZZLE_128B, version 1.
//   K-major  tile: rows of 64 bf16 (128 B), 8-row swizzle atoms 1024 B apart      -> SBO = 1024, LBO unused (1)
//   MN-major tile: K-rows of 64 MN elements (128 B); 8-K-row atoms 1024 B apart (SBO),
//                  consecutive 64-wide MN chunks `lbo` bytes apart (LBO)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;          // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;          // layout type SWIZZLE_128B
  return d;
}

constexpr int TC_EPI_PITCH = 144;                       // bytes per staged row: 128 B of payload + 16 B pad (bank-conflict free)
constexpr int TC_EPI_WARPS = 8;
constexpr int TC_EPI_BYTES = TC_EPI_WARPS * 32 * TC_EPI_PITCH;    // one 32-row staging tile per epilogue warp

template <int BN> struct TcCfg {
#ifndef B2C_STAGES64
#define B2C_STAGES64 4
#endif
#ifndef B2C_STAGES128
#define B2C_STAGES128 4
#endif
  static constexpr int STAGES = BN == 256 ? 3 : (BN == 128 ? B2C_STAGES128 : B2C_STAGES64);      // 48 KB stages at BN = 256: three fit beside the epilogue staging
  static constexpr uint32_t B_BYTES = BN * TC_BK * 2;
  static constexpr uint32_t STAGE_BYTES = TC_A_BYTES + B_BYTES;
  static constexpr uint32_t TMEM_COLS = 2 * BN;          // two accumulator stages (128 / 256 / 512 columns)
  static constexpr size_t SMEM_BYTES = (size_t)STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/ + TC_EPI_BYTES;
};

__device__ __forceinline__ uint4 epi_combine_bf16(uint4 acc, uint4 old, float beta) {
  uint4 o;
  o.x = pack_bf16(bf16_lo(acc.x) + beta * bf16_lo(old.x), bf16_hi(acc.x) + beta * bf16_hi(old.x));
  o.y = pack_bf16(bf16_lo(acc.y) + beta * bf16_lo(old.y), bf16_hi(acc.y) + beta * bf16_hi(old.y));
  o.z = pack_bf16(bf16_lo(acc.z) + beta * bf16_lo(old.z), bf16_hi(acc.z) + beta * bf16_hi(old.z));
  o.w = pack_bf16(bf16_lo(acc.w) + beta * bf16_lo(old.w), bf16_hi(acc.w) + beta * bf16_hi(old.w));
  return o;
}
__device__ __forceinline__ uint4 epi_combine_f32(uint4 acc, uint4 old, float beta) {
  uint4 o;
  o.x = __float_as_uint(__uint_as_float(acc.x) + beta * __uint_as_float(old.x));
  o.y = __float_as_uint(__uint_as_float(acc.y) + beta * __uint_as_float(old.y));
  o.z = __float_as_uint(__uint_as_float(acc.z) + beta * __uint_as_float(old.z));
  o.w = __float_as_uint(__uint_as_float(acc.w) + beta * __uint_as_float(old.w));
  return o;
}

// Persistent: grid = min(work items, SMs); work item = (M tile, N tile, K split).  With K splits > 1 (fp32 output only) every split adds its partial tile into C with
// red.global.add.f32; the host has zeroed C (beta == 0) or C already holds the value to accumulate onto (beta == 1).
// LSTM = true: the instantiation used by the recurrence (fused cell epilogue only); false: the general epilogues only.  Two
// kernels instead of one with both keep each one's code small: the recurrence's kernels are short and run back to back with
// other kernels, so every launch starts with a cold instruction cache.
// EPI selects ONE epilogue flavour per instantiation: 0 = the general store epilogues, 1 = fused LSTM cell, 2 = argmax partials (greedy
// decode), 3 = validation partials (6 / 7: the same with bf16 / f16 teacher logits).  Each flavour is its own kernel so none of them carries the others' code: these kernels run back to back
// with cold instruction caches, and code that is never executed still costs (round 1: 66 -> 23-32 KB per kernel bought 40 us per step;
// round 2: ~300 inlined instructions of a dropout hash in the general epilogue cost 8 % of the whole step).
template <int BN, bool A_MN, bool B_MN, typename TC, int EPI = 0>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               int M, int N, int K, float alpha, float beta, TC* __restrict__ C, long ldc,
               const float* __restrict__ bias, int relu, int kb_per_split, int tiles_m, int tiles_n, int splits,
               int row_unperm_h, const __grid_constant__ LstmEpi le) {
  constexpr bool LSTM = (EPI == 1 || EPI == 5);          // 5: the cell epilogue without the inter-layer dropout code (eval mode, p = 0)
  constexpr bool LSTM_DROP = (EPI == 1);
  using Cfg = TcCfg<BN>;
  constexpr int TC_STAGES = Cfg::STAGES;
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* base = reinterpret_cast<unsigned char*>(((uintptr_t)smem_dyn + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(base + (size_t)TC_STAGES * Cfg::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + TC_STAGES;
  uint64_t* tfull_bar = empty_bar + TC_STAGES;          // [2] accumulator stage complete (MMA -> epilogue)
  uint64_t* tempty_bar = tfull_bar + 2;                 // [2] accumulator stage drained  (epilogue -> MMA), one arrival per epilogue warp
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  unsigned char* epi_stage = base + (size_t)TC_STAGES * Cfg::STAGE_BYTES + 256;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_kb_total = (K + TC_BK - 1) / TC_BK;
  const int tiles_mn = tiles_m * tiles_n;
  const int total = tiles_mn * splits;                  // work items (M tile, N tile, K split), dealt round-robin to the CTAs
  const bool split = splits > 1;

  pdl_launch_dependents();                   // the next kernel on the chain may begin its own prologue
  // a step past the batch's length: no barrier, no TMEM, but still griddepcontrol.wait, so that this grid completes only after its
  // predecessors did (invariant I1, api.cu).  The step count is read before the wait: it is written before the recurrence's first,
  // fully serialised kernel starts, and nothing on the chain writes it.
  if (le.steps != nullptr && le.step >= __ldg(le.steps)) { pdl_wait(); return; }
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB); }
  if (warp == 1) {
    if (lane == 0) {
      for (int i = 0; i < TC_STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
      for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], TC_EPI_WARPS); }
      fence_barrier_init();
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(tmem_slot)), "r"(Cfg::TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();                                // prologue done; operands / C of the previous kernels are complete from here on

  if (warp == 0) {
    // ------------------------------------------------ TMA producer
    if (lane == 0) {
      int it = 0;
      for (int w = blockIdx.x; w < total; w += gridDim.x) {
        const int sp = w / tiles_mn, rem = w - sp * tiles_mn;
        const int m0 = (rem / tiles_n) * TC_BM, n0 = (rem % tiles_n) * BN;
        const int kb_begin = sp * kb_per_split, kb_end = min(num_kb_total, kb_begin + kb_per_split);
        for (int kb = kb_begin; kb < kb_end; ++kb, ++it) {
          const int s = it % TC_STAGES; const uint32_t ph = (it / TC_STAGES) & 1;
          mbar_wait(&empty_bar[s], ph ^ 1);
          unsigned char* sa = base + (size_t)s * Cfg::STAGE_BYTES;
          unsigned char* sb = sa + TC_A_BYTES;
          mbar_arrive_expect_tx(&full_bar[s], Cfg::STAGE_BYTES);
          const int k0 = kb * TC_BK;
          if (!A_MN) {
            tma_load_2d(sa, &tmA, k0, m0, &full_bar[s]);                      // box {64 k, 128 m}
          } else {
#pragma unroll
            for (int j = 0; j < TC_BM / 64; ++j) tma_load_2d(sa + j * 8192, &tmA, m0 + j * 64, k0, &full_bar[s]);   // box {64 m, 64 k}
          }
          if (!B_MN) {
            tma_load_2d(sb, &tmB, k0, n0, &full_bar[s]);                      // box {64 k, BN n}
          } else {
#pragma unroll
            for (int j = 0; j < BN / 64; ++j) tma_load_2d(sb + j * 8192, &tmB, n0 + j * 64, k0, &full_bar[s]);      // box {64 n, 64 k}
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------ MMA issuer (one thread), two TMEM accumulator stages
    if (lane == 0) {
      constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((A_MN ? 1u : 0u) << 15) | ((B_MN ? 1u : 0u) << 16) |
                                 ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
      int it = 0, t = 0;
      for (int w = blockIdx.x; w < total; w += gridDim.x, ++t) {
        const int sp = w / tiles_mn;
        const int kb_begin = sp * kb_per_split, kb_end = min(num_kb_total, kb_begin + kb_per_split);
        const int as = t & 1; const uint32_t aph = (t >> 1) & 1;
        mbar_wait(&tempty_bar[as], aph ^ 1);                                  // the epilogue has drained this accumulator stage
        tc_fence_after();
        const uint32_t tacc = tmem_base + (uint32_t)(as * BN);
        for (int kb = kb_begin; kb < kb_end; ++kb, ++it) {
          const int s = it % TC_STAGES; const uint32_t ph = (it / TC_STAGES) & 1;
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(base + (size_t)s * Cfg::STAGE_BYTES);
          const uint32_t sb = sa + TC_A_BYTES;
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k) {
            const uint64_t adesc = A_MN ? make_smem_desc(sa + k * 2048, 8192, 1024) : make_smem_desc(sa + k * 32, 16, 1024);
            const uint64_t bdesc = B_MN ? make_smem_desc(sb + k * 2048, 8192, 1024) : make_smem_desc(sb + k * 32, 16, 1024);
            tc_mma_bf16(tacc, adesc, bdesc, idesc, (kb > kb_begin || k > 0) ? 1u : 0u);
          }
          tc_commit(&empty_bar[s]);            // frees the smem slot once these MMAs have read it
        }
        tc_commit(&tfull_bar[as]);             // accumulator stage complete
      }
    }
  } else {
    // ------------------------------------------------ epilogue: warps 2..5 -> TMEM lane quarters (warp % 4).
    // TMEM -> registers (one accumulator row per lane) -> alpha/bias/ReLU -> 128-byte row chunks staged in shared memory
    // -> written out with each quarter-warp covering one contiguous 128-byte row segment (full sectors, 16-byte accesses).
    const int q = warp & 3;                              // TMEM lane quarter this warp may read (warp id % 4)
    const int half = (warp - 2) >> 2;                    // two warps per quarter: each drains half of the tile's columns
    unsigned char* my = epi_stage + (size_t)(warp - 2) * 32 * TC_EPI_PITCH;
    constexpr int PER = 16 / (int)sizeof(TC);           // elements per 16-byte unit: 8 (bf16) or 4 (fp32)
    constexpr int CH = 128 / (int)sizeof(TC);           // columns per staged chunk: 64 (bf16) or 32 (fp32)
    const bool vec_ok = (((uintptr_t)C) % 16 == 0) && ((ldc * (long)sizeof(TC)) % 16 == 0);
    int t = 0;
    for (int w = blockIdx.x; w < total; w += gridDim.x, ++t) {
    const int sp = w / tiles_mn, rem = w - sp * tiles_mn;
    const int m0 = (rem / tiles_n) * TC_BM, n0 = (rem % tiles_n) * BN;
    const int as = t & 1; const uint32_t aph = (t >> 1) & 1;
    const bool add_bias = (bias != nullptr) && (sp == 0);
    // LSTM epilogue: the operands that do not come from the MMA (bias, the time-batched addend, c_{t-1}) of this warp's first 32
    // columns are fetched BEFORE waiting for the accumulator, so their L2 latency runs under the main loop.
    [[maybe_unused]] float4 pre_b[8]; [[maybe_unused]] uint4 pre_a[4]; [[maybe_unused]] float4 pre_c0, pre_c1; [[maybe_unused]] float4 pre_r[8];
    [[maybe_unused]] int pre_ci = -1;
    if constexpr (LSTM) {
      constexpr int NC32 = BN / 32, C32_PER = (NC32 + 1) / 2;
      const int ci = half * C32_PER, col0 = n0 + ci * 32, grow = m0 + q * 32 + lane;
      if (ci < NC32 && col0 < N && grow < M) {
        pre_ci = ci;
        if (le.bias) {
#pragma unroll
          for (int j = 0; j < 8; ++j) pre_b[j] = *reinterpret_cast<const float4*>(le.bias + col0 + 4 * j);
        }
        if (le.addend) {
          const uint4* ap = reinterpret_cast<const uint4*>(reinterpret_cast<const bf16*>(le.addend) + (long)grow * N + col0);
#pragma unroll
          for (int j = 0; j < 4; ++j) pre_a[j] = ap[j];
        }
        if (le.addend32) {
          const float4* rp = reinterpret_cast<const float4*>(le.addend32 + (long)grow * le.ld_addend32 + col0);
#pragma unroll
          for (int j = 0; j < 8; ++j) pre_r[j] = __ldcg(rp + j);
        }
        pre_c0 = *reinterpret_cast<const float4*>(le.c_prev + (long)grow * le.H + (col0 >> 2));
        pre_c1 = *reinterpret_cast<const float4*>(le.c_prev + (long)grow * le.H + (col0 >> 2) + 4);
      }
    }
    mbar_wait(&tfull_bar[as], aph);
    tc_fence_after();
    const uint32_t tacc = tmem_base + (uint32_t)(as * BN) + ((uint32_t)(q * 32) << 16);
    if constexpr (LSTM) {
      // ---- fused LSTM cell: 32 accumulator columns = 8 hidden units x (i,f,g,o); straight from TMEM to the cell state buffers
      const int H = le.H, N4 = N;                        // N == 4H
      const int grow = m0 + q * 32 + lane;
      [[maybe_unused]] const float inv_keep = (LSTM_DROP && le.drop_p > 0.f) ? 1.0f / (1.0f - le.drop_p) : 1.0f;
      [[maybe_unused]] const uint64_t dseed = (LSTM_DROP && le.drop_p > 0.f) ? drop_seed(le.seed, le.seed_dev) : 0;
      constexpr int NC32 = BN / 32, C32_PER = (NC32 + 1) / 2;
#pragma unroll 1
      for (int ci = half * C32_PER; ci < (half + 1) * C32_PER && ci < NC32; ++ci) {
        const int col0 = n0 + ci * 32;
        if (col0 >= N) break;
        float v[32];
        tmem_ld32(tacc + (uint32_t)(ci * 32), v);
        if (grow < M) {
          const bool pre = (ci == pre_ci);
          if (le.bias) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 b4 = pre ? pre_b[j >> 2] : *reinterpret_cast<const float4*>(le.bias + col0 + j);
              v[j] += b4.x; v[j + 1] += b4.y; v[j + 2] += b4.z; v[j + 3] += b4.w;
            }
          }
          if (le.addend) {
            const uint4* ap = reinterpret_cast<const uint4*>(reinterpret_cast<const bf16*>(le.addend) + (long)grow * N4 + col0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint4 a = pre ? pre_a[j] : ap[j];
              v[j * 8 + 0] += bf16_lo(a.x); v[j * 8 + 1] += bf16_hi(a.x); v[j * 8 + 2] += bf16_lo(a.y); v[j * 8 + 3] += bf16_hi(a.y);
              v[j * 8 + 4] += bf16_lo(a.z); v[j * 8 + 5] += bf16_hi(a.z); v[j * 8 + 6] += bf16_lo(a.w); v[j * 8 + 7] += bf16_hi(a.w);
            }
          }
          if (le.addend32) {
            const float4* rp = reinterpret_cast<const float4*>(le.addend32 + (long)grow * le.ld_addend32 + col0);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 r4 = pre ? pre_r[j] : __ldcg(rp + j);
              v[4 * j] += r4.x; v[4 * j + 1] += r4.y; v[4 * j + 2] += r4.z; v[4 * j + 3] += r4.w;
            }
          }
          const int u0 = col0 >> 2;
          const float4 cp0 = pre ? pre_c0 : *reinterpret_cast<const float4*>(le.c_prev + (long)grow * H + u0);
          const float4 cp1 = pre ? pre_c1 : *reinterpret_cast<const float4*>(le.c_prev + (long)grow * H + u0 + 4);
          const float cp[8] = {cp0.x, cp0.y, cp0.z, cp0.w, cp1.x, cp1.y, cp1.z, cp1.w};
          float cn[8], hn[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            float pre[4] = {v[4 * u], v[4 * u + 1], v[4 * u + 2], v[4 * u + 3]}, act[4];
            lstm_cell_unit<bf16>(pre, cp[u], act, cn[u], hn[u]);
            v[4 * u] = act[0]; v[4 * u + 1] = act[1]; v[4 * u + 2] = act[2]; v[4 * u + 3] = act[3];
          }
          *reinterpret_cast<float4*>(le.c_out + (long)grow * H + u0) = make_float4(cn[0], cn[1], cn[2], cn[3]);
          *reinterpret_cast<float4*>(le.c_out + (long)grow * H + u0 + 4) = make_float4(cn[4], cn[5], cn[6], cn[7]);
          if (le.gates_out) {
            uint4* gp = reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(le.gates_out) + (long)grow * N4 + col0);
#pragma unroll
            for (int j = 0; j < 4; ++j)
              gp[j] = make_uint4(pack_bf16(v[j * 8], v[j * 8 + 1]), pack_bf16(v[j * 8 + 2], v[j * 8 + 3]), pack_bf16(v[j * 8 + 4], v[j * 8 + 5]), pack_bf16(v[j * 8 + 6], v[j * 8 + 7]));
          }
          const uint4 hp = make_uint4(pack_bf16(hn[0], hn[1]), pack_bf16(hn[2], hn[3]), pack_bf16(hn[4], hn[5]), pack_bf16(hn[6], hn[7]));
          if (le.h_rec) *reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(le.h_rec) + (long)grow * le.ld_rec + u0) = hp;
          if (le.h_top) *reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(le.h_top) + (long)grow * le.ld_top + u0) = hp;
          if (le.h_next) {
            uint4 hd = hp;
            if (LSTM_DROP && le.drop_p > 0.f) {
              float hm[8];
#pragma unroll
              for (int u = 0; u < 8; ++u) hm[u] = hn[u] * dropout_scale(dseed, le.site, (uint64_t)((le.row_base + grow) * H + u0 + u), le.drop_p, inv_keep);
              hd = make_uint4(pack_bf16(hm[0], hm[1]), pack_bf16(hm[2], hm[3]), pack_bf16(hm[4], hm[5]), pack_bf16(hm[6], hm[7]));
            }
            *reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(le.h_next) + (long)grow * le.ld_next + u0) = hd;
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[as]);
      continue;
    } else {
    constexpr int NCHUNK = BN / CH;                      // 128-byte column chunks per tile row
    constexpr int C_PER = (NCHUNK + 1) / 2;
    if constexpr (EPI == 3 || EPI == 6 || EPI == 7) {
      // ---- validation epilogue (EvalEpi): this thread owns one logits row and C_PER * CH columns of it
      using TZ = typename std::conditional<EPI == 3, float, typename std::conditional<EPI == 6, bf16, f16>::type>::type;
      const TZ* zt = reinterpret_cast<const TZ*>(le.addend);
      const int64_t* tg = reinterpret_cast<const int64_t*>(le.h_rec);
      float* parts = le.c_out;
      const int nparts = le.H, grow = m0 + q * 32 + lane;
      const float inv_temp = le.drop_p, L2E = 1.4426950408889634f, kT = inv_temp * L2E;
      const bool row_ok = grow < M;
      const long tcol = row_ok ? (long)tg[grow] : -1;
      float my = -INFINITY, s1 = 0.f, sT = 0.f, mz = -INFINITY, sZ = 0.f, sA = 0.f, ytgt = 0.f; int bidx = 0x7fffffff;
#pragma unroll 1
      for (int ci = half * C_PER; ci < (half + 1) * C_PER && ci < NCHUNK; ++ci) {
#pragma unroll 1
        for (int h = 0; h < CH / 32; ++h) {
          const int colb = n0 + ci * CH + h * 32;
          if (colb >= N) break;                             // warp-uniform
          float v[32], z[32];
          tmem_ld32(tacc + (uint32_t)(ci * CH + h * 32), v);
          const bool full = colb + 32 <= N;
          const TZ* zr = zt + (long)(row_ok ? grow : 0) * N + colb;
          if (full && ((((uintptr_t)zr) & 15) == 0)) {
            if constexpr (sizeof(TZ) == 4) {
#pragma unroll
              for (int j = 0; j < 8; ++j) { const float4 t4 = __ldg(reinterpret_cast<const float4*>(zr) + j); z[4 * j] = t4.x; z[4 * j + 1] = t4.y; z[4 * j + 2] = t4.z; z[4 * j + 3] = t4.w; }
            } else {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const uint4 t4 = __ldg(reinterpret_cast<const uint4*>(zr) + j);
                const uint32_t w[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) { z[8 * j + 2 * k] = lo_f<TZ>(w[k]); z[8 * j + 2 * k + 1] = hi_f<TZ>(w[k]); }
              }
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) z[j] = (colb + j < N) ? to_f<TZ>(__ldg(zr + j)) : -INFINITY;
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = (colb + j < N) ? fmaf(alpha, v[j], bias != nullptr ? __ldg(bias + colb + j) : 0.f) : -INFINITY;
          // chunk-local maxima, then merge the running sums onto the new maxima
          float cmy = v[0], cmz = z[0];
#pragma unroll
          for (int j = 1; j < 32; ++j) { cmy = fmaxf(cmy, v[j]); cmz = fmaxf(cmz, z[j]); }
          if (cmy > my) {                                   // strict: an equal later value keeps the earlier (lower) column
#pragma unroll
            for (int j = 31; j >= 0; --j) if (v[j] == cmy) bidx = colb + j;
          }
          const float nmy = fmaxf(my, cmy), nmz = fmaxf(mz, cmz);
          const float ry = my - nmy, rz = (mz - nmz) * inv_temp;          // <= 0 (-inf on the first chunk)
          const float c1 = ex2_ftz(ry * L2E), cT = ex2_ftz(ry * kT), cZ = ex2_ftz(rz * L2E);
          // sA' = cZ (sA + sZ (rz - ry / Temp));  guard the first chunk (sZ = 0, rz = -inf)
          sA = (sZ > 0.f) ? cZ * (sA + sZ * (rz - ry * inv_temp)) : 0.f;
          s1 *= c1; sT *= cT; sZ *= cZ;
          my = nmy; mz = nmz;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float yd = v[j] - my, zd = (z[j] - mz) * inv_temp;
            const float eT = ex2_ftz(yd * kT), e1 = ex2_ftz(yd * L2E), ez = ex2_ftz(zd * L2E);
            s1 += e1; sT += eT; sZ += ez;
            sA += (ez > 0.f) ? ez * (zd - yd * inv_temp) : 0.f;       // masked columns: e^{-inf} * (-inf + inf) must not produce NaN
          }
          if (tcol >= colb && tcol < colb + 32) {
#pragma unroll
            for (int j = 0; j < 32; ++j) if (colb + j == tcol) ytgt = v[j];
          }
        }
      }
      if (row_ok) {
        const int part = (n0 + half * C_PER * CH) / (C_PER * CH);
        if (part < nparts) {
          float4* o = reinterpret_cast<float4*>(parts + ((long)grow * nparts + part) * EVAL_PART_FLOATS);
          o[0] = make_float4(my, s1, sT, mz);
          o[1] = make_float4(sZ, sA, ytgt, __int_as_float(bidx));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[as]);
      continue;
    }
    if constexpr (EPI == 2) {
      // ---- argmax epilogue (ArgmaxEpi): this thread owns one row and C_PER * CH columns of it: running (max, lowest index)
      float* pmax = le.c_out; int* pidx = reinterpret_cast<int*>(le.gates_out);
      const int nparts = le.H, grow = m0 + q * 32 + lane;
      float best = -INFINITY; int bidx = 0x7fffffff;
#pragma unroll 1
      for (int ci = half * C_PER; ci < (half + 1) * C_PER && ci < NCHUNK; ++ci) {
#pragma unroll 1
        for (int h = 0; h < CH / 32; ++h) {
          const int colb = n0 + ci * CH + h * 32;
          if (colb >= N) break;                             // warp-uniform
          float v[32];
          tmem_ld32(tacc + (uint32_t)(ci * CH + h * 32), v);
          if (colb + 32 <= N && bias != nullptr && (((uintptr_t)bias) & 15) == 0) {
            const float4* b4 = reinterpret_cast<const float4*>(bias + colb);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 bb = __ldg(b4 + j);
              v[4 * j] = fmaf(alpha, v[4 * j], bb.x); v[4 * j + 1] = fmaf(alpha, v[4 * j + 1], bb.y);
              v[4 * j + 2] = fmaf(alpha, v[4 * j + 2], bb.z); v[4 * j + 3] = fmaf(alpha, v[4 * j + 3], bb.w);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = fmaf(alpha, v[j], (bias != nullptr && colb + j < N) ? bias[colb + j] : 0.f);
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) if (colb + j < N && v[j] > best) { best = v[j]; bidx = colb + j; }     // ascending: ties keep the lowest index
        }
      }
      if (grow < M) {
        const int part = (n0 + half * C_PER * CH) / (C_PER * CH);
        if (part < nparts) { pmax[(long)grow * nparts + part] = best; pidx[(long)grow * nparts + part] = bidx; }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[as]);
      continue;
    }
    if constexpr (EPI == 0 || EPI == 4) {
    // (EPI == 4: every tile of this launch satisfies the fast path's conditions -- the host checked -- so the generic path is not even compiled in)
    // ---- fast path: a full interior tile, written once (beta = 0) or K-split partial sums reduced into fp32 C; 16-byte aligned C.  Straight-line
    // code without per-element predicates: the generic path below spends most of its issue slots (and instruction-cache
    // misses: ncu stall_no_inst + branch_resolving = 24 % of the samples of the vocab-head GEMM) on range / mode checks.
    if (EPI == 4 || ((split ? sizeof(TC) == 4 : beta == 0.f) && vec_ok && m0 + TC_BM <= M && n0 + BN <= N && (((uintptr_t)bias) & 15) == 0)) {
#pragma unroll 1
      for (int ci = half * C_PER; ci < (half + 1) * C_PER && ci < NCHUNK; ++ci) {
        const int c0 = ci * CH;
#pragma unroll
        for (int h = 0; h < CH / 32; ++h) {
          float v[32];
          tmem_ld32(tacc + (uint32_t)(c0 + h * 32), v);
          if (add_bias) {
            const float4* b4 = reinterpret_cast<const float4*>(bias + n0 + c0 + h * 32);     // n0, c0 multiples of 32: 16-byte aligned when bias is
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 bb = __ldg(b4 + j);
              v[4 * j] = fmaf(alpha, v[4 * j], bb.x); v[4 * j + 1] = fmaf(alpha, v[4 * j + 1], bb.y);
              v[4 * j + 2] = fmaf(alpha, v[4 * j + 2], bb.z); v[4 * j + 3] = fmaf(alpha, v[4 * j + 3], bb.w);
            }
          } else if (alpha != 1.0f) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] *= alpha;
          }
          if (relu) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
          }
          unsigned char* dst = my + lane * TC_EPI_PITCH + h * 32 * sizeof(TC);
          if (sizeof(TC) == 2) {
#pragma unroll
            for (int j = 0; j < 32; j += 8)
              *reinterpret_cast<uint4*>(dst + j * 2) = make_uint4(pack_bf16(v[j], v[j + 1]), pack_bf16(v[j + 2], v[j + 3]), pack_bf16(v[j + 4], v[j + 5]), pack_bf16(v[j + 6], v[j + 7]));
          } else {
#pragma unroll
            for (int j = 0; j < 32; j += 4)
              *reinterpret_cast<uint4*>(dst + j * 4) = make_uint4(__float_as_uint(v[j]), __float_as_uint(v[j + 1]), __float_as_uint(v[j + 2]), __float_as_uint(v[j + 3]));
          }
        }
        __syncwarp();
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int r = it * 4 + (lane >> 3), grow = m0 + q * 32 + r;
          const long orow = row_unperm_h ? (long)(grow & 3) * row_unperm_h + (grow >> 2) : (long)grow;   // interleaved -> gate-major row
          TC* cp = C + orow * ldc + n0 + c0 + (lane & 7) * PER;
          const uint4 acc = *reinterpret_cast<const uint4*>(my + r * TC_EPI_PITCH + (lane & 7) * 16);
          if (split) {                               // K-split partial sums (fp32 C): one 16-byte vector reduction
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" :: "l"(cp), "f"(__uint_as_float(acc.x)), "f"(__uint_as_float(acc.y)),
                         "f"(__uint_as_float(acc.z)), "f"(__uint_as_float(acc.w)) : "memory");
          } else {
            *reinterpret_cast<uint4*>(cp) = acc;
          }
        }
        __syncwarp();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[as]);
      continue;
    }
    if constexpr (EPI == 0) {
#pragma unroll 1
    for (int ci = half * C_PER; ci < (half + 1) * C_PER && ci < NCHUNK; ++ci) {
      const int c0 = ci * CH;
      if (n0 + c0 >= N) break;
#pragma unroll
      for (int h = 0; h < CH / 32; ++h) {
        float v[32];
        tmem_ld32(tacc + (uint32_t)(c0 + h * 32), v);
        const int colb = n0 + c0 + h * 32;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          float x = alpha * v[j];
          if (add_bias && colb + j < N) x += bias[colb + j];
          if (relu) x = fmaxf(x, 0.f);
          v[j] = x;
        }
        unsigned char* dst = my + lane * TC_EPI_PITCH + h * 32 * sizeof(TC);
        if (sizeof(TC) == 2) {
#pragma unroll
          for (int j = 0; j < 32; j += 8)
            *reinterpret_cast<uint4*>(dst + j * 2) = make_uint4(pack_bf16(v[j], v[j + 1]), pack_bf16(v[j + 2], v[j + 3]), pack_bf16(v[j + 4], v[j + 5]), pack_bf16(v[j + 6], v[j + 7]));
        } else {
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<uint4*>(dst + j * 4) = make_uint4(__float_as_uint(v[j]), __float_as_uint(v[j + 1]), __float_as_uint(v[j + 2]), __float_as_uint(v[j + 3]));
        }
      }
      __syncwarp();
#pragma unroll 1                             // edge tiles / beta != 0 only: keep the code small
      for (int it = 0; it < 8; ++it) {
        const int r = it * 4 + (lane >> 3), part = lane & 7;
        const int grow = m0 + q * 32 + r, gcol = n0 + c0 + part * PER;
        if (grow < M && gcol < N) {
          const uint4 acc = *reinterpret_cast<const uint4*>(my + r * TC_EPI_PITCH + part * 16);
          const long orow = row_unperm_h ? (long)(grow & 3) * row_unperm_h + (grow >> 2) : (long)grow;   // interleaved -> gate-major row
          TC* cp = C + orow * ldc + gcol;
          if (split) {
            if (vec_ok && gcol + 4 <= N) {         // one 16-byte vector reduction instead of four scalar atomics
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" :: "l"(cp), "f"(__uint_as_float(acc.x)), "f"(__uint_as_float(acc.y)),
                           "f"(__uint_as_float(acc.z)), "f"(__uint_as_float(acc.w)) : "memory");
            } else {
              const float* a = reinterpret_cast<const float*>(&acc);
#pragma unroll
              for (int e = 0; e < 4; ++e) if (gcol + e < N) atomicAdd(reinterpret_cast<float*>(cp) + e, a[e]);
            }
          } else if (vec_ok && gcol + PER <= N) {
            uint4 o = acc;
            if (beta != 0.f) {
              const uint4 old = *reinterpret_cast<const uint4*>(cp);
              o = (sizeof(TC) == 2) ? epi_combine_bf16(acc, old, beta) : epi_combine_f32(acc, old, beta);
            }
            *reinterpret_cast<uint4*>(cp) = o;
          } else {
            const TC* a = reinterpret_cast<const TC*>(&acc);
#pragma unroll
            for (int e = 0; e < PER; ++e) {
              if (gcol + e < N) {
                float x = to_f<TC>(a[e]);
                if (beta != 0.f) x += beta * to_f<TC>(cp[e]);
                cp[e] = from_f<TC>(x);
              }
            }
          }
        }
      }
      __syncwarp();
    }
    tc_fence_before();                         // order this warp's tcgen05.ld before releasing the accumulator stage
    __syncwarp();
    if (lane == 0) mbar_arrive(&tempty_bar[as]);
    }   // generic path (EPI == 0 only)
    }   // EPI == 0 || EPI == 4
    }   // general epilogues
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(Cfg::TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

// 2-D bf16 tensor map: inner (contiguous) extent `inner`, `outer` rows of pitch `ld` elements; box {64, box_outer}.
inline int make_tmap_bf16(CUtensorMap* map, const void* ptr, long inner, long outer, long ld, int box_outer) {
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return set_err(B2C_ECUDA, "cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {64u, (cuuint32_t)box_outer};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return set_err(B2C_ECUDA, "cuTensorMapEncodeTiled failed (%d): ptr=%p inner=%ld outer=%ld ld=%ld box=%d", (int)r, ptr, inner, outer, ld, box_outer);
  return 0;
}

struct GemmArgs {
  int M, N, K;
  float alpha, beta;
  const void* A; long lda; int a_mn;
  const void* B; long ldb; int b_mn;
  void* C; long ldc;
  const float* bias; int relu;
  int row_unperm_h = 0;              // != 0: output row m is written to row (m & 3) * H + (m >> 2) (gate-interleaved -> gate-major)
  const LstmEpi* lstm = nullptr;     // fused LSTM-cell epilogue instead of writing C
  ArgmaxEpi* amax = nullptr;         // per-row partial argmax instead of writing C (tcgen05 path only; nparts / cols_per_part are filled in)
  EvalEpi* eval = nullptr;           // per-row partials of token KD / CE / argmax instead of writing C (tcgen05 path only; nparts filled in)
  const int* steps = nullptr;        // != null: the launch is step `step` of a variable-length recurrence and does nothing when step >= *steps
  int step = 0;
};

inline bool tc_eligible(const GemmArgs& g) {
  return ((uintptr_t)g.A % 16 == 0) && ((uintptr_t)g.B % 16 == 0) && (g.lda % 8 == 0) && (g.ldb % 8 == 0);
}

// Tile / split-K plan.  Every CTA has to pull (128 + BN) x 64 bf16 per k-block through its L2 port, which is what bounds these
// GEMMs (not the tensor pipe), so the plan minimises  waves x k-blocks-per-item x (128 + BN)  over BN in {256,128,64}, with K
// splits (fp32 output, no ReLU, beta 0 or 1: partial tiles are added with red.global.add.f32) filling the SMs when M*N is small.
struct TcPlan { int bn, splits, kb_per_split; };
inline TcPlan plan_tc(const GemmArgs& g, int elem_c, int sms) {
  const int num_kb = cdiv(g.K, TC_BK);
  const bool can_split = (elem_c == 4) && !g.relu && (g.beta == 0.f || g.beta == 1.f) && (g.lstm == nullptr) && (g.amax == nullptr) && (g.eval == nullptr);
  TcPlan best{64, 1, num_kb}; double best_cost = 1e30;
  const int cand[3] = {256, 128, 64};
  for (int ci = 0; ci < 3; ++ci) {
    const int bn = cand[ci];
    if (bn > 64 && g.N <= bn / 2) continue;                   // mostly-empty tiles
    const long tiles = (long)cdiv(g.M, TC_BM) * cdiv(g.N, bn);
    int splits = 1;
    if (can_split && tiles < 2L * sms && num_kb >= 16) {
      splits = (int)((2L * sms) / tiles); if (splits > num_kb / 8) splits = num_kb / 8; if (splits < 1) splits = 1;
    }
    const int kbs = cdiv(num_kb, splits); splits = cdiv(num_kb, kbs);
    const long items = tiles * splits;
    const long waves = (items + sms - 1) / sms;
    // per item: k-block feed + fixed cost (pipeline fill, epilogue of a 128 x bn tile); split items pay the atomics
    const double cost = (double)waves * ((double)kbs * (128 + bn) + 6.0 * (128 + bn) + (splits > 1 ? 2.0 : 1.0) * bn * 4.0);
    if (cost < best_cost) { best_cost = cost; best = TcPlan{bn, splits, kbs}; }
  }
  return best;
}

inline bool fast_only_enabled() { static int on = -1; if (on < 0) { const char* e = getenv("B2C_GEMM_FAST_ONLY"); on = (e && e[0] == '0') ? 0 : 1; } return on != 0; }
inline int sm_count() {
  static int n = 0;
  if (n == 0) { int dev = 0; cudaGetDevice(&dev); if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148; }
  return n;
}

// Background contractions.  The tcgen05 GEMM is persistent: a CTA keeps its SM (160-220 KB of shared memory) until the kernel ends, so
// a full-grid GEMM on a side stream starves a latency-bound chain on another stream even when that chain has the higher priority
// (measured: the first four steps of the reverse recurrence took 83 / 65 / 63 / 50 us instead of 37 under the output head's weight
// gradients).  The chain's own GEMMs never use more than 128 CTAs, so work issued as "background" is confined to `cap` CTAs (20 =
// 148 - 128).  Thread-local and scoped: the issuing code sets it around its side-stream launches.
inline int& gemm_cta_cap() { static thread_local int c = 0; return c; }
struct GemmCapScope {
  int saved;
  explicit GemmCapScope(int cap) : saved(gemm_cta_cap()) { gemm_cta_cap() = cap; }
  ~GemmCapScope() { gemm_cta_cap() = saved; }
};
inline int gemm_sms() { const int n = sm_count(), c = gemm_cta_cap(); return (c > 0 && c < n) ? c : n; }

template <int BN, bool A_MN, bool B_MN, typename TC>
int launch_tc(const GemmArgs& g, const TcPlan& plan, cudaStream_t st) {
  CUtensorMap ta, tb;
  if (!A_MN) B2C_TRY(make_tmap_bf16(&ta, g.A, g.K, g.M, g.lda, TC_BM)); else B2C_TRY(make_tmap_bf16(&ta, g.A, g.M, g.K, g.lda, 64));
  if (!B_MN) B2C_TRY(make_tmap_bf16(&tb, g.B, g.K, g.N, g.ldb, BN)); else B2C_TRY(make_tmap_bf16(&tb, g.B, g.N, g.K, g.ldb, 64));
  constexpr bool CAN_LSTM = !A_MN && !B_MN && sizeof(TC) == 4;       // the special epilogues exist for K-major operands and fp32 "outputs" only
  void (*kern)(const CUtensorMap, const CUtensorMap, int, int, int, float, float, TC*, long, const float*, int, int, int, int, int, int, const LstmEpi) =
      gemm_tc_kernel<BN, A_MN, B_MN, TC, 0>;
  int flavour = g.lstm ? ((g.lstm->drop_p > 0.f && g.lstm->h_next) ? 1 : 5) : (g.amax ? 2 : (g.eval ? 3 : 0));
  if (g.eval && g.eval->teacher_dtype != B2C_F32) flavour = g.eval->teacher_dtype == B2C_BF16 ? 6 : 7;
  if (flavour == 0 && fast_only_enabled() && g.M % TC_BM == 0 && g.N % BN == 0 && (plan.splits > 1 ? sizeof(TC) == 4 : g.beta == 0.f) &&
      ((uintptr_t)g.C) % 16 == 0 && (g.ldc * (long)sizeof(TC)) % 16 == 0 && (((uintptr_t)g.bias) & 15) == 0) {
    flavour = 4;                       // every tile takes the straight-line epilogue: the kernel without the generic path
    kern = gemm_tc_kernel<BN, A_MN, B_MN, TC, 4>;
  }
  if (flavour != 0 && flavour != 4) {
    if constexpr (CAN_LSTM) {
      kern = flavour == 1 ? gemm_tc_kernel<BN, A_MN, B_MN, TC, 1> : (flavour == 5 ? gemm_tc_kernel<BN, A_MN, B_MN, TC, 5> :
             (flavour == 2 ? gemm_tc_kernel<BN, A_MN, B_MN, TC, 2> : (flavour == 6 ? gemm_tc_kernel<BN, A_MN, B_MN, TC, 6> :
             (flavour == 7 ? gemm_tc_kernel<BN, A_MN, B_MN, TC, 7> : gemm_tc_kernel<BN, A_MN, B_MN, TC, 3>))));
    } else return set_err(B2C_EINVAL, "the fused LSTM / argmax / validation epilogues need K-major operands and the fp32 instantiation");
  }
  static bool attr_set[8] = {false, false, false, false, false, false, false, false};      // per template instantiation and epilogue flavour
  if (!attr_set[flavour]) {
    B2C_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TcCfg<BN>::SMEM_BYTES));
    attr_set[flavour] = true;
  }
  const int kb_per_split = plan.kb_per_split, splits = plan.splits;
  if (splits > 1 && g.beta == 0.f)
    B2C_CUDA(cudaMemset2DAsync(g.C, (size_t)g.ldc * sizeof(TC), 0, (size_t)g.N * sizeof(TC), (size_t)g.M, st));
  const int tiles_m = cdiv(g.M, TC_BM), tiles_n = cdiv(g.N, BN);
  const long total = (long)tiles_m * tiles_n * splits;
  const int grid = (int)(total < gemm_sms() ? total : gemm_sms());
  LstmEpi epi = g.lstm ? *g.lstm : LstmEpi{};
  if (g.amax) {
    B2C_CHECK_ARG(!g.lstm && splits == 1 && g.amax->pmax && g.amax->pidx, "argmax epilogue: no K split, no LSTM epilogue, partial buffers required");
    constexpr int CHc = 128 / (int)sizeof(TC), CPER = (BN / CHc + 1) / 2;
    g.amax->cols_per_part = CPER * CHc;
    g.amax->nparts = cdiv(g.N, g.amax->cols_per_part);
    epi = pack_argmax(*g.amax);
  }
  if (g.eval) {
    B2C_CHECK_ARG(!g.lstm && !g.amax && splits == 1 && g.eval->teacher && g.eval->targets && g.eval->parts, "validation epilogue: no K split, no other epilogue, buffers required");
    constexpr int CHc = 128 / (int)sizeof(TC), CPER = (BN / CHc + 1) / 2;
    g.eval->cols_per_part = CPER * CHc;
    g.eval->nparts = cdiv(g.N, g.eval->cols_per_part);          // the caller sized `parts` for the smallest part (32 columns)
    epi = pack_eval(*g.eval);
  }
  epi.steps = g.steps; epi.step = g.step;
  B2C_CUDA(launch_pdl(kern, dim3(grid), dim3(TC_THREADS), TcCfg<BN>::SMEM_BYTES, st, ta, tb, g.M, g.N, g.K, g.alpha, g.beta, (TC*)g.C, g.ldc,
                      g.bias, g.relu, kb_per_split, tiles_m, tiles_n, splits, g.row_unperm_h, epi));
  B2C_LAUNCH_CHECK("gemm_tc_kernel");
  return 0;
}

template <int BN, typename TC>
int launch_tc_major(const GemmArgs& g, const TcPlan& plan, cudaStream_t st) {
  if (!g.a_mn && !g.b_mn) return launch_tc<BN, false, false, TC>(g, plan, st);
  if (!g.a_mn && g.b_mn) return launch_tc<BN, false, true, TC>(g, plan, st);
  if (g.a_mn && g.b_mn) return launch_tc<BN, true, true, TC>(g, plan, st);
  return launch_tc<BN, true, false, TC>(g, plan, st);
}

// bf16 operands on tensor cores; TC = bf16 or float output.
template <typename TC>
int gemm_bf16_tc(const GemmArgs& g, cudaStream_t st) {
  const TcPlan plan = plan_tc(g, (int)sizeof(TC), gemm_sms());
  if (plan.bn == 256) return launch_tc_major<256, TC>(g, plan, st);
  if (plan.bn == 128) return launch_tc_major<128, TC>(g, plan, st);
  return launch_tc_major<64, TC>(g, plan, st);
}

template <typename TA, typename TB, typename TC>
int gemm_simt(const GemmArgs& g, cudaStream_t st) {
  dim3 grid(cdiv(g.N, SG_BN), cdiv(g.M, SG_BM));
  LstmEpi le = g.lstm ? *g.lstm : LstmEpi{};
  le.steps = g.steps; le.step = g.step;
  B2C_CUDA(launch_pdl(gemm_simt_kernel<TA, TB, TC>, grid, dim3(256), 0, st, g.M, g.N, g.K, g.alpha, (const TA*)g.A, g.lda, g.a_mn,
                      (const TB*)g.B, g.ldb, g.b_mn, g.beta, (TC*)g.C, g.ldc, g.bias, g.relu, g.row_unperm_h, le));
  B2C_LAUNCH_CHECK("gemm_simt_kernel");
  return 0;
}

// Precision-mode dispatch used by the decoder: T = operand type, TC = output type.
template <typename T, typename TC> struct Gemm;
template <typename TC> struct Gemm<float, TC> {
  static int run(const GemmArgs& g, cudaStream_t st) { return gemm_simt<float, float, TC>(g, st); }
};
template <typename TC> struct Gemm<bf16, TC> {
  static int run(const GemmArgs& g, cudaStream_t st) {
    if (tc_eligible(g)) return gemm_bf16_tc<TC>(g, st);
    return gemm_simt<bf16, bf16, TC>(g, st);     // row pitch TMA cannot describe (e.g. odd vocab): CUDA-core tiles
  }
};

}  // namespace b2c
