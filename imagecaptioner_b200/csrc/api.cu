// b2c C ABI: host-side orchestration of the decoder / loss kernels.  See include/b2c.h for the contract and
// oracle/manual_backward.py for the (CPU, test-only) blueprint of exactly this dataflow.
#include <stdlib.h>
#include "gemm.cuh"
#include "loss_kernels.cuh"
#include "decoder_kernels.cuh"
#include "recurrent.cuh"
#include "recur_cluster.cuh"
#include "refine_kernels.cuh"
#include "mha_mma.cuh"
#include "optim_kernels.cuh"

using namespace b2c;

namespace {

constexpr int MAXL = B2C_MAX_LAYERS;
constexpr int COLSUM_RS = 160;

// ------------------------------------------------------------------ device check (sm_100 only, no fallback)
int check_device() {
  static int cached = 1;   // 1 = not checked, 0 = ok, <0 error
  if (cached <= 0) return cached;
  int dev = 0;
  B2C_CUDA(cudaGetDevice(&dev));
  int major = 0;
  B2C_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) { cached = B2C_EARCH; return set_err(B2C_EARCH, "b2c kernels are built for sm_100a only; device has compute capability major %d", major); }
  cached = 0;
  return 0;
}

struct Carver {
  unsigned char* base; size_t off;
  template <typename U> U* take(size_t n) {
    off = align_up(off, 256);
    U* p = base ? reinterpret_cast<U*>(base + off) : reinterpret_cast<U*>((uintptr_t)0);
    off += n * sizeof(U);
    return p;
  }
};

inline int in_dim(const B2CShape& s, int k) { return k == 0 ? s.E : s.H; }

int check_shape(const B2CShape* s) {
  B2C_CHECK_ARG(s != nullptr, "shape is NULL");
  B2C_CHECK_ARG(s->B > 0 && s->T > 0 && s->S > 0 && s->V > 1, "bad shape B=%d T=%d S=%d V=%d", s->B, s->T, s->S, s->V);
  B2C_CHECK_ARG(s->L >= 1 && s->L <= MAXL, "L=%d outside [1,%d]", s->L, MAXL);
  B2C_CHECK_ARG(s->E > 0 && s->E % 8 == 0 && s->H > 0 && s->H % 8 == 0, "E=%d and H=%d must be positive multiples of 8", s->E, s->H);
  B2C_CHECK_ARG((long)s->B * 4 * s->H < 2147483647L && (long)s->B * s->S * s->E < 2147483647L, "B*4H and B*S*E must stay below 2^31 (32-bit index arithmetic in the per-step kernels)");
  return 0;
}

// ------------------------------------------------------------------ packed operand weights (compute type)
// Gate rows are INTERLEAVED in every 4H-sized object (row 4j+g = gate g of hidden unit j) so that the gate contraction's
// epilogue holds the four pre-activations of one unit together (fused cell, gemm.cuh).  attention_combine is folded into
// layer 0 (oracle/manual_backward.py v2):  Wcat[0] = [W_ih0 W_cc | W_hh0],  We = W_ih0 W_ce,  bx = W_ih0 b_c + b_ih0 + b_hh0.
template <typename T> struct Weights {
  T *Wf, *Wh, *Wce, *Wcc, *W1, *W2, *Wih0, *We; T* Wcat[MAXL]; float* bcat[MAXL]; float* bx;
  T* Wuh;      // [W_h ; W_hh of the top layer (interleaved rows)], (E + 4H) x H: both act on the top layer's h_{t-1}, one contraction
  void carve(Carver& c, const B2CShape& s) {
    Wf = c.take<T>((size_t)s.E * s.E); Wh = c.take<T>((size_t)s.E * s.H);
    Wce = c.take<T>((size_t)s.E * s.E); Wcc = c.take<T>((size_t)s.E * s.E);
    W1 = c.take<T>((size_t)s.E * s.H); W2 = c.take<T>((size_t)s.V * s.E);
    Wih0 = c.take<T>((size_t)4 * s.H * s.E); We = c.take<T>((size_t)4 * s.H * s.E); bx = c.take<float>((size_t)4 * s.H);
    for (int k = 0; k < s.L; ++k) { Wcat[k] = c.take<T>((size_t)4 * s.H * (in_dim(s, k) + s.H)); bcat[k] = c.take<float>((size_t)4 * s.H); }
    Wuh = c.take<T>((size_t)(s.E + 4 * s.H) * s.H);
  }
};

template <typename T, typename TC>
int gemm(cudaStream_t st, int M, int N, int K, const T* A, long lda, int a_mn, const T* B, long ldb, int b_mn,
         TC* C, long ldc, float beta = 0.f, const float* bias = nullptr, int relu = 0, float alpha = 1.f, int row_unperm_h = 0);

template <typename T>
int pack_params(const B2CShape& s, const B2CParams& p, const Weights<T>& w, cudaStream_t st) {
  B2C_CHECK_ARG(p.embedding && p.attn_w && p.attn_b && p.comb_w && p.comb_b && p.out0_w && p.out0_b && p.out3_w && p.out3_b, "NULL parameter pointer");
  PackTable tab; tab.n = 0;
  auto add = [&](const float* src, void* dst, int rows, int cols, long lds, long ldd, int perm_h = 0, const float* src2 = nullptr, int as_float = 0) {
    PackSeg& g = tab.seg[tab.n++]; g.src = src; g.dst = dst; g.src2 = src2; g.rows = rows; g.cols = cols; g.lds = lds; g.ldd = ldd; g.as_float = as_float; g.perm_h = perm_h;
  };
  const int E = s.E, H = s.H;
  add(p.attn_w, w.Wh, E, H, H + E, H);
  add(p.attn_w + H, w.Wf, E, E, H + E, E);
  add(p.comb_w, w.Wce, E, E, 2 * E, E);
  add(p.comb_w + E, w.Wcc, E, E, 2 * E, E);
  add(p.out0_w, w.W1, E, H, H, H);
  add(p.out3_w, w.W2, s.V, E, E, E);
  for (int k = 0; k < s.L; ++k) {
    B2C_CHECK_ARG(p.w_ih[k] && p.w_hh[k] && p.b_ih[k] && p.b_hh[k], "NULL LSTM parameter pointer (layer %d)", k);
    const int in = in_dim(s, k);
    if (k == 0) add(p.w_ih[0], w.Wih0, 4 * H, E, E, E, H);                      // its product with W_cc fills Wcat[0][:, :E] below
    else add(p.w_ih[k], w.Wcat[k], 4 * H, in, in, in + H, H);
    add(p.w_hh[k], w.Wcat[k] + in, 4 * H, H, H, in + H, H);
    if (k > 0) add(p.b_ih[k], w.bcat[k], 4 * H, 1, 1, 1, H, p.b_hh[k], 1);
  }
  add(p.attn_w, w.Wuh, E, H, H + E, H);
  add(p.w_hh[s.L - 1], w.Wuh + (size_t)E * H, 4 * H, H, H, H, H);
  pack_params_kernel<T><<<dim3(96, tab.n), 256, 0, st>>>(tab);
  B2C_LAUNCH_CHECK("pack_params_kernel");
  // W_x = W_ih0 W_cc -> Wcat[0][:, :E];  W_e = W_ih0 W_ce;  b_x
  B2C_TRY((gemm<T, T>(st, 4 * H, E, E, w.Wih0, E, 0, w.Wcc, E, 1, w.Wcat[0], E + H)));
  B2C_TRY((gemm<T, T>(st, 4 * H, E, E, w.Wih0, E, 0, w.Wce, E, 1, w.We, E)));
  bias_fold_kernel<<<cdiv(4 * H * 32, 256), 256, 0, st>>>(p.w_ih[0], p.comb_b, p.b_ih[0], p.b_hh[0], H, E, w.bx);
  B2C_LAUNCH_CHECK("bias_fold_kernel");
  return 0;
}

// ------------------------------------------------------------------ cluster recurrence (recur_cluster.cuh): shapes and plan
constexpr int CR_MAX_CLUSTERS = 16;
inline bool cluster_shape_ok(const B2CShape& s) { return s.H == CR_H && s.E == CR_E && s.L == CR_L && s.S <= CR_SMAX && s.S >= 1; }
inline bool cluster_enabled() {
  static int on = -1;
  // opt-in (B2C_CLUSTER=1): correct, but measured SLOWER than the per-step kernels on B200 (42 vs 31 us per step at B = 512): every
  // cluster re-streams all 7.6 MB of recurrent weights per step and one SM cannot pull more than ~35 B/clk through TMA
  // (tools/probe_ingest.cu, profiles/r2_cluster_recurrence.md)
  if (on < 0) { const char* e = getenv("B2C_CLUSTER"); on = (e && e[0] == '1') ? 1 : 0; }
  return on != 0;
}
// clusters of 8 CTAs the device keeps resident at once (B200: 15); 0 if the query fails
inline int cluster_max_active() {
  static int n = -1;
  if (n >= 0) return n;
  n = 0;
  if (cudaFuncSetAttribute(recur_cluster_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CR_SMEM_BYTES) != cudaSuccess) { cudaGetLastError(); return n; }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(CR_CL * CR_MAX_CLUSTERS); cfg.blockDim = dim3(CR_THREADS); cfg.dynamicSmemBytes = CR_SMEM_BYTES;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = CR_CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  int m = 0;
  if (cudaOccupancyMaxActiveClusters(&m, recur_cluster_fwd_kernel, &cfg) != cudaSuccess) { cudaGetLastError(); return n; }
  if (const char* e = getenv("B2C_CLUSTER_MAX")) { const int lim = atoi(e); if (lim > 0 && lim < m) m = lim; }
  n = m > CR_MAX_CLUSTERS ? CR_MAX_CLUSTERS : m;
  return n;
}
// number of row slices (clusters) for batch B: every slice <= 40 rows and all clusters co-resident; 0 = shape not covered
inline int cluster_plan(const B2CShape& s) {
  if (!cluster_enabled() || !cluster_shape_ok(s)) return 0;
  const int mx = cluster_max_active();
  if (mx <= 0) return 0;
  int ncl = cdiv(s.B, 32); if (ncl > mx) ncl = mx;
  if (cdiv(s.B, ncl) > CR_RMAX) return 0;
  return ncl;
}

// ------------------------------------------------------------------ workspaces
template <typename T> struct TrainWs {
  Weights<T> w;
  float *P, *u; T *emb, *G0, *o1; T* xh[MAXL]; T* gates[MAXL]; float* c[MAXL];
  T* dgates[MAXL]; float* dxh0; float* dxh[MAXL]; float* dc[MAXL]; T* do1; float* dHext; float* ds; T* du; T* dq; T* dP; float* demb; float* partial;
  float *dWx32, *dWe32; T *dWxT, *dWeT; float* partial_side;
  unsigned int* sync;                 // grid-barrier arrival counters of the persistent recurrence kernels (recurrent.cuh)
  float* EP;                          // e^{2P} (B, S, E) fp32: the attention phase of the persistent forward kernel streams it instead of P
  float* evalp;                       // (T*B, ceil(V/32), 8) partials of the validation epilogue of the vocabulary-head GEMM
  T* G0T;                             // (T, ncl, 4H, 40): G0 re-laid out per row slice for the cluster recurrence kernel (recur_cluster.cuh)
  float* UR;                          // (B, E + 4H) fp32, one step: [u_t | W_hh h_{t-1} of the top layer] from the merged contraction
  size_t bytes;
  void carve(void* base, const B2CShape& s) {
    Carver c{reinterpret_cast<unsigned char*>(base), 0};
    const size_t B = s.B, Tn = s.T, S = s.S, E = s.E, H = s.H, TB = Tn * B;
    w.carve(c, s);
    P = c.take<float>(B * S * E); emb = c.take<T>(TB * E); u = c.take<float>(TB * E); G0 = c.take<T>(TB * 4 * H); o1 = c.take<T>(TB * E);
    for (int k = 0; k < s.L; ++k) {
      xh[k] = c.take<T>((Tn + 1) * B * (in_dim(s, k) + H));        // layer 0: [ctx_t ; h0_{t-1}]
      gates[k] = c.take<T>(TB * 4 * H);
      this->c[k] = c.take<float>((Tn + 1) * B * H);
    }
    for (int k = 0; k < s.L; ++k) {
      dgates[k] = c.take<T>(TB * 4 * H);
      dxh[k] = k == 0 ? nullptr : c.take<float>(TB * 2 * H);       // fp32, one slot per step (split-K GEMMs add into zeroed slots)
      dc[k] = c.take<float>(B * H);
    }
    dxh0 = c.take<float>(TB * (E + H));                             // [dctx_t ; dh0 carry], fp32
    do1 = c.take<T>(TB * E); dHext = c.take<float>(TB * H); ds = c.take<float>(TB * S);
    du = c.take<T>(TB * E); dq = c.take<T>(B * H); dP = c.take<T>(B * S * E); demb = c.take<float>(TB * E);
    dWx32 = c.take<float>(4 * H * E); dWe32 = c.take<float>(4 * H * E); dWxT = c.take<T>(4 * H * E); dWeT = c.take<T>(4 * H * E);
    size_t mc = (size_t)s.V; if ((size_t)4 * H > mc) mc = 4 * H; if (E > mc) mc = E;
    partial = c.take<float>((size_t)COLSUM_RS * mc); partial_side = c.take<float>((size_t)COLSUM_RS * mc);
    sync = c.take<unsigned int>(128 + 160 * 32);         // four arrival-counter lines + one 128-byte flag line per CTA
    EP = c.take<float>(B * S * E);
    evalp = c.take<float>(TB * (size_t)cdiv(s.V, 32) * EVAL_PART_FLOATS);
    G0T = c.take<T>(cluster_shape_ok(s) ? Tn * (size_t)CR_MAX_CLUSTERS * 4 * H * CR_RMAX : 0);
    UR = c.take<float>(B * (E + 4 * H));
    bytes = align_up(c.off, 256);
  }
};

template <typename T> struct DecodeWs {
  Weights<T> w;
  float *P, *u; T *emb, *G0, *o1; T* xh[MAXL]; float* c[MAXL]; float* logits; int64_t* cur; int32_t* done; float* amax_v; int* amax_i;
  size_t bytes;
  void carve(void* base, const B2CShape& s) {
    Carver c{reinterpret_cast<unsigned char*>(base), 0};
    const size_t B = s.B, S = s.S, E = s.E, H = s.H;
    w.carve(c, s);
    P = c.take<float>(B * S * E); emb = c.take<T>(B * E); u = c.take<float>(B * E); G0 = c.take<T>(B * 4 * H); o1 = c.take<T>(B * E);
    for (int k = 0; k < s.L; ++k) { xh[k] = c.take<T>(2 * B * (in_dim(s, k) + H)); this->c[k] = c.take<float>(B * H); }   // two [input;h] slots (ping-pong)
    logits = c.take<float>(B * (size_t)s.V); cur = c.take<int64_t>(B); done = c.take<int32_t>(B);
    amax_v = c.take<float>(B * (size_t)cdiv(s.V, 32)); amax_i = c.take<int>(B * (size_t)cdiv(s.V, 32));      // argmax partials (<= one per 32 columns)
    bytes = align_up(c.off, 256);
  }
};


// ------------------------------------------------------------------ launch helpers
// Variable-length recurrences: the contractions issued inside a StepScope belong to step `t` of a recurrence with the device step
// count `steps` and do nothing when t >= *steps (GemmArgs::steps).  Thread-local and scoped, like GemmCapScope.
struct StepGate { const int* steps; int t; };
inline StepGate& step_gate() { static thread_local StepGate g{nullptr, 0}; return g; }
struct StepScope {
  StepGate saved;
  StepScope(const int* steps, int t) : saved(step_gate()) { step_gate() = StepGate{steps, t}; }
  ~StepScope() { step_gate() = saved; }
};

template <typename T, typename TC>
int gemm(cudaStream_t st, int M, int N, int K, const T* A, long lda, int a_mn, const T* B, long ldb, int b_mn,
         TC* C, long ldc, float beta, const float* bias, int relu, float alpha, int row_unperm_h) {
  GemmArgs g{M, N, K, alpha, beta, A, lda, a_mn, B, ldb, b_mn, C, ldc, bias, relu};
  g.row_unperm_h = row_unperm_h;
  g.steps = step_gate().steps; g.step = step_gate().t;
  return Gemm<T, TC>::run(g, st);
}
// gate contraction with the LSTM cell fused into the epilogue (no C is written)
template <typename T>
int gemm_lstm(cudaStream_t st, int M, int H, int K, const T* A, long lda, const T* Wcat, long ldb, const LstmEpi& le) {
  GemmArgs g{M, 4 * H, K, 1.f, 0.f, A, lda, 0, Wcat, ldb, 0, nullptr, 4 * H, nullptr, 0};
  g.lstm = &le;
  g.steps = step_gate().steps; g.step = step_gate().t;
  return Gemm<T, float>::run(g, st);
}

// zero the rows of steps >= *steps of up to TAIL_MAX_SEGS (Tn, B, .) buffers in one launch (decoder_kernels.cuh tail_zero_kernel);
// each buffer: base, bytes per step (a multiple of 4), steps
struct TailFill {
  TailTable tab; TailFill() { tab.n = 0; }
  void add(void* base, size_t step_bytes, int n_steps) { tab.seg[tab.n++] = TailSeg{base, (long)(step_bytes / 4), n_steps}; }
  int launch(const int* steps, cudaStream_t st) {
    if (tab.n == 0) return 0;
    tail_zero_kernel<<<dim3(2 * 148, tab.n), 256, 0, st>>>(tab, steps);
    B2C_LAUNCH_CHECK("tail_zero_kernel");
    return 0;
  }
};

inline int ew_grid(long n) { long g = (n + 255) / 256; if (g > 148 * 8) g = 148 * 8; if (g < 1) g = 1; return (int)g; }

template <typename T>
int colsum(cudaStream_t st, const T* A, long rows, int cols, long ld, float* partial, float* out, float* out2 = nullptr, int unperm_h = 0) {
  if (ld == cols && cols % 8 == 0 && ((uintptr_t)A & 15) == 0 && rows >= 256) {
    // contiguous, 16-byte rows: the vectorised kernel (a warp covers 256 columns of a row with one 512-byte access, four rows in flight)
    const int gx = cdiv(cols, 256);
    int rs = (int)((rows + 31) / 32); if (rs > 592 / gx) rs = 592 / gx; if (rs > COLSUM_RS) rs = COLSUM_RS; if (rs < 1) rs = 1;
    colsum_vec_kernel<T, false><<<dim3(gx, rs), 256, 0, st>>>(const_cast<T*>(A), (const T*)nullptr, rows, cols, 1.f, partial);
    B2C_LAUNCH_CHECK("colsum_vec_kernel");
    colsum_final_kernel<<<cdiv(cols, 256), 256, 0, st>>>(partial, rs, cols, out, out2, unperm_h);
    B2C_LAUNCH_CHECK("colsum_final_kernel");
    return 0;
  }
  if (ld != cols && ld % 8 == 0 && cols <= ld && ((uintptr_t)A & 15) == 0 && rows >= 256) {
    // pitched 16-byte rows (the padded logits gradient): the same vectorised read, padding columns summed but not written
    const int gx = cdiv(cols, 256);
    int rs = (int)((rows + 31) / 32); if (rs > 592 / gx) rs = 592 / gx; if (rs > COLSUM_RS) rs = COLSUM_RS; if (rs < 1) rs = 1;
    colsum_vec_pitched_kernel<T><<<dim3(gx, rs), 256, 0, st>>>(A, rows, cols, ld, partial);
    B2C_LAUNCH_CHECK("colsum_vec_pitched_kernel");
    colsum_final_kernel<<<cdiv(cols, 256), 256, 0, st>>>(partial, rs, cols, out, out2, unperm_h);
    B2C_LAUNCH_CHECK("colsum_final_kernel");
    return 0;
  }
  int rs = (int)((rows + 255) / 256); if (rs > COLSUM_RS) rs = COLSUM_RS; if (rs < 1) rs = 1;
  colsum_partial_kernel<T><<<dim3(cdiv(cols, 32), rs), 256, 0, st>>>(A, rows, cols, ld, partial);
  B2C_LAUNCH_CHECK("colsum_partial_kernel");
  colsum_final_kernel<<<cdiv(cols, 256), 256, 0, st>>>(partial, rs, cols, out, out2, unperm_h);
  B2C_LAUNCH_CHECK("colsum_final_kernel");
  return 0;
}

template <typename K> int set_smem(K kern, size_t bytes) {
  B2C_CHECK_ARG(bytes <= 227 * 1024, "kernel needs %zu bytes of shared memory (> 227 KB): shape too large for this path", bytes);
  if (bytes > 48 * 1024) B2C_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return 0;
}

// Preconditions (see decoder_kernels.cuh): P and F are complete before the kernel that precedes this one in the stream
// started -- callers issue pdl_full_dependency_next() once between the producers of P / F and that kernel.
template <typename T>
int attn_fwd(cudaStream_t st, const B2CShape& s, const float* P, const T* F, const float* u, T* ctx, long ldctx, float* attw,
             long ldu = 0, float* u_save = nullptr, const int* steps = nullptr, int t = 0) {
  if (ldu == 0) ldu = s.E;
  const size_t smem = (size_t)s.S * s.E * sizeof(T) + (size_t)(s.E + s.S) * 4;
  const int nq = s.S <= ATT_MAXTOK * (ATT_THREADS / 32) ? cdiv(s.E / 4, 32) : 4;       // more tokens than the register rows hold: generic kernel
  // E <= 256: 4 of the <= 7 token rows per warp are fetched in the prologue, the kernel fits 64 registers and all B = 512 CTAs
  // are resident in one wave (measured on B200: 3.23 ms / step vs 3.28 with all 7 rows up front at 80 registers, 3 CTAs / SM)
#define B2C_ATT_(NQ, KA) do { B2C_TRY(set_smem(attn_step_fwd_kernel<T, NQ, KA>, smem)); \
    B2C_CUDA(launch_pdl(attn_step_fwd_kernel<T, NQ, KA>, dim3(s.B), dim3(ATT_THREADS), smem, st, P, F, u, ldu, s.S, s.E, ctx, ldctx, attw, u_save, steps, t)); } while (0)
  if (nq == 1) B2C_ATT_(1, 4); else if (nq == 2) B2C_ATT_(2, 4); else if (nq == 3) B2C_ATT_(3, ATT_MAXTOK); else B2C_ATT_(0, ATT_MAXTOK);
#undef B2C_ATT_
  B2C_LAUNCH_CHECK("attn_step_fwd_kernel");
  return 0;
}

template <typename T>
int attn_bwd(cudaStream_t st, int B, int S, int E, const float* P, const T* F, const float* u, const float* attw, const float* dctx, long lddctx,
             float* ds, T* du, const int* steps = nullptr, int t = 0) {
  const size_t smem = (size_t)S * E * sizeof(T) + (size_t)(E + 2 * S) * 4;
  constexpr int PB = 13;            // P rows per batch of the du phase (measured: 8 -> 3.25, 13 -> 3.23, 25 -> 3.32 ms / step)
#define B2C_ATTB(PB, SMALL) do { B2C_TRY(set_smem(attn_step_bwd_kernel<T, PB, SMALL>, smem)); \
    B2C_CUDA(launch_pdl(attn_step_bwd_kernel<T, PB, SMALL>, dim3(B), dim3(ATT_THREADS), smem, st, P, F, u, (long)E, attw, dctx, lddctx, S, E, ds, du, (long)E, steps, t)); } while (0)
  if (E <= 256) B2C_ATTB(PB, true); else B2C_ATTB(PB, false);
#undef B2C_ATTB
  B2C_LAUNCH_CHECK("attn_step_bwd_kernel");
  return 0;
}

// one LSTM layer step: gates = [in ; h] Wcat^T (+ bias | + time-batched addend), cell fused into the contraction's epilogue
template <typename T>
int lstm_layer_fwd(cudaStream_t st, const B2CShape& s, const Weights<T>& w, int k, const T* xh_t, const T* addend,
                   const float* c_prev, float* c_out, T* gates_out, T* h_rec, T* h_next, T* h_top,
                   const B2CDropout& dr, long row_base, const float* rec32 = nullptr, long ld_rec32 = 0) {
  const int in = in_dim(s, k), ld = in + s.H;
  LstmEpi le{};
  le.addend32 = rec32; le.ld_addend32 = ld_rec32;
  le.enabled = 1; le.H = s.H; le.addend = addend; le.bias = (k == 0) ? nullptr : w.bcat[k];     // layer 0: b_x is inside the addend
  le.c_prev = c_prev; le.c_out = c_out; le.gates_out = gates_out;
  le.h_rec = h_rec; le.ld_rec = ld; le.h_next = h_next; le.ld_next = 2 * s.H; le.h_top = h_top; le.ld_top = s.H;
  le.drop_p = dr.p; le.seed = dr.seed; le.site = (unsigned)k; le.row_base = row_base; le.seed_dev = (const unsigned long long*)dr.seed_dev;
  // rec32 != null: the recurrent half W_hh h_{t-1} is already in rec32, only the input half (K = in) is contracted here
  return gemm_lstm<T>(st, s.B, s.H, rec32 ? in : ld, xh_t, ld, w.Wcat[k], ld, le);
}

// ------------------------------------------------------------------ sub-batch streams
// The T-step recurrence is a serial chain of small kernels (a 128..512-row GEMM, a per-sample attention kernel, a pointwise
// kernel), each bound by launch / prologue / L2 latency rather than by the machine's throughput.  Samples are independent,
// so the batch is cut into NS contiguous sub-batches whose chains run on NS forked streams and overlap on the GPU; all
// buffers keep their (T, B, .) layout (a sub-batch is a row range), so the time-batched GEMMs before and after the loop
// still see whole tensors.  Fork / join use events, which CUDA graph capture records as parallel branches.
constexpr int MAX_SUB = 5;          // 4 sub-batch branches (B2C_SUB_BATCHES) + 1 side stream for work hidden under the recurrence
struct SubStreams { cudaStream_t s[MAX_SUB]; cudaEvent_t fork; cudaEvent_t join[MAX_SUB]; cudaEvent_t ev[4]; };
constexpr int MAX_DEVICES = 64;
int get_substreams(SubStreams** out) {
  // one stream / event set per device (created on first use with that device current): a process may drive several GPUs
  static SubStreams all[MAX_DEVICES]; static bool all_ready[MAX_DEVICES] = {false};
  int dev = 0;
  B2C_CUDA(cudaGetDevice(&dev));
  B2C_CHECK_ARG(dev >= 0 && dev < MAX_DEVICES, "device index %d outside [0,%d)", dev, MAX_DEVICES);
  SubStreams& ss = all[dev]; bool& ready = all_ready[dev];
  if (!ready) {
    for (int i = 0; i < MAX_SUB; ++i) {
      B2C_CUDA(cudaStreamCreateWithFlags(&ss.s[i], cudaStreamNonBlocking));
      B2C_CUDA(cudaEventCreateWithFlags(&ss.join[i], cudaEventDisableTiming));
    }
    B2C_CUDA(cudaEventCreateWithFlags(&ss.fork, cudaEventDisableTiming));
    for (int i = 0; i < 4; ++i) B2C_CUDA(cudaEventCreateWithFlags(&ss.ev[i], cudaEventDisableTiming));
    ready = true;
  }
  *out = &ss;
  return 0;
}
// Measured on B200 (round 1, tools/microbench_streams.py): the branches do overlap 4-way, but a 128-row gate GEMM takes as
// long as the 512-row one (7.8 vs 8.6 us) — the chain is bound by per-kernel latency x chain length, which a narrower
// kernel does not shorten — so the whole step got 5 % slower (4x the launches).  Off unless B2C_SUB_BATCHES=2|4 is set.
inline int pick_sub_batches(int B) {
  static int want = -1;
  if (want < 0) { const char* e = getenv("B2C_SUB_BATCHES"); want = e ? atoi(e) : 1; if (want != 2 && want != 4) want = 1; }
  if (want > 1 && B >= 32 * want && B % want == 0) return want;
  return 1;
}
struct SubPlan { int ns; cudaStream_t st[MAX_SUB]; int b0[MAX_SUB]; int bn[MAX_SUB]; SubStreams* ss; cudaStream_t main; };
int fork_subs(SubPlan& sp, int B, cudaStream_t st, bool allow_split = true) {
  sp.ns = allow_split ? pick_sub_batches(B) : 1; sp.main = st; sp.ss = nullptr;
  if (sp.ns == 1) { sp.st[0] = st; sp.b0[0] = 0; sp.bn[0] = B; return 0; }
  B2C_TRY(get_substreams(&sp.ss));
  B2C_CUDA(cudaEventRecord(sp.ss->fork, st));
  for (int i = 0; i < sp.ns; ++i) {
    sp.st[i] = sp.ss->s[i]; sp.bn[i] = B / sp.ns; sp.b0[i] = i * sp.bn[i];
    B2C_CUDA(cudaStreamWaitEvent(sp.st[i], sp.ss->fork, 0));
  }
  return 0;
}
int join_subs(SubPlan& sp) {
  if (sp.ns == 1) return 0;
  for (int i = 0; i < sp.ns; ++i) {
    B2C_CUDA(cudaEventRecord(sp.ss->join[i], sp.st[i]));
    B2C_CUDA(cudaStreamWaitEvent(sp.main, sp.ss->join[i], 0));
  }
  return 0;
}

// ------------------------------------------------------------------ persistent forward recurrence (recurrent.cuh)
// Debug aid (B2C_RECUR_TRACE=1): per CTA, per step, 8 clock64() stamps of the epilogue group, read back with b2c_debug_recur_trace.
struct RecurTrace { unsigned long long* dev; size_t n; int grid, T; };
inline RecurTrace& recur_trace_state() { static RecurTrace t{nullptr, 0, 0, 0}; return t; }
inline unsigned long long* recur_trace_buffer(size_t n) {
  static const bool on = getenv("B2C_RECUR_TRACE") != nullptr;
  if (!on) return nullptr;
  RecurTrace& t = recur_trace_state();
  if (t.n < n) { if (t.dev) cudaFree(t.dev); t.dev = nullptr; if (cudaMalloc(&t.dev, n * 8) != cudaSuccess) { t.n = 0; return nullptr; } t.n = n; }
  return t.dev;
}

template <typename T> int recur_forward(cudaStream_t, const B2CShape&, const RecurPlan&, const TrainWs<T>&, const T*, T*, float*, const B2CDropout&) {
  return set_err(B2C_EINVAL, "the persistent recurrence kernel is bf16 only");
}
template <>
int recur_forward<bf16>(cudaStream_t st, const B2CShape& s, const RecurPlan& pl, const TrainWs<bf16>& W, const bf16* feats, bf16* hid_top, float* attw,
                        const B2CDropout& dr) {
  RecurMaps maps; RecurParams p{};
  p.B = s.B; p.T = s.T; p.S = s.S; p.E = s.E; p.H = s.H; p.L = s.L;
  p.tiles_m = pl.tiles_m; p.tiles_n = pl.tiles_n; p.u_tiles_n = pl.u_tiles_n; p.n_fbuf = pl.n_fbuf; p.f_resident = pl.f_resident; p.tmem_cols = pl.tmem_cols;
  p.P = W.P; p.EP = W.EP; p.F = feats; p.u = W.u; p.attw = attw; p.G0 = W.G0; p.hid_top = hid_top;
  p.trace = recur_trace_buffer((size_t)pl.grid * s.T * 16);
  for (int k = 0; k < s.L; ++k) {
    const int in = in_dim(s, k), ld = in + s.H;
    p.xh[k] = W.xh[k]; p.ld[k] = ld; p.in[k] = in; p.bias[k] = (k == 0) ? nullptr : W.w.bcat[k]; p.c[k] = W.c[k]; p.gates[k] = W.gates[k];
    B2C_TRY(make_tmap_bf16_3d(&maps.a[k], W.xh[k], ld, s.B, s.T + 1, ld, TC_BM));
    B2C_TRY(make_tmap_bf16(&maps.w[k], W.w.Wcat[k], ld, 4 * s.H, ld, RC_BN));
  }
  for (int k = s.L; k < RC_MAXL; ++k) { maps.a[k] = maps.a[0]; maps.w[k] = maps.w[0]; }
  B2C_TRY(make_tmap_bf16(&maps.wh, W.w.Wh, s.H, s.E, s.H, RC_BNU));
  p.drop_p = dr.p; p.seed = dr.seed; p.seed_dev = (const unsigned long long*)dr.seed_dev;
  { const char* e = getenv("B2C_RECUR_EARLY"); p.early = (e && e[0] == '0') ? 0 : 1; }
  { const char* e = getenv("B2C_RECUR_EPNC"); p.ep_nc = (e && e[0] == '1') ? 1 : 0; }
  p.barrier = W.sync; p.flags = W.sync + 128;
  B2C_CHECK_ARG(pl.grid <= 160, "unexpected grid %d", pl.grid);
  B2C_CUDA(cudaMemsetAsync(W.sync, 0, (128 + 160 * 32) * sizeof(unsigned int), st));
  void (*kern)(const RecurMaps, const RecurParams) = pl.nq == 1 ? recur_fwd_kernel<1> : (pl.nq == 2 ? recur_fwd_kernel<2> : recur_fwd_kernel<3>);
  B2C_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(pl.grid); cfg.blockDim = dim3(RC_THREADS); cfg.dynamicSmemBytes = pl.smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative; attr[0].val.cooperative = 1;      // every CTA is resident: they wait on one another
  cfg.attrs = attr; cfg.numAttrs = 1;
  B2C_CUDA(cudaLaunchKernelEx(&cfg, kern, maps, p));
  B2C_LAUNCH_CHECK("recur_fwd_kernel");
  recur_trace_state().grid = pl.grid; recur_trace_state().T = s.T;
  return 0;
}

// ------------------------------------------------------------------ cluster forward recurrence (recur_cluster.cuh)
template <typename T> int cluster_forward(cudaStream_t, const B2CShape&, int, const TrainWs<T>&, const T*, T*, float*) {
  return set_err(B2C_EINVAL, "the cluster recurrence kernel is bf16 only");
}
template <>
int cluster_forward<bf16>(cudaStream_t st, const B2CShape& s, int ncl, const TrainWs<bf16>& W, const bf16* feats, bf16* hid_top, float* attw) {
  ClusterMaps maps; ClusterParams p{};
  p.B = s.B; p.T = s.T; p.S = s.S; p.ncl = ncl;
  p.P = W.P; p.EP = W.EP; p.F = feats; p.u = W.u; p.attw = attw; p.xh0 = W.xh[0]; p.xh1 = W.xh[1];
  p.G0T = W.G0T; p.bias1 = W.w.bcat[1]; p.c0 = W.c[0]; p.c1 = W.c[1]; p.gates0 = W.gates[0]; p.gates1 = W.gates[1]; p.hid_top = hid_top;
  p.trace = recur_trace_buffer((size_t)ncl * CR_CL * s.T * 8);
  const long rows = (long)(s.T + 1) * s.B;
  B2C_TRY(make_tmap_bf16(&maps.w0, W.w.Wcat[0], CR_E + CR_H, 4 * CR_H, CR_E + CR_H, 128));
  B2C_TRY(make_tmap_bf16(&maps.w1, W.w.Wcat[1], 2 * CR_H, 4 * CR_H, 2 * CR_H, 128));
  B2C_TRY(make_tmap_bf16(&maps.wh, W.w.Wh, CR_H, CR_E, CR_H, CR_UCOLS));
  B2C_TRY(make_tmap_bf16(&maps.h0, W.xh[0], CR_E + CR_H, rows, CR_E + CR_H, CR_RMAX));
  B2C_TRY(make_tmap_bf16(&maps.h1, W.xh[1], 2 * CR_H, rows, 2 * CR_H, CR_RMAX));
  B2C_TRY(make_tmap_bf16(&maps.ctx, W.xh[0], CR_E + CR_H, rows, CR_E + CR_H, CR_SPC));
  B2C_CUDA(cudaFuncSetAttribute(recur_cluster_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CR_SMEM_BYTES));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(ncl * CR_CL); cfg.blockDim = dim3(CR_THREADS); cfg.dynamicSmemBytes = CR_SMEM_BYTES; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension; attr[0].val.clusterDim.x = CR_CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  B2C_CUDA(cudaLaunchKernelEx(&cfg, recur_cluster_fwd_kernel, maps, p));
  B2C_LAUNCH_CHECK("recur_cluster_fwd_kernel");
  recur_trace_state().grid = ncl * CR_CL; recur_trace_state().T = s.T;
  return 0;
}

// ------------------------------------------------------------------ decoder forward (teacher forced)
// Per step: u = q W_h^T  ->  attention (ctx lands in layer 0's operand)  ->  L fused gate-GEMM + cell kernels.
// The feature-independent part of the forward: packed operands (bf16 copies, attention_combine folded into layer 0), embedding
// rows, the time-batched embedding half of layer 0's gates and the zero initial state, all into the TRAIN workspace.
template <typename T>
int decoder_prepare_impl(const B2CShape& s, const B2CParams& p, const int64_t* cap, void* ws, size_t ws_bytes, cudaStream_t st) {
  TrainWs<T> W; W.carve(ws, s);
  B2C_CHECK_ARG(ws_bytes >= W.bytes, "workspace too small: %zu < %zu", ws_bytes, W.bytes);
  const int B = s.B, Tn = s.T, E = s.E, H = s.H, L = s.L, V = s.V;
  const long TB = (long)Tn * B;
  B2C_TRY(pack_params<T>(s, p, W.w, st));
  embedding_gather_kernel<T><<<ew_grid(TB * E / 4), 256, 0, st>>>(p.embedding, cap, TB, E, V, W.emb, E);
  B2C_LAUNCH_CHECK("embedding_gather_kernel");
  for (int k = 0; k < L; ++k) {
    B2C_CUDA(cudaMemsetAsync(W.xh[k], 0, (size_t)B * (in_dim(s, k) + H) * sizeof(T), st));   // h_{-1} = 0
    B2C_CUDA(cudaMemsetAsync(W.c[k], 0, (size_t)B * H * sizeof(float), st));                  // c_{-1} = 0
  }
  // embedding half of layer 0's gate pre-activations for all steps:  G0 = emb (W_ih0 W_ce)^T + b_x
  B2C_TRY((gemm<T, T>(st, (int)TB, 4 * H, E, W.emb, E, 0, W.w.We, E, 0, W.G0, 4 * H, 0.f, W.w.bx)));
  if constexpr (sizeof(T) == 2) {
    // the cluster recurrence kernel reads the addend per gate row with the samples of a row slice contiguous
    if (const int ncl = cluster_plan(s)) {
      g0_cluster_layout_kernel<<<dim3(4 * H / 64, ncl, Tn), 256, 0, st>>>(reinterpret_cast<const bf16*>(W.G0), B, Tn, ncl, reinterpret_cast<bf16*>(W.G0T));
      B2C_LAUNCH_CHECK("g0_cluster_layout_kernel");
    }
  }
  return 0;
}

template <typename T>
int set_initial_state_impl(const B2CShape& s, const float* h0, const float* c0, void* ws, size_t ws_bytes, cudaStream_t st) {
  TrainWs<T> W; W.carve(ws, s);
  B2C_CHECK_ARG(ws_bytes >= W.bytes, "workspace too small: %zu < %zu", ws_bytes, W.bytes);
  for (int k = 0; k < s.L; ++k) {
    const int in = in_dim(s, k);
    // slot 0 of layer k's operand rows is [input_0 ; h_{-1}], slot 0 of its cell buffer is c_{-1}
    initial_state_kernel<T><<<ew_grid((long)s.B * s.H), 256, 0, st>>>(h0 + (size_t)k * s.B * s.H, c0 + (size_t)k * s.B * s.H, s.B, s.H,
                                                                     W.xh[k] + in, in + s.H, W.c[k]);
    B2C_LAUNCH_CHECK("initial_state_kernel");
  }
  return 0;
}

struct EvalOut { const void* teacher; int teacher_dtype; const int64_t* targets; float temperature; float* row_kl; float* row_ce; int* argmax; };

template <typename T>
int decoder_forward_impl(const B2CShape& s, const B2CParams& p, const T* feats, const int64_t* cap, T* logits, T* hid_top,
                         float* attw, void* ws, size_t ws_bytes, const B2CDropout& dr, cudaStream_t st, bool prepared,
                         const EvalOut* ev = nullptr, const int* steps = nullptr) {
  TrainWs<T> W; W.carve(ws, s);
  B2C_CHECK_ARG(ws_bytes >= W.bytes, "workspace too small: %zu < %zu", ws_bytes, W.bytes);
  const int B = s.B, Tn = s.T, S = s.S, E = s.E, H = s.H, L = s.L, V = s.V;
  const long TB = (long)Tn * B;
  if (!prepared) B2C_TRY(decoder_prepare_impl<T>(s, p, cap, ws, ws_bytes, st));
  // time-invariant half of the attention projection: P = F W_f^T + b_a
  B2C_TRY((gemm<T, float>(st, B * S, E, E, feats, E, 0, W.w.Wf, E, 0, W.P, E, 0.f, p.attn_b)));
  const int inL = in_dim(s, L - 1), ldL = inL + H;
  // A device step count (variable-length batch) takes the per-step kernels, which skip the steps past it; the whole-sequence kernels
  // (B2C_PERSISTENT, B2C_CLUSTER) and sub-batch streams (B2C_SUB_BATCHES) are not used then.
  SubPlan sp;
  B2C_TRY(fork_subs(sp, B, st, steps == nullptr));
  pdl_full_dependency_next();        // P / F are final before any kernel of the recurrence can start (attention prologues read them early)
  // bf16 mode: the whole T loop as ONE persistent cooperative kernel when the shape fits its plan (recurrent.cuh); the
  // per-step kernels below remain for fp32 parity mode, other shapes and B2C_PERSISTENT=0 (A/B)
  static const bool merge_rec = []() { const char* e = getenv("B2C_MERGE_REC"); return !(e && e[0] == '0'); }();      // A/B switch
  RecurPlan rplan{}; rplan.ok = false;
  // first choice: independent 8-CTA clusters, one per row slice (recur_cluster.cuh); no inter-layer dropout in that kernel yet
  int ncl = 0;
  if (sizeof(T) == 2 && sp.ns == 1 && !(dr.p > 0.f) && !steps) ncl = cluster_plan(s);
  if (ncl > 0) { B2C_TRY(cluster_forward<T>(st, s, ncl, W, feats, hid_top, attw)); rplan.ok = true; }
  else {
  if (sizeof(T) == 2 && sp.ns == 1 && !steps) rplan = recur_plan(s);
  if (rplan.ok) B2C_TRY(recur_forward<T>(st, s, rplan, W, feats, hid_top, attw, dr));
  }
  for (int t = 0; t < (rplan.ok ? 0 : Tn); ++t) {
    for (int i = 0; i < sp.ns; ++i) {
      cudaStream_t ss = sp.st[i];
      const long b0 = sp.b0[i];
      B2CShape sh = s; sh.B = sp.bn[i];
      StepScope gate(steps, t);              // every kernel of this step does nothing when t >= *steps
      const long row = (long)t * B + b0;                       // first row of this sub-batch at step t in a (T,B,.) buffer
      const T* q = W.xh[L - 1] + row * ldL + inL;
      float* u_t = W.u + row * E;
      // bf16 mode: W_h and the top layer's W_hh both act on the top layer's h_{t-1}, so ONE contraction [u_t | W_hh h_{t-1}] =
      // h_{t-1} [W_h ; W_hh]^T (N = E + 4H: 144 tiles instead of 16 at the same per-CTA feed, so the same ~5.5 us) takes the
      // recurrent half out of the top layer's gate GEMM: its K drops from in + H to in (393 -> 196 KB of TMA feed per CTA, the
      // bound of that kernel).  The attention kernel writes the dense u_t the backward reads.
      const bool merged = merge_rec && sizeof(T) == 2;
      const long ldur = E + 4 * H;
      float* ur = W.UR + b0 * ldur;
      if (merged) {
        B2C_TRY((gemm<T, float>(ss, sh.B, E + 4 * H, H, q, ldL, 0, W.w.Wuh, H, 0, ur, ldur)));
        B2C_TRY(attn_fwd<T>(ss, sh, W.P + b0 * S * E, feats + b0 * S * E, ur, W.xh[0] + row * (E + H), E + H, attw + row * S, ldur, u_t, steps, t));
      } else {
        B2C_TRY((gemm<T, float>(ss, sh.B, E, H, q, ldL, 0, W.w.Wh, H, 0, u_t, E)));
        B2C_TRY(attn_fwd<T>(ss, sh, W.P + b0 * S * E, feats + b0 * S * E, u_t, W.xh[0] + row * (E + H), E + H, attw + row * S, 0, nullptr, steps, t));
      }
      for (int k = 0; k < L; ++k) {
        const int in = in_dim(s, k), ld = in + H;
        const bool rec = merged && k == L - 1;
        B2C_TRY(lstm_layer_fwd<T>(ss, sh, W.w, k, W.xh[k] + row * ld, k == 0 ? W.G0 + row * 4 * H : (const T*)nullptr,
                                  W.c[k] + row * H, W.c[k] + (row + B) * H,
                                  W.gates[k] + row * 4 * H, W.xh[k] + (row + B) * ld + in,
                                  k + 1 < L ? W.xh[k + 1] + row * 2 * H : nullptr, k == L - 1 ? hid_top + row * H : nullptr,
                                  dr, row, rec ? ur + E : nullptr, ldur));
      }
    }
  }
  B2C_TRY(join_subs(sp));
  if (steps) {
    // Invariant I2 (variable-length batch): the time-batched work below and in the backward keeps M / K = Tn*B, and multiplies
    // the rows of the skipped steps by exact zeros (their logits and hidden-state gradients are zero, invariant I3).  Those rows of
    // the saves it reads must be finite for that (0 x NaN = NaN), and the workspace may hold anything: zero them.
    TailFill f;
    f.add(hid_top, (size_t)B * H * sizeof(T), Tn);
    f.add(attw, (size_t)B * S * sizeof(float), Tn);
    f.add(W.u, (size_t)B * E * sizeof(float), Tn);
    for (int k = 0; k < L; ++k) f.add(W.xh[k], (size_t)B * (in_dim(s, k) + H) * sizeof(T), Tn);
    B2C_TRY(f.launch(steps, st));
  }
  // output head, time-batched: y = W2 Drop(ReLU(W1 h + b1)) + b2
  B2C_TRY((gemm<T, T>(st, (int)TB, E, H, hid_top, H, 0, W.w.W1, H, 0, W.o1, E, 0.f, p.out0_b, 1)));
  if (dr.p > 0.f) {
    dropout_inplace_kernel<T><<<ew_grid(TB * E), 256, 0, st>>>(W.o1, TB * E, dr.p, dr.seed, 100u, (const unsigned long long*)dr.seed_dev);
    B2C_LAUNCH_CHECK("dropout_inplace_kernel");
  }
  if (ev) {
    // validation: the vocabulary-head GEMM reduces its tiles to per-row partials of token KD / CE / argmax against the teacher
    // logits (no logits tensor is written or read back), merged by one small kernel
    GemmArgs gv{(int)TB, V, E, 1.f, 0.f, W.o1, (long)E, 0, W.w.W2, (long)E, 0, nullptr, (long)V, p.out3_b, 0};
    B2C_CHECK_ARG(sizeof(T) == 2 && tc_eligible(gv), "the logits-free validation forward needs bf16 mode and a TMA-describable vocabulary head");
    EvalEpi ee{ev->teacher, ev->targets, W.evalp, 1.0f / ev->temperature, 0, 0, ev->teacher_dtype};
    gv.eval = &ee;
    B2C_TRY((Gemm<T, float>::run(gv, st)));
    kd_eval_combine_kernel<<<cdiv(TB, 8), 256, 0, st>>>(W.evalp, ee.nparts, TB, V, ev->targets, 1.0f / ev->temperature, ev->row_kl, ev->row_ce, ev->argmax);
    B2C_LAUNCH_CHECK("kd_eval_combine_kernel");
    return 0;
  }
  B2C_TRY((gemm<T, T>(st, (int)TB, V, E, W.o1, E, 0, W.w.W2, E, 0, logits, V, 0.f, p.out3_b)));
  return 0;
}



// CTAs granted to each persistent GEMM that runs on a side stream UNDER a recurrence (B2C_BG_CTAS, 0 = no limit; default 10: two side
// streams -- this library's and the caller's projector backward -- share the 20 SMs the chain's <= 128-CTA kernels leave free), and the number of time-step chunks in which the LSTM weight gradients are contracted under
// the reverse recurrence instead of after it (B2C_WGRAD_CHUNKS, 0 = all after the loop).  Measured on B200, same box (KD step):
// no cap 2.675 ms; cap 20 -> 2.660; cap 20 + 2 / 4 / 5 chunks under the loop -> 2.666 / 2.857 / 3.07 ms (20 CTAs do not finish a chunk
// before the next one is due, and the post-loop work queues behind them); cap 12 / 32 with 4 chunks -> 3.22 / 2.71 ms.
// With the merged recurrent half (2.645 ms without a cap): cap 8 / 10 / 14 / 20 -> 2.628 / 2.626 / 2.648 / 2.634 ms.
inline int bg_ctas() { static int v = -1; if (v < 0) { const char* e = getenv("B2C_BG_CTAS"); v = e ? atoi(e) : 10; } return v; }
inline bool attn_post_occ3() { static int v = -1; if (v < 0) { const char* e = getenv("B2C_POST_OCC3"); v = (e && e[0] == '0') ? 0 : 1; } return v != 0; }
inline int wgrad_chunks() { static int v = -1; if (v < 0) { const char* e = getenv("B2C_WGRAD_CHUNKS"); v = e ? atoi(e) : 0; } return v; }

// ------------------------------------------------------------------ decoder backward (BPTT), oracle/manual_backward.py v2
template <typename T>
int decoder_backward_impl(const B2CShape& s, const B2CParams& p, const T* feats, const int64_t* cap, const T* hid_top,
                          const float* attw, const T* dlogits, const T* dhid, const B2CGrads& g, float* dfeats,
                          void* ws, size_t ws_bytes, const B2CDropout& dr, cudaStream_t st, int flags, long ld_dl = 0 /* 0 = V */,
                          const int* steps = nullptr) {
  TrainWs<T> W; W.carve(ws, s);
  B2C_CHECK_ARG(ws_bytes >= W.bytes, "workspace too small: %zu < %zu", ws_bytes, W.bytes);
  B2C_CHECK_ARG(g.embedding && g.attn_w && g.attn_b && g.comb_w && g.comb_b && g.out0_w && g.out0_b && g.out3_w && g.out3_b && dfeats, "NULL gradient pointer");
  const int B = s.B, Tn = s.T, S = s.S, E = s.E, H = s.H, L = s.L, V = s.V;
  const long TB = (long)Tn * B;
  if (ld_dl == 0) ld_dl = V;
  const float inv_keep = dr.p > 0.f ? 1.0f / (1.0f - dr.p) : 1.0f;
  SubStreams* hs = nullptr;
  B2C_TRY(get_substreams(&hs));
  cudaStream_t side = hs->s[MAX_SUB - 1];
  // input-gradient slots of every layer and step, zeroed once (the dxh GEMMs accumulate with beta = 1 so they may split K):
  // 70 MB of fills, on the side stream while the head runs, joined before the recurrence
  for (int k = 0; k < L; ++k) B2C_CHECK_ARG(g.w_ih[k] && g.w_hh[k] && g.b_ih[k] && g.b_hh[k], "NULL LSTM gradient pointer (layer %d)", k);
  B2C_CUDA(cudaEventRecord(hs->ev[3], st));
  B2C_CUDA(cudaStreamWaitEvent(side, hs->ev[3], 0));
  B2C_CUDA(cudaMemsetAsync(W.dxh0, 0, (size_t)TB * (E + H) * sizeof(float), side));
  for (int k = 1; k < L; ++k) B2C_CUDA(cudaMemsetAsync(W.dxh[k], 0, (size_t)TB * 2 * H * sizeof(float), side));
  if (steps) {
    // Invariant I3 (variable-length batch): the skipped steps write no gate, u or score gradients, and the post-loop contractions
    // read Tn*B rows of them: zero those rows.  (dxh0 / dxh[k] are zeroed above; the dlogits / dhidden_top rows of the skipped
    // steps are zeros by the caller's contract, so d(o1) and dH_ext are too.)
    TailFill f;
    for (int k = 0; k < L; ++k) f.add(W.dgates[k], (size_t)B * 4 * H * sizeof(T), Tn);
    f.add(W.du, (size_t)B * E * sizeof(T), Tn);
    f.add(W.ds, (size_t)B * S * sizeof(float), Tn);
    B2C_TRY(f.launch(steps, side));
  }
  B2C_CUDA(cudaEventRecord(hs->ev[3], side));
  // ---- output head (time-batched).  Only d(o1) -> dH_ext feeds the time loop; the head's weight gradients run on a side
  // stream underneath the (latency-bound) recurrence and are joined after it.
  B2C_TRY((gemm<T, T>(st, (int)TB, E, V, dlogits, ld_dl, 0, W.w.W2, E, 1, W.do1, E)));
  relu_bwd_inplace_kernel<T><<<ew_grid(TB * E), 256, 0, st>>>(W.do1, W.o1, TB * E, inv_keep);
  B2C_LAUNCH_CHECK("relu_bwd_inplace_kernel");
  B2C_CUDA(cudaEventRecord(hs->fork, st));
  B2C_CUDA(cudaStreamWaitEvent(side, hs->fork, 0));
  {
    GemmCapScope bg(bg_ctas());          // these run under the reverse recurrence: confined to the SMs the chain leaves free
    B2C_TRY((gemm<T, float>(side, V, E, (int)TB, dlogits, ld_dl, 1, W.o1, E, 1, g.out3_w, E)));
    B2C_TRY(colsum<T>(side, dlogits, TB, V, ld_dl, W.partial_side, g.out3_b));
    B2C_TRY((gemm<T, float>(side, E, H, (int)TB, W.do1, E, 1, hid_top, H, 1, g.out0_w, H)));
    B2C_TRY(colsum<T>(side, W.do1, TB, E, E, W.partial_side, g.out0_b));
  }
  B2C_CUDA(cudaEventRecord(hs->join[MAX_SUB - 1], side));
  B2C_TRY((gemm<T, float>(st, (int)TB, H, E, W.do1, E, 0, W.w.W1, H, 1, W.dHext, H)));
  // ---- reverse time loop
  B2C_CUDA(cudaStreamWaitEvent(st, hs->ev[3], 0));                 // the zeroed dxh slots
  SubPlan sp;
  B2C_TRY(fork_subs(sp, B, st, steps == nullptr));       // a device step count: no sub-batch streams (as in the forward)
  // Time-batched LSTM weight gradients over rows [r0, r1) of the (T*B, .) buffers (4H-sized rows come out interleaved and are
  // written gate-major).  They run on the side stream after the recurrence, next to the attn_post -> dF chain on the main one.
  // (Measured on B200: contracting the finished half of the steps on the side stream UNDER the recurrence slowed the chain by
  // as much as it hid: 3.29 vs 3.26 ms / step.)
  auto weight_grads = [&](cudaStream_t s2, long r0, long r1, float beta) -> int {
    const int K = (int)(r1 - r0);
    for (int k = 1; k < L; ++k) {
      const int in = in_dim(s, k), ld = in + H;
      B2C_TRY((gemm<T, float>(s2, 4 * H, in, K, W.dgates[k] + r0 * 4 * H, 4 * H, 1, W.xh[k] + r0 * ld, ld, 1, g.w_ih[k], in, beta, nullptr, 0, 1.f, H)));
      B2C_TRY((gemm<T, float>(s2, 4 * H, H, K, W.dgates[k] + r0 * 4 * H, 4 * H, 1, W.xh[k] + r0 * ld + in, ld, 1, g.w_hh[k], H, beta, nullptr, 0, 1.f, H)));
    }
    B2C_TRY((gemm<T, float>(s2, 4 * H, E, K, W.dgates[0] + r0 * 4 * H, 4 * H, 1, W.xh[0] + r0 * (E + H), E + H, 1, W.dWx32, E, beta)));
    B2C_TRY((gemm<T, float>(s2, 4 * H, E, K, W.dgates[0] + r0 * 4 * H, 4 * H, 1, W.emb + r0 * E, E, 1, W.dWe32, E, beta)));
    B2C_TRY((gemm<T, float>(s2, 4 * H, H, K, W.dgates[0] + r0 * 4 * H, 4 * H, 1, W.xh[0] + r0 * (E + H) + E, E + H, 1, g.w_hh[0], H, beta, nullptr, 0, 1.f, H)));
    return 0;
  };
  // LSTM weight gradients of the steps already traversed, contracted in chunks on the side stream while the loop goes on (capped
  // grid, see gemm_cta_cap): the side branch that used to end ~70 us after the main chain is mostly done when the loop ends.
  const int n_chunks = (sp.ns == 1 && bg_ctas() > 0 && !steps) ? wgrad_chunks() : 0;      // not with a device step count (steps unknown here)
  const int chunk_steps = n_chunks > 0 ? cdiv(Tn, n_chunks) : 0;
  long wg_done_from = TB;              // rows [wg_done_from, TB) have been contracted
  bool wg_any = false;
  pdl_full_dependency_next();        // the forward's saves (P, u, attention weights) are final before the reverse recurrence starts
  // Variable-length batch: every kernel of step t >= *steps does nothing but its griddepcontrol.launch_dependents / wait (invariant
  // I1: without the wait, a skipped grid could complete before its predecessors, and the post-loop kernels, which wait for the last
  // grid of the chain only, would race with step *steps - 1).  The cell adjoint of step *steps - 1 treats itself as the last step
  // (invariant I4: no carry, no dq, no dc from the skipped steps or an earlier call).
  for (int t = Tn - 1; t >= 0; --t) {
    const bool last = (t == Tn - 1);
    for (int i = 0; i < sp.ns; ++i) {
      cudaStream_t ss = sp.st[i];
      const long b0 = sp.b0[i];
      const int Bh = sp.bn[i];
      StepScope gate(steps, t);
      const long row = (long)t * B + b0;
      for (int k = L - 1; k >= 0; --k) {
        const int in = in_dim(s, k), ld = in + H;
        const float* carry = last ? nullptr : (k == 0 ? W.dxh0 + (row + B) * (E + H) + E : W.dxh[k] + (row + B) * 2 * H + H);
        const float* above = (k < L - 1) ? W.dxh[k + 1] + row * 2 * H : nullptr;
        const bool top = (k == L - 1);
        B2C_CUDA(launch_pdl(lstm_pointwise_bwd_kernel<T>, dim3(ew_grid((long)Bh * H)), dim3(256), 0, ss,
            (const T*)(W.gates[k] + row * 4 * H), (const float*)(W.c[k] + row * H), (const float*)(W.c[k] + (row + B) * H), W.dc[k] + b0 * H, last ? 1 : 0,
            carry, (long)ld, above, (long)(2 * H), (const float*)(top ? W.dHext + row * H : nullptr), (const T*)((top && dhid) ? dhid + row * H : nullptr),
            (const T*)((top && !last) ? W.dq + b0 * H : nullptr), (long)H, W.dgates[k] + row * 4 * H, Bh, H, dr.p, dr.seed, (uint32_t)k, row, (const unsigned long long*)dr.seed_dev,
            steps, t));
        B2C_LAUNCH_CHECK("lstm_pointwise_bwd_kernel");
        float* out = (k == 0) ? W.dxh0 + row * (E + H) : W.dxh[k] + row * 2 * H;
        B2C_TRY((gemm<T, float>(ss, Bh, ld, 4 * H, W.dgates[k] + row * 4 * H, 4 * H, 0, W.w.Wcat[k], ld, 1, out, ld, 1.f)));
      }
      // layer 0's input gradient IS d(ctx_t): no context GEMM on the chain
      const float* dctx_t = W.dxh0 + row * (E + H);
      T* du_t = W.du + row * E;
      B2C_TRY(attn_bwd<T>(ss, Bh, S, E, W.P + b0 * S * E, feats + b0 * S * E, W.u + row * E, attw + row * S, dctx_t, (long)(E + H), W.ds + row * S, du_t, steps, t));
      if (t > 0) B2C_TRY((gemm<T, T>(ss, Bh, H, E, du_t, E, 0, W.w.Wh, H, 1, W.dq + b0 * H, H)));
    }
    if (chunk_steps > 0 && t > 0 && (Tn - t) % chunk_steps == 0 && t >= chunk_steps) {
      // steps t .. t + chunk_steps - 1 are final (their dgates rows are written by the cell adjoints above)
      B2C_CUDA(cudaEventRecord(hs->ev[0], st));
      B2C_CUDA(cudaStreamWaitEvent(side, hs->ev[0], 0));
      GemmCapScope bg(bg_ctas());
      B2C_TRY(weight_grads(side, (long)t * B, wg_done_from, wg_any ? 1.f : 0.f));
      wg_done_from = (long)t * B; wg_any = true;
    }
  }
  B2C_TRY(join_subs(sp));
  // ---- post-loop.  Main stream: the chain the caller waits for (attn_post -> dF).  Side stream: every weight gradient.
  B2C_CUDA(cudaEventRecord(hs->ev[1], st));
  B2C_CUDA(cudaStreamWaitEvent(side, hs->ev[1], 0));
  B2C_TRY(weight_grads(side, 0, wg_done_from, wg_any ? 1.f : 0.f));
  for (int k = 0; k < L; ++k) B2C_TRY(colsum<T>(side, W.dgates[k], TB, 4 * H, 4 * H, W.partial_side, g.b_ih[k], g.b_hh[k], H));
  {
    // layer 0 with attention_combine folded in:  dW_x = dg0^T ctx,  dW_e = dg0^T emb,  db_x = colsum(dg0)
    cast_f32_kernel<T><<<ew_grid((long)4 * H * E / 8), 256, 0, side>>>(W.dWx32, W.dWxT, (long)4 * H * E);
    B2C_LAUNCH_CHECK("cast_f32_kernel");
    cast_f32_kernel<T><<<ew_grid((long)4 * H * E / 8), 256, 0, side>>>(W.dWe32, W.dWeT, (long)4 * H * E);
    B2C_LAUNCH_CHECK("cast_f32_kernel");
    // dW_ih0 = dW_x W_cc^T + dW_e W_ce^T + db_x (x) b_c
    B2C_TRY((gemm<T, float>(side, 4 * H, E, E, W.dWxT, E, 0, W.w.Wcc, E, 0, g.w_ih[0], E, 0.f, nullptr, 0, 1.f, H)));
    B2C_TRY((gemm<T, float>(side, 4 * H, E, E, W.dWeT, E, 0, W.w.Wce, E, 0, g.w_ih[0], E, 1.f, nullptr, 0, 1.f, H)));
    rank1_add_kernel<<<ew_grid((long)4 * H * E), 256, 0, side>>>(g.w_ih[0], g.b_ih[0], p.comb_b, (long)4 * H, E);
    B2C_LAUNCH_CHECK("rank1_add_kernel");
    // dW_c = [W_ih0^T dW_e | W_ih0^T dW_x],  db_c = W_ih0^T db_x
    B2C_TRY((gemm<T, float>(side, E, E, 4 * H, W.w.Wih0, E, 1, W.dWeT, E, 1, g.comb_w, 2 * E)));
    B2C_TRY((gemm<T, float>(side, E, E, 4 * H, W.w.Wih0, E, 1, W.dWxT, E, 1, g.comb_w + E, 2 * E)));
    B2C_CUDA(cudaMemsetAsync(g.comb_b, 0, (size_t)E * sizeof(float), side));
    bias_fold_bwd_kernel<<<dim3(cdiv(E, 32), 32), 256, 0, side>>>(p.w_ih[0], g.b_ih[0], 4 * H, E, g.comb_b);
    B2C_LAUNCH_CHECK("bias_fold_bwd_kernel");
    // embedding rows: demb = dg0 W_e
    B2C_TRY((gemm<T, float>(side, (int)TB, E, 4 * H, W.dgates[0], 4 * H, 0, W.w.We, E, 1, W.demb, E)));
    B2C_CUDA(cudaMemsetAsync(g.embedding, 0, (size_t)V * E * sizeof(float), side));
    embedding_scatter_add_kernel<<<ew_grid(TB * E), 256, 0, side>>>(W.demb, cap, TB, E, V, g.embedding);
    B2C_LAUNCH_CHECK("embedding_scatter_add_kernel");
  }
  const int inL = in_dim(s, L - 1), ldL = inL + H;
  B2C_TRY((gemm<T, float>(side, E, H, (int)TB, W.du, E, 1, W.xh[L - 1] + inL, ldL, 1, g.attn_w, H + E)));          // dW_a[:, :H]
  if (Tn <= 24) {                       // u / dctx of all steps in registers (decoder_kernels.cuh)
    // one CTA per sample: the 2 x Tn register loads of a thread are amortised over all S tokens (measured: 1 split 2.76 ms / step,
    // 2 -> 2.79, 4 -> 2.79, 7 -> 2.81)
    const int splits = 1, per = cdiv(S, splits), TP = (Tn + 3) & ~3;
    const size_t psmem = (size_t)2 * per * TP * 4;
    if (Tn <= 20 && attn_post_occ3()) {        // u / dctx of 20 instead of 24 steps in registers: 64 registers, four CTAs per SM, all B = 512 CTAs in ONE wave
                                               // (ncu: 52 % long-scoreboard stalls at 25 % occupancy; 85 -> 65 us, KD step 2.63 -> 2.61 ms)
      B2C_TRY(set_smem(attn_post_reg_kernel<T, 20>, psmem));
      attn_post_reg_kernel<T, 20><<<dim3(B, splits), ATT_THREADS, psmem, st>>>(W.P, W.u, W.dxh0, (long)(E + H), attw, W.ds, Tn, B, S, E, W.dP, dfeats);
    } else {
      B2C_TRY(set_smem(attn_post_reg_kernel<T, 24>, psmem));          // > 48 KB only for very long token lists
      attn_post_reg_kernel<T, 24><<<dim3(B, splits), ATT_THREADS, psmem, st>>>(W.P, W.u, W.dxh0, (long)(E + H), attw, W.ds, Tn, B, S, E, W.dP, dfeats);
    }
    B2C_LAUNCH_CHECK("attn_post_reg_kernel");
  } else {
    const size_t smem = (size_t)Tn * (2 * E + 2 * S) * 4;
    B2C_TRY(set_smem(attn_post_kernel<T>, smem));
    attn_post_kernel<T><<<B, ATT_THREADS, smem, st>>>(W.P, W.u, W.dxh0, (long)(E + H), attw, W.ds, Tn, B, S, E, W.dP, dfeats);
    B2C_LAUNCH_CHECK("attn_post_kernel");
  }
  B2C_CUDA(cudaEventRecord(hs->ev[2], st));
  B2C_TRY((gemm<T, float>(st, B * S, E, E, W.dP, E, 0, W.w.Wf, E, 1, dfeats, E, 1.f)));                             // dF += dP W_f
  B2C_CUDA(cudaStreamWaitEvent(side, hs->ev[2], 0));
  B2C_TRY((gemm<T, float>(side, E, E, B * S, W.dP, E, 1, feats, E, 1, g.attn_w + H, H + E)));                      // dW_a[:, H:]
  B2C_TRY(colsum<T>(side, W.dP, (long)B * S, E, E, W.partial_side, g.attn_b));
  B2C_CUDA(cudaEventRecord(hs->join[MAX_SUB - 1], side));
  if (flags & B2C_BWD_DEFER_JOIN) return 0;                         // the caller joins with b2c_join_side_work
  B2C_CUDA(cudaStreamWaitEvent(st, hs->join[MAX_SUB - 1], 0));      // every weight gradient is complete when the call's work on `stream` is
  return 0;
}


inline bool fuse_argmax_off() { static const bool off = getenv("B2C_DECODE_LOGITS") != nullptr; return off; }     // A/B + debugging

// ------------------------------------------------------------------ greedy decode (eval, argmax fed back on device)
template <typename T>
int greedy_decode_impl(const B2CShape& s, const B2CParams& p, const T* feats, int64_t start_id, int64_t end_id,
                       int64_t* tokens, int32_t* lengths, void* ws, size_t ws_bytes, cudaStream_t st) {
  DecodeWs<T> W; W.carve(ws, s);
  B2C_CHECK_ARG(ws_bytes >= W.bytes, "workspace too small: %zu < %zu", ws_bytes, W.bytes);
  const int B = s.B, Tn = s.T, S = s.S, E = s.E, H = s.H, L = s.L, V = s.V;
  const B2CDropout nodrop{0.f, 0, nullptr};
  B2C_TRY(pack_params<T>(s, p, W.w, st));
  B2C_TRY((gemm<T, float>(st, B * S, E, E, feats, E, 0, W.w.Wf, E, 0, W.P, E, 0.f, p.attn_b)));
  for (int k = 0; k < L; ++k) {
    B2C_CUDA(cudaMemsetAsync(W.xh[k], 0, (size_t)2 * B * (in_dim(s, k) + H) * sizeof(T), st));
    B2C_CUDA(cudaMemsetAsync(W.c[k], 0, (size_t)B * H * sizeof(float), st));
  }
  fill_i64_kernel<<<ew_grid(B), 256, 0, st>>>(W.cur, B, start_id);
  B2C_LAUNCH_CHECK("fill_i64_kernel");
  const int inL = in_dim(s, L - 1), ldL = inL + H;
  for (int t = 0; t < Tn; ++t) {
    // The fused cell writes h_t while other CTAs of the same gate GEMM still read [input ; h_{t-1}]: two slots per layer,
    // step t reads slot t & 1 and writes the recurrent h into the other one.
    const int pcur = t & 1, pnxt = pcur ^ 1;
    auto slot = [&](int k, int which) { return W.xh[k] + (size_t)which * B * (in_dim(s, k) + H); };
    embedding_gather_kernel<T><<<ew_grid((long)B * E / 4), 256, 0, st>>>(p.embedding, W.cur, B, E, V, W.emb, E);
    B2C_LAUNCH_CHECK("embedding_gather_kernel");
    B2C_TRY((gemm<T, T>(st, B, 4 * H, E, W.emb, E, 0, W.w.We, E, 0, W.G0, 4 * H, 0.f, W.w.bx)));
    B2C_TRY((gemm<T, float>(st, B, E, H, slot(L - 1, pcur) + inL, ldL, 0, W.w.Wh, H, 0, W.u, E)));
    B2C_TRY(attn_fwd<T>(st, s, W.P, feats, W.u, slot(0, pcur), E + H, nullptr));
    for (int k = 0; k < L; ++k) {
      const int in = in_dim(s, k);
      B2C_TRY(lstm_layer_fwd<T>(st, s, W.w, k, slot(k, pcur), k == 0 ? W.G0 : (const T*)nullptr, W.c[k], W.c[k], (T*)nullptr, slot(k, pnxt) + in,
                                k + 1 < L ? slot(k + 1, pcur) : nullptr, (T*)nullptr, nodrop, 0));
    }
    B2C_TRY((gemm<T, T>(st, B, E, H, slot(L - 1, pnxt) + inL, ldL, 0, W.w.W1, H, 0, W.o1, E, 0.f, p.out0_b, 1)));
    // vocabulary head.  bf16 mode on the tcgen05 path: the GEMM's epilogue reduces every tile to per-row partial (max, index)
    // pairs, the logits are never written; otherwise (fp32 parity mode, or a pitch TMA cannot describe): logits + argmax kernel.
    GemmArgs gv{B, V, E, 1.f, 0.f, W.o1, (long)E, 0, W.w.W2, (long)E, 0, W.logits, (long)V, p.out3_b, 0};
    if (sizeof(T) == 2 && tc_eligible(gv) && !fuse_argmax_off()) {
      ArgmaxEpi ae{W.amax_v, W.amax_i, 0, 0};
      gv.amax = &ae;
      B2C_TRY((Gemm<T, float>::run(gv, st)));
      argmax_parts_feedback_kernel<<<cdiv(B, 8), 256, 0, st>>>(W.amax_v, W.amax_i, ae.nparts, B, end_id, t, W.cur, tokens + (long)t * B, lengths, W.done);
      B2C_LAUNCH_CHECK("argmax_parts_feedback_kernel");
    } else {
      B2C_TRY((Gemm<T, float>::run(gv, st)));
      argmax_feedback_kernel<<<B, 256, 0, st>>>(W.logits, V, V, end_id, t, W.cur, tokens + (long)t * B, lengths, W.done);
      B2C_LAUNCH_CHECK("argmax_feedback_kernel");
    }
  }
  finish_lengths_kernel<<<cdiv(B, 256), 256, 0, st>>>(lengths, B, Tn);
  B2C_LAUNCH_CHECK("finish_lengths_kernel");
  return 0;
}


template <typename T> struct AttnWs {
  T *Wh, *Wf; float *P, *u; size_t bytes;
  void carve(void* base, const B2CShape& s) {
    Carver c{reinterpret_cast<unsigned char*>(base), 0};
    Wh = c.take<T>((size_t)s.E * s.H); Wf = c.take<T>((size_t)s.E * s.E);
    P = c.take<float>((size_t)s.B * s.S * s.E); u = c.take<float>((size_t)s.B * s.E);
    bytes = align_up(c.off, 256);
  }
};

template <typename T>
int attention_step_impl(const B2CShape& s, const float* attn_w, const float* attn_b, const T* hidden, const T* feats,
                        T* context, float* weights, void* ws, size_t ws_bytes, cudaStream_t st) {
  AttnWs<T> W; W.carve(ws, s);
  B2C_CHECK_ARG(ws_bytes >= W.bytes, "workspace too small: %zu < %zu", ws_bytes, W.bytes);
  const int B = s.B, S = s.S, E = s.E, H = s.H;
  PackTable tab; tab.n = 2;
  tab.seg[0] = PackSeg{attn_w, W.Wh, nullptr, E, H, (long)H + E, (long)H, 0};
  tab.seg[1] = PackSeg{attn_w + H, W.Wf, nullptr, E, E, (long)H + E, (long)E, 0};
  pack_params_kernel<T><<<dim3(32, 2), 256, 0, st>>>(tab);
  B2C_LAUNCH_CHECK("pack_params_kernel");
  B2C_TRY((gemm<T, float>(st, B * S, E, E, feats, E, 0, W.Wf, E, 0, W.P, E, 0.f, attn_b)));
  pdl_full_dependency_next();        // the u contraction starts only after P is complete, so the attention prologue may read P
  B2C_TRY((gemm<T, float>(st, B, E, H, hidden, H, 0, W.Wh, H, 0, W.u, E)));
  return attn_fwd<T>(st, s, W.P, feats, W.u, context, (long)s.E, weights);
}

// ------------------------------------------------------------------ AttentionRefinement / FeatureProjector (SURVEY.md §8f rows 1-2)
constexpr int LN_GRID = 148 * 3;
template <typename T> struct RefineWs {
  T *Win, *Wo, *W1, *W2;                                         // packed operand weights
  T *x, *qkv, *probs, *attn, *proj, *x1, *f1, *f2;               // forward saves
  float *mean1, *rstd1, *mean2, *rstd2;
  T *dz2, *df1, *dz1, *dattn, *dqkv; float *dz1f, *lnpart, *partial;
  float *x1f, *dz2f;                                              // fp32 residual stream: LN1's output, and its gradient
  size_t bytes;
  void carve(void* base, const B2CShape& s) {
    Carver c{reinterpret_cast<unsigned char*>(base), 0};
    const size_t R = (size_t)s.B * s.S, E = s.E, heads = s.H;
    Win = c.take<T>(3 * E * E); Wo = c.take<T>(E * E); W1 = c.take<T>(2 * E * E); W2 = c.take<T>(2 * E * E);
    x = c.take<T>(R * E); qkv = c.take<T>(R * 3 * E); probs = c.take<T>((size_t)s.B * heads * s.S * (s.S > 64 ? s.S : 64)) /* mma path: row pitch 64 */; attn = c.take<T>(R * E);
    proj = c.take<T>(R * E); x1 = c.take<T>(R * E); f1 = c.take<T>(R * 2 * E); f2 = c.take<T>(R * E);
    mean1 = c.take<float>(R); rstd1 = c.take<float>(R); mean2 = c.take<float>(R); rstd2 = c.take<float>(R);
    dz2 = c.take<T>(R * E); df1 = c.take<T>(R * 2 * E); dz1 = c.take<T>(R * E); dattn = c.take<T>(R * E); dqkv = c.take<T>(R * 3 * E);
    dz1f = c.take<float>(R * E); lnpart = c.take<float>((size_t)LN_GRID * 3 * E); partial = c.take<float>((size_t)COLSUM_RS * 3 * E);
    x1f = c.take<float>(R * E); dz2f = c.take<float>(R * E);
    bytes = align_up(c.off, 256);
  }
};

int check_refine_shape(const B2CShape* s) {
  B2C_CHECK_ARG(s != nullptr, "shape is NULL");
  B2C_CHECK_ARG(s->B > 0 && s->S > 0 && s->E > 0 && s->H > 0, "bad refinement shape B=%d S=%d E=%d heads=%d", s->B, s->S, s->E, s->H);
  B2C_CHECK_ARG(s->E % 8 == 0 && s->E <= 256 * LN_MAXC && s->E % s->H == 0, "E=%d must be a multiple of 8 and of heads=%d, and <= %d", s->E, s->H, 256 * LN_MAXC);
  const size_t hd = s->E / s->H;
  B2C_CHECK_ARG(hd % 4 == 0, "head_dim=%zu must be a multiple of 4", hd);
  B2C_CHECK_ARG((4 * (size_t)s->S * mha_pitch((int)hd) + 3 * (size_t)s->S * mha_pitch(s->S)) * 4 <= 200 * 1024, "S=%d x head_dim=%zu does not fit the attention core's shared memory", s->S, hd);
  return 0;
}

template <typename TX, typename TR, typename TY>
int ln_fwd(cudaStream_t st, const TX* x, const TR* res, const float* g, const float* b, TY* y, float* y32, float* mean, float* rstd, long R, int E) {
  long grid = (R + 7) / 8; if (grid > 148 * 8) grid = 148 * 8;
  if (E <= 256) ln_fwd_kernel<TX, TR, TY, 1><<<(unsigned)grid, LN_THREADS, 0, st>>>(x, res, g, b, y, y32, mean, rstd, R, E, 1e-5f);
  else ln_fwd_kernel<TX, TR, TY, 2><<<(unsigned)grid, LN_THREADS, 0, st>>>(x, res, g, b, y, y32, mean, rstd, R, E, 1e-5f);
  B2C_LAUNCH_CHECK("ln_fwd_kernel");
  return 0;
}
// LayerNorm backward; dy is a tensor (dpool == nullptr) or pooled window gradients (projector).  dbias_prev (optional) receives
// the column sums of dz = the bias gradient of the Linear whose output entered the LayerNorm.
template <typename TX, typename TR, typename TDY, typename TDZ>
int ln_bwd(cudaStream_t st, const TDY* dy, const float* dpool, int L, int O, const TX* x, const TR* res, const float* mean, const float* rstd,
           const float* gamma, TDZ* dz, float* dz32, float* part, float* dgamma, float* dbeta, float* dbias_prev, long R, int E) {
  long grid = (R + 7) / 8; if (grid > LN_GRID) grid = LN_GRID;
  const size_t smem = (size_t)(LN_THREADS / 32) * 3 * E * 4;
#define B2C_LNB(POOLED, NC) do { B2C_TRY(set_smem(ln_bwd_kernel<TX, TR, TDY, TDZ, POOLED, NC>, smem)); \
    ln_bwd_kernel<TX, TR, TDY, TDZ, POOLED, NC><<<(unsigned)grid, LN_THREADS, smem, st>>>(dy, dpool, L, O, x, res, mean, rstd, gamma, dz, dz32, part, R, E); } while (0)
  if (dpool) { if (E <= 256) B2C_LNB(true, 1); else B2C_LNB(true, 2); }
  else { if (E <= 256) B2C_LNB(false, 1); else B2C_LNB(false, 2); }
#undef B2C_LNB
  B2C_LAUNCH_CHECK("ln_bwd_kernel");
  ln_param_grad_kernel<<<dim3(cdiv(E, 32), 3), 256, 0, st>>>(part, (int)grid, E, dgamma, dbeta, dbias_prev);
  B2C_LAUNCH_CHECK("ln_param_grad_kernel");
  return 0;
}

// column sums of a contiguous (rows, cols) matrix, cols % 8 == 0, optionally fused with the in-place ReLU backward
template <typename T>
int colsum_vec(cudaStream_t st, T* A, const T* act, long rows, int cols, float inv_keep, float* partial, float* out) {
  const int gx = cdiv(cols, 256);
  int rs = (int)((rows + 31) / 32); if (rs > 592 / gx) rs = 592 / gx; if (rs > COLSUM_RS) rs = COLSUM_RS; if (rs < 1) rs = 1;
  dim3 grid(gx, rs);
  if (act) colsum_vec_kernel<T, true><<<grid, 256, 0, st>>>(A, act, rows, cols, inv_keep, partial);
  else colsum_vec_kernel<T, false><<<grid, 256, 0, st>>>(A, act, rows, cols, inv_keep, partial);
  B2C_LAUNCH_CHECK("colsum_vec_kernel");
  colsum_final_kernel<<<cdiv(cols, 256), 256, 0, st>>>(partial, rs, cols, out, nullptr);
  B2C_LAUNCH_CHECK("colsum_final_kernel");
  return 0;
}

template <typename T>
int refine_pack(const B2CShape& s, const B2CRefineParams& p, const RefineWs<T>& W, cudaStream_t st) {
  B2C_CHECK_ARG(p.in_w && p.in_b && p.out_w && p.out_b && p.ffn0_w && p.ffn0_b && p.ffn3_w && p.ffn3_b && p.n1_w && p.n1_b && p.n2_w && p.n2_b, "NULL refinement parameter");
  const int E = s.E;
  PackTable tab; tab.n = 4;
  tab.seg[0] = PackSeg{p.in_w, W.Win, nullptr, 3 * E, E, (long)E, (long)E, 0};
  tab.seg[1] = PackSeg{p.out_w, W.Wo, nullptr, E, E, (long)E, (long)E, 0};
  tab.seg[2] = PackSeg{p.ffn0_w, W.W1, nullptr, 2 * E, E, (long)E, (long)E, 0};
  tab.seg[3] = PackSeg{p.ffn3_w, W.W2, nullptr, E, 2 * E, (long)2 * E, (long)2 * E, 0};
  pack_params_kernel<T><<<dim3(48, 4), 256, 0, st>>>(tab);
  B2C_LAUNCH_CHECK("pack_params_kernel");
  return 0;
}

// bf16 mode, head_dim 64, at most 64 tokens: tensor-core kernels (mha_mma.cuh); anything else: FFMA register tiles
template <typename T> inline bool mha_use_mma(int S, int hd) { return false; }
template <> inline bool mha_use_mma<bf16>(int S, int hd) {
  static const bool off = getenv("B2C_MHA_FFMA") != nullptr;
  return !off && hd == 64 && S <= 64;
}

template <typename T>
int refinement_forward_impl(const B2CShape& s, const B2CRefineParams& p, const float* x, float* out, void* ws, size_t ws_bytes,
                            const B2CDropout& dr, cudaStream_t st, T* out_compute = nullptr) {
  RefineWs<T> W; W.carve(ws, s);
  B2C_CHECK_ARG(ws_bytes >= W.bytes, "workspace too small: %zu < %zu", ws_bytes, W.bytes);
  const int B = s.B, S = s.S, E = s.E, heads = s.H, hd = E / heads;
  const long R = (long)B * S;
  B2C_TRY(refine_pack<T>(s, p, W, st));
  cast_f32_kernel<T><<<ew_grid(R * E / 4), 256, 0, st>>>(x, W.x, R * E);
  B2C_LAUNCH_CHECK("cast_f32_kernel");
  B2C_TRY((gemm<T, T>(st, (int)R, 3 * E, E, W.x, E, 0, W.Win, E, 0, W.qkv, 3 * E, 0.f, p.in_b)));
  if (mha_use_mma<T>(S, hd)) {
    mha_fwd_mma_kernel<<<dim3(B, heads), MM_THREADS, 0, st>>>((const bf16*)W.qkv, (bf16*)W.attn, (bf16*)W.probs, S, E, heads, 1.0f / sqrtf((float)hd),
                                                             dr.p, dr.seed, MHA_DROP_SITE, (const unsigned long long*)dr.seed_dev);
    B2C_LAUNCH_CHECK("mha_fwd_mma_kernel");
  } else {
    const size_t smem = ((size_t)3 * S * mha_pitch(hd) + (size_t)S * mha_pitch(S)) * 4;
    B2C_TRY(set_smem(mha_fwd_kernel<T>, smem));
    mha_fwd_kernel<T><<<dim3(B, heads), MHA_THREADS, smem, st>>>(W.qkv, W.attn, W.probs, S, E, heads, 1.0f / sqrtf((float)hd), dr.p, dr.seed, (const unsigned long long*)dr.seed_dev);
    B2C_LAUNCH_CHECK("mha_fwd_kernel");
  }
  B2C_TRY((gemm<T, T>(st, (int)R, E, E, W.attn, E, 0, W.Wo, E, 0, W.proj, E, 0.f, p.out_b)));
  // The residual stream stays in fp32 in both modes (torch.autocast runs LayerNorm in fp32 too): LN1 takes the fp32 block input
  // + the branch output and leaves x1 twice, in the compute type (operand of the FFN contractions) and in fp32 (residual of LN2).
  B2C_TRY((ln_fwd<float, T, T>(st, x, W.proj, p.n1_w, p.n1_b, W.x1, W.x1f, W.mean1, W.rstd1, R, E)));
  B2C_TRY((gemm<T, T>(st, (int)R, 2 * E, E, W.x1, E, 0, W.W1, E, 0, W.f1, 2 * E, 0.f, p.ffn0_b, 1)));
  if (dr.p > 0.f) {
    dropout_inplace_kernel<T><<<ew_grid(R * 2 * E), 256, 0, st>>>(W.f1, R * 2 * E, dr.p, dr.seed, 201u, (const unsigned long long*)dr.seed_dev);
    B2C_LAUNCH_CHECK("dropout_inplace_kernel");
  }
  B2C_TRY((gemm<T, T>(st, (int)R, E, 2 * E, W.f1, 2 * E, 0, W.W2, 2 * E, 0, W.f2, E, 0.f, p.ffn3_b)));
  if (out_compute) B2C_TRY((ln_fwd<float, T, T>(st, W.x1f, W.f2, p.n2_w, p.n2_b, out_compute, out, W.mean2, W.rstd2, R, E)));      // both copies from one pass
  else B2C_TRY((ln_fwd<float, T, float>(st, W.x1f, W.f2, p.n2_w, p.n2_b, (float*)nullptr, out, W.mean2, W.rstd2, R, E)));
  return 0;
}

template <typename T>
int refinement_backward_impl(const B2CShape& s, const B2CRefineParams& p, const float* x, const float* dout, const B2CRefineGrads& g, float* dx,
                             void* ws, size_t ws_bytes, const B2CDropout& dr, cudaStream_t st) {
  RefineWs<T> W; W.carve(ws, s);
  B2C_CHECK_ARG(ws_bytes >= W.bytes, "workspace too small: %zu < %zu", ws_bytes, W.bytes);
  B2C_CHECK_ARG(g.in_w && g.in_b && g.out_w && g.out_b && g.ffn0_w && g.ffn0_b && g.ffn3_w && g.ffn3_b && g.n1_w && g.n1_b && g.n2_w && g.n2_b && dx, "NULL refinement gradient");
  const int B = s.B, S = s.S, E = s.E, heads = s.H, hd = E / heads;
  const long R = (long)B * S;
  const float inv_keep = dr.p > 0.f ? 1.0f / (1.0f - dr.p) : 1.0f;
  // out = LN2(x1 + f2);  f2 = f1 W2^T + b2  (its bias gradient = column sums of dz2, produced by the same kernel)
  // (fp32 residual stream: dout arrives in fp32, d(x1 + f2) leaves in the compute type for the contractions AND in fp32)
  B2C_TRY((ln_bwd<float, T, float, T>(st, dout, nullptr, 0, 0, W.x1f, W.f2, W.mean2, W.rstd2, p.n2_w, W.dz2, W.dz2f, W.lnpart, g.n2_w, g.n2_b, g.ffn3_b, R, E)));
  B2C_TRY((gemm<T, float>(st, E, 2 * E, (int)R, W.dz2, E, 1, W.f1, 2 * E, 1, g.ffn3_w, 2 * E)));
  B2C_TRY((gemm<T, T>(st, (int)R, 2 * E, E, W.dz2, E, 0, W.W2, 2 * E, 1, W.df1, 2 * E)));
  // f1 = Drop(ReLU(x1 W1^T + b1)): mask in place + bias gradient in one pass
  B2C_TRY(colsum_vec<T>(st, W.df1, W.f1, R, 2 * E, inv_keep, W.partial, g.ffn0_b));
  B2C_TRY((gemm<T, float>(st, 2 * E, E, (int)R, W.df1, 2 * E, 1, W.x1, E, 1, g.ffn0_w, E)));
  B2C_TRY((gemm<T, float>(st, (int)R, E, 2 * E, W.df1, 2 * E, 0, W.W1, E, 1, W.dz2f, E, 1.f)));      // dz2f <- d(x1) = dz2 + df1 W1, accumulated in fp32
  // x1 = LN1(x + proj);  proj = attn Wo^T + bo
  B2C_TRY((ln_bwd<float, T, float, T>(st, W.dz2f, nullptr, 0, 0, x, W.proj, W.mean1, W.rstd1, p.n1_w, W.dz1, W.dz1f, W.lnpart, g.n1_w, g.n1_b, g.out_b, R, E)));
  B2C_TRY((gemm<T, float>(st, E, E, (int)R, W.dz1, E, 1, W.attn, E, 1, g.out_w, E)));
  B2C_TRY((gemm<T, T>(st, (int)R, E, E, W.dz1, E, 0, W.Wo, E, 1, W.dattn, E)));
  if (mha_use_mma<T>(S, hd)) {
    const size_t smem = (size_t)(dr.p > 0.f ? 7 : 6) * MM_TILE * sizeof(bf16);
    B2C_TRY(set_smem(mha_bwd_mma_kernel, smem));
    mha_bwd_mma_kernel<<<dim3(B, heads), MM_THREADS, smem, st>>>((const bf16*)W.qkv, (const bf16*)W.probs, (const bf16*)W.dattn, (bf16*)W.dqkv, S, E, heads,
                                                                1.0f / sqrtf((float)hd), dr.p, dr.seed, MHA_DROP_SITE, (const unsigned long long*)dr.seed_dev);
    B2C_LAUNCH_CHECK("mha_bwd_mma_kernel");
  } else {
    const size_t smem = ((size_t)4 * S * mha_pitch(hd) + (size_t)(dr.p > 0.f ? 3 : 2) * S * mha_pitch(S)) * 4;
    B2C_TRY(set_smem(mha_bwd_kernel<T>, smem));
    mha_bwd_kernel<T><<<dim3(B, heads), MHA_THREADS, smem, st>>>(W.qkv, W.probs, W.dattn, W.dqkv, S, E, heads, 1.0f / sqrtf((float)hd), dr.p, dr.seed, (const unsigned long long*)dr.seed_dev);
    B2C_LAUNCH_CHECK("mha_bwd_kernel");
  }
  // qkv = x Win^T + b
  B2C_TRY((gemm<T, float>(st, 3 * E, E, (int)R, W.dqkv, 3 * E, 1, W.x, E, 1, g.in_w, E)));
  B2C_TRY(colsum_vec<T>(st, W.dqkv, (const T*)nullptr, R, 3 * E, 1.f, W.partial, g.in_b));
  B2C_CUDA(cudaMemcpyAsync(dx, W.dz1f, (size_t)R * E * sizeof(float), cudaMemcpyDeviceToDevice, st));   // residual path
  B2C_TRY((gemm<T, float>(st, (int)R, E, 3 * E, W.dqkv, 3 * E, 0, W.Win, E, 1, dx, E, 1.f)));        // dx += dqkv Win
  return 0;
}

template <typename T> struct ProjWs {
  T *Wp, *xb, *h, *dh; float *mean, *rstd, *lnpart, *partial;
  size_t bytes;
  void carve(void* base, const B2CShape& s, bool identity) {
    Carver c{reinterpret_cast<unsigned char*>(base), 0};
    const size_t R = (size_t)s.B * s.S, Et = s.E, Es = s.H;
    if (!identity) {
      Wp = c.take<T>(Es * Et); xb = c.take<T>(R * Et); h = c.take<T>(R * Es);
      dh = c.take<T>(R * Es); mean = c.take<float>(R); rstd = c.take<float>(R);
      lnpart = c.take<float>((size_t)LN_GRID * 3 * Es); partial = c.take<float>((size_t)COLSUM_RS * Es);
    }
    bytes = align_up(c.off + 256, 256);
  }
};
int check_proj_shape(const B2CShape* s) {
  B2C_CHECK_ARG(s != nullptr, "shape is NULL");
  B2C_CHECK_ARG(s->B > 0 && s->S > 0 && s->E > 0 && s->H > 0 && s->T > 0 && s->T <= s->S, "bad projector shape B=%d St=%d Et=%d Es=%d So=%d", s->B, s->S, s->E, s->H, s->T);
  B2C_CHECK_ARG(s->E % 8 == 0 && s->H % 8 == 0 && s->H <= 256 * LN_MAXC, "Et=%d / Es=%d must be multiples of 8 and Es <= %d", s->E, s->H, 256 * LN_MAXC);
  B2C_CHECK_ARG((long)s->B * s->S < 2147483647L && (long)s->S * s->T < 2147483647L, "B*St and St*So must stay below 2^31 (32-bit index arithmetic in the pooled LayerNorm kernels)");
  return 0;
}

template <typename T, typename TZ>          // TZ: the teacher features' type (float, bf16 or f16)
int projector_forward_impl(const B2CShape& s, const B2CProjParams& p, const TZ* x, float* out, void* ws, size_t ws_bytes,
                           const B2CDropout& dr, cudaStream_t st) {
  const bool identity = (p.w == nullptr);
  const int B = s.B, St = s.S, Et = s.E, Es = s.H, So = s.T;
  const long R = (long)B * St;
  if (identity) {
    B2C_CHECK_ARG(Et == Es && !p.b && !p.ln_w && !p.ln_b, "identity projection needs Et == Es and no parameters");
    pool_fwd_kernel<TZ><<<ew_grid((long)B * So * Es), 256, 0, st>>>(x, out, B, St, So, Es);
    B2C_LAUNCH_CHECK("pool_fwd_kernel");
    return 0;
  }
  B2C_CHECK_ARG(p.b && p.ln_w && p.ln_b, "NULL projector parameter");
  ProjWs<T> W; W.carve(ws, s, false);
  B2C_CHECK_ARG(ws_bytes >= W.bytes, "workspace too small: %zu < %zu", ws_bytes, W.bytes);
  PackTable tab; tab.n = 1;
  tab.seg[0] = PackSeg{p.w, W.Wp, nullptr, Es, Et, (long)Et, (long)Et, 0};
  pack_params_kernel<T><<<dim3(48, 1), 256, 0, st>>>(tab);
  B2C_LAUNCH_CHECK("pack_params_kernel");
  cast_f32_kernel<T, TZ><<<ew_grid(R * Et / 4), 256, 0, st>>>(x, W.xb, R * Et);
  B2C_LAUNCH_CHECK("cast_f32_kernel");
  B2C_TRY((gemm<T, T>(st, (int)R, Es, Et, W.xb, Et, 0, W.Wp, Et, 0, W.h, Es, 0.f, p.b, 1)));
  if (dr.p > 0.f) {
    dropout_inplace_kernel<T><<<ew_grid(R * Es), 256, 0, st>>>(W.h, R * Es, dr.p, dr.seed, 210u, (const unsigned long long*)dr.seed_dev);
    B2C_LAUNCH_CHECK("dropout_inplace_kernel");
  }
  {
    long grid = ((long)B * So + 7) / 8; if (grid > 148 * 8) grid = 148 * 8;
    if (Es <= 256) ln_pool_fwd_kernel<T, 1><<<(unsigned)grid, LN_THREADS, 0, st>>>(W.h, p.ln_w, p.ln_b, out, W.mean, W.rstd, B, St, So, Es, 1e-5f);
    else ln_pool_fwd_kernel<T, 2><<<(unsigned)grid, LN_THREADS, 0, st>>>(W.h, p.ln_w, p.ln_b, out, W.mean, W.rstd, B, St, So, Es, 1e-5f);
    B2C_LAUNCH_CHECK("ln_pool_fwd_kernel");
  }
  return 0;
}

template <typename T>
int projector_backward_impl(const B2CShape& s, const B2CProjParams& p, const float* dout, const B2CProjGrads& g, void* ws,
                            size_t ws_bytes, const B2CDropout& dr, cudaStream_t st) {
  if (p.w == nullptr) return 0;                     // identity projection: no parameters, teacher features carry no gradient
  B2C_CHECK_ARG(g.w && g.b && g.ln_w && g.ln_b, "NULL projector gradient");
  ProjWs<T> W; W.carve(ws, s, false);
  B2C_CHECK_ARG(ws_bytes >= W.bytes, "workspace too small: %zu < %zu", ws_bytes, W.bytes);
  const int B = s.B, St = s.S, Et = s.E, Es = s.H, So = s.T;
  const long R = (long)B * St;
  const float inv_keep = dr.p > 0.f ? 1.0f / (1.0f - dr.p) : 1.0f;
  // un-pool + LayerNorm backward in one pass (dy is rebuilt from the pooled gradient), then ReLU mask + bias gradient in one pass
  B2C_TRY((ln_bwd<T, T, T, T>(st, (const T*)nullptr, dout, St, So, W.h, (const T*)nullptr, W.mean, W.rstd, p.ln_w, W.dh, nullptr, W.lnpart,
                           g.ln_w, g.ln_b, nullptr, R, Es)));
  B2C_TRY(colsum_vec<T>(st, W.dh, W.h, R, Es, inv_keep, W.partial, g.b));
  B2C_TRY((gemm<T, float>(st, Es, Et, (int)R, W.dh, Es, 1, W.xb, Et, 1, g.w, Et)));
  return 0;
}

template <typename TS, typename TZ>         // TZ: the teacher logits' type (float, bf16 or f16)
int kd_token_loss_impl(const TS* y, const TZ* z, const int64_t* tgt, long N, int V, float temperature, float alpha,
                       float w_ce_eff, const int* n_valid, TS* dy, float* row_kl, float* row_ce, cudaStream_t st, int* argmax_out = nullptr,
                       long ld = 0 /* dy pitch; 0 = V */, const int* steps = nullptr, long rows_per_step = 0) {
  if (ld == 0) ld = V;
  const bool eval = (dy == nullptr) || (argmax_out != nullptr);      // losses only (+ predictions): the row-in-smem kernel
  const bool vec = (V % 8 == 0) && (ld == V) && ((uintptr_t)y % 16 == 0) && ((uintptr_t)z % 16 == 0) && ((uintptr_t)dy % 16 == 0);
  const bool t4 = (temperature == 4.0f);
  const size_t smem = align_up((size_t)V * 4, 16) + align_up((size_t)V * sizeof(TS), 16);
  const float inv_temp = 1.0f / temperature, kd_coef = alpha * temperature / (float)N;
  const float kd_num = alpha * temperature;        // with a device step count the kernels form kd_coef = kd_num / (*steps * rows_per_step)
  // default: persistent CTAs, TMA double-buffered row prefetch, register-resident math (V % 8 == 0, V <= 16384)
  const size_t psmem = 2 * ((size_t)V * sizeof(TZ) + (size_t)V * sizeof(TS));     // double-buffered row pair; larger rows take the row-in-smem kernel
  if (vec && V <= 8 * KDR_THREADS * 8 && !eval && psmem <= 200 * 1024) {
    const int need = cdiv(V / 8, KDR_THREADS);
    int per_sm = (int)((200 * 1024) / (psmem + 1024)); if (per_sm < 1) per_sm = 1;
    const int reg_cap = need <= 3 ? 3 : (need <= 5 ? 2 : 1);      // matches the kernel's __launch_bounds__ min-blocks
    if (per_sm > reg_cap) per_sm = reg_cap;
    long grid = (long)sm_count() * per_sm; if (grid > N) grid = N;
#define B2C_KDP(NCH, T4)                                                                                                   \
  do {                                                                                                                     \
    B2C_TRY(set_smem(kd_token_loss_pipe_kernel<TS, TZ, NCH, T4>, psmem));                                                  \
    kd_token_loss_pipe_kernel<TS, TZ, NCH, T4><<<(unsigned)grid, KDR_THREADS, psmem, st>>>(y, z, tgt, N, V, inv_temp, temperature, kd_coef, w_ce_eff, n_valid, dy, row_kl, row_ce, steps, rows_per_step, kd_num); \
  } while (0)
#define B2C_KDP2(NCH) do { if (t4) B2C_KDP(NCH, true); else B2C_KDP(NCH, false); } while (0)
    switch (need) {
      case 1: B2C_KDP2(1); break; case 2: B2C_KDP2(2); break; case 3: B2C_KDP2(3); break; case 4: B2C_KDP2(4); break;
      case 5: B2C_KDP2(5); break; case 6: B2C_KDP2(6); break; case 7: B2C_KDP2(7); break; default: B2C_KDP2(8); break;
    }
#undef B2C_KDP2
#undef B2C_KDP
    B2C_LAUNCH_CHECK("kd_token_loss_pipe_kernel");
    return 0;
  }
  // bf16 rows of any length / alignment with a 16-byte-aligned dy of pitch ld % 8 == 0: the same pipeline on the rows'
  // enclosing 16-byte ranges (slot = the ranges plus one word of read-ahead)
  const int Vp = (V + 7) & ~7;
  const size_t usmem = 2 * ((size_t)(Vp + 16 / sizeof(TZ)) * sizeof(TZ) + (size_t)(Vp + 8) * sizeof(TS));
  if constexpr (sizeof(TS) == 2) if (!vec && !eval && ld % 8 == 0 && ld >= Vp && (uintptr_t)dy % 16 == 0 && V <= 8 * KDR_THREADS * 8 && usmem <= 200 * 1024) {
    const int need = cdiv(Vp / 8, KDR_THREADS);
    int per_sm = (int)((200 * 1024) / (usmem + 1024)); if (per_sm < 1) per_sm = 1;
    const int reg_cap = need <= 3 ? 3 : (need <= 5 ? 2 : 1);
    if (per_sm > reg_cap) per_sm = reg_cap;
    long grid = (long)sm_count() * per_sm; if (grid > N) grid = N;
    const bf16* yb = reinterpret_cast<const bf16*>(y);
    bf16* dyb = reinterpret_cast<bf16*>(dy);
#define B2C_KDU(NCH, T4)                                                                                                   \
  do {                                                                                                                     \
    B2C_TRY(set_smem(kd_token_loss_pipe_unaligned_kernel<TZ, NCH, T4>, usmem));                                            \
    kd_token_loss_pipe_unaligned_kernel<TZ, NCH, T4><<<(unsigned)grid, KDR_THREADS, usmem, st>>>(yb, z, tgt, N, V, ld, inv_temp, temperature, kd_coef, w_ce_eff, n_valid, dyb, row_kl, row_ce, steps, rows_per_step, kd_num); \
  } while (0)
#define B2C_KDU2(NCH) do { if (t4) B2C_KDU(NCH, true); else B2C_KDU(NCH, false); } while (0)
    switch (need) {
      case 1: B2C_KDU2(1); break; case 2: B2C_KDU2(2); break; case 3: B2C_KDU2(3); break; case 4: B2C_KDU2(4); break;
      case 5: B2C_KDU2(5); break; case 6: B2C_KDU2(6); break; case 7: B2C_KDU2(7); break; default: B2C_KDU2(8); break;
    }
#undef B2C_KDU2
#undef B2C_KDU
    B2C_LAUNCH_CHECK("kd_token_loss_pipe_unaligned_kernel");
    return 0;
  }
  B2C_CHECK_ARG(ld == V, "dlogits pitch %ld != V=%d needs bf16, a 16-byte-aligned dlogits with pitch %% 8 == 0 and >= roundup(V, 8), and V <= 16384", ld, V);
#define B2C_KD_LAUNCH(G, T4)                                                                                             \
  do {                                                                                                                   \
    B2C_TRY(set_smem(kd_token_loss_kernel<TS, TZ, G, T4>, smem));                                                        \
    kd_token_loss_kernel<TS, TZ, G, T4><<<(unsigned)N, KD_THREADS, smem, st>>>(y, z, tgt, V, inv_temp, kd_coef, w_ce_eff, n_valid, dy, row_kl, row_ce, argmax_out, steps, rows_per_step, kd_num); \
  } while (0)
  if (vec && t4) B2C_KD_LAUNCH(8, true);
  else if (vec) B2C_KD_LAUNCH(8, false);
  else if (t4) B2C_KD_LAUNCH(1, true);
  else B2C_KD_LAUNCH(1, false);
#undef B2C_KD_LAUNCH
  B2C_LAUNCH_CHECK("kd_token_loss_kernel");
  return 0;
}

template <typename TF, typename TH, typename TZ>
int aux_loss_impl(const TF* fs, const float* ft, int B, int Ss, int St, int E, const TH* hs, const TZ* ht, int Tn, int Th, int H,
                  float beta, float gamma, float* dfs, float* dft, TH* dhs, float* feat_part, float* hid_part, cudaStream_t st,
                  const int* steps = nullptr) {
  const int nfb = fs ? B : 0;
  const long all_rows = hs ? (long)Tn * B : 0;
  const int hid_blocks = (int)((all_rows + 7) / 8);
  if (nfb + hid_blocks == 0) return 0;
  const size_t smem = fs ? (size_t)(2 * Ss + 2 * St + 2 * E + 8 * 2 * E + 8) * 4 : 0;       // + per-warp column partials [8][2][E]
  B2C_TRY(set_smem(aux_loss_kernel<TF, TH, TZ>, smem));
  aux_loss_kernel<TF, TH, TZ><<<nfb + hid_blocks, 256, smem, st>>>(fs, ft, nfb, B, Ss, St, E, hs, ht, (int)((long)Th * B), (int)all_rows, H, Th, beta, gamma,
                                                               dfs, dft, dhs, feat_part, hid_part, steps);
  B2C_LAUNCH_CHECK("aux_loss_kernel");
  return 0;
}

// Calls f with the teacher data `p` as a pointer to its element type: B2C_F32, B2C_BF16 or B2C_F16.
template <typename F>
int with_teacher(const void* p, int teacher_dtype, F&& f) {
  if (teacher_dtype == B2C_F32) return f(static_cast<const float*>(p));
  if (teacher_dtype == B2C_BF16) return f(static_cast<const bf16*>(p));
  if (teacher_dtype == B2C_F16) return f(static_cast<const f16*>(p));
  return set_err(B2C_EINVAL, "bad teacher dtype %d (B2C_F32, B2C_BF16 or B2C_F16)", teacher_dtype);
}

}  // namespace

// ====================================================================================== extern "C"
extern "C" {

int b2c_abi_version(void) { return B2C_ABI_VERSION; }
const char* b2c_last_error(void) { return err_buf(); }
uint64_t b2c_launch_count(void) { return (uint64_t)launch_counter(); }

size_t b2c_workspace_bytes(const B2CShape* shape, int dtype, int mode) {
  if (mode != B2C_WS_REFINE && mode != B2C_WS_PROJ && check_shape(shape) != 0) return 0;
  if (mode == B2C_WS_TRAIN) {
    if (dtype == B2C_F32) { TrainWs<float> w; w.carve(nullptr, *shape); return w.bytes; }
    if (dtype == B2C_BF16) { TrainWs<bf16> w; w.carve(nullptr, *shape); return w.bytes; }
  } else if (mode == B2C_WS_DECODE) {
    if (dtype == B2C_F32) { DecodeWs<float> w; w.carve(nullptr, *shape); return w.bytes; }
    if (dtype == B2C_BF16) { DecodeWs<bf16> w; w.carve(nullptr, *shape); return w.bytes; }
  } else if (mode == B2C_WS_REFINE) {
    if (check_refine_shape(shape) != 0) return 0;
    if (dtype == B2C_F32) { RefineWs<float> w; w.carve(nullptr, *shape); return w.bytes; }
    if (dtype == B2C_BF16) { RefineWs<bf16> w; w.carve(nullptr, *shape); return w.bytes; }
  } else if (mode == B2C_WS_PROJ) {
    if (check_proj_shape(shape) != 0) return 0;
    if (dtype == B2C_F32) { ProjWs<float> w; w.carve(nullptr, *shape, false); return w.bytes; }
    if (dtype == B2C_BF16) { ProjWs<bf16> w; w.carve(nullptr, *shape, false); return w.bytes; }
  } else if (mode == B2C_WS_ATTN) {
    if (dtype == B2C_F32) { AttnWs<float> w; w.carve(nullptr, *shape); return w.bytes; }
    if (dtype == B2C_BF16) { AttnWs<bf16> w; w.carve(nullptr, *shape); return w.bytes; }
  }
  set_err(B2C_EINVAL, "bad dtype %d / mode %d", dtype, mode);
  return 0;
}

static int decoder_forward_entry(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                                 void* logits, void* hidden_top, float* attn_w, void* workspace, size_t ws_bytes,
                                 int dtype, const B2CDropout* dropout, void* stream, bool prepared, const int32_t* steps = nullptr) {
  B2C_TRY(check_shape(shape)); B2C_TRY(check_device());
  B2C_CHECK_ARG(params && feats && captions && logits && hidden_top && attn_w && workspace, "NULL argument");
  const B2CDropout dr = dropout ? *dropout : B2CDropout{0.f, 0, nullptr};
  B2C_CHECK_ARG(dr.p >= 0.f && dr.p < 1.f, "dropout p=%f outside [0,1)", dr.p);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B2C_F32) return decoder_forward_impl<float>(*shape, *params, (const float*)feats, captions, (float*)logits, (float*)hidden_top, attn_w, workspace, ws_bytes, dr, st, prepared, nullptr, steps);
  if (dtype == B2C_BF16) return decoder_forward_impl<bf16>(*shape, *params, (const bf16*)feats, captions, (bf16*)logits, (bf16*)hidden_top, attn_w, workspace, ws_bytes, dr, st, prepared, nullptr, steps);
  return set_err(B2C_EINVAL, "bad dtype %d", dtype);
}
int b2c_decoder_forward(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                        void* logits, void* hidden_top, float* attn_w, void* workspace, size_t ws_bytes,
                        int dtype, const B2CDropout* dropout, void* stream) {
  return decoder_forward_entry(shape, params, feats, captions, logits, hidden_top, attn_w, workspace, ws_bytes, dtype, dropout, stream, false);
}
int b2c_decoder_forward_prepared(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                                 void* logits, void* hidden_top, float* attn_w, void* workspace, size_t ws_bytes,
                                 int dtype, const B2CDropout* dropout, void* stream) {
  return decoder_forward_entry(shape, params, feats, captions, logits, hidden_top, attn_w, workspace, ws_bytes, dtype, dropout, stream, true);
}
int b2c_decoder_forward_steps(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                              void* logits, void* hidden_top, float* attn_w, void* workspace, size_t ws_bytes,
                              int dtype, const B2CDropout* dropout, const int32_t* steps, void* stream) {
  return decoder_forward_entry(shape, params, feats, captions, logits, hidden_top, attn_w, workspace, ws_bytes, dtype, dropout, stream, false, steps);
}
int b2c_decoder_forward_prepared_steps(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                                       void* logits, void* hidden_top, float* attn_w, void* workspace, size_t ws_bytes,
                                       int dtype, const B2CDropout* dropout, const int32_t* steps, void* stream) {
  return decoder_forward_entry(shape, params, feats, captions, logits, hidden_top, attn_w, workspace, ws_bytes, dtype, dropout, stream, true, steps);
}
int b2c_decoder_forward_eval(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                             const float* teacher_logits, const int64_t* targets, float temperature,
                             void* hidden_top, float* attn_w, float* row_kl, float* row_ce, int32_t* argmax_out,
                             void* workspace, size_t ws_bytes, int dtype, void* stream) {
  return b2c_decoder_forward_eval_teacher(shape, params, feats, captions, teacher_logits, B2C_F32, targets, temperature, hidden_top, attn_w,
                                          row_kl, row_ce, argmax_out, workspace, ws_bytes, dtype, stream);
}
int b2c_decoder_forward_eval_teacher(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                                     const void* teacher_logits, int teacher_dtype, const int64_t* targets, float temperature,
                                     void* hidden_top, float* attn_w, float* row_kl, float* row_ce, int32_t* argmax_out,
                                     void* workspace, size_t ws_bytes, int dtype, void* stream) {
  B2C_TRY(check_shape(shape)); B2C_TRY(check_device());
  B2C_CHECK_ARG(params && feats && captions && teacher_logits && targets && hidden_top && attn_w && row_kl && row_ce && workspace, "NULL argument");
  B2C_CHECK_ARG(temperature > 0.f, "temperature %f", temperature);
  B2C_CHECK_ARG(dtype == B2C_BF16, "the logits-free validation forward is a bf16-mode path (fp32 parity mode keeps the logits)");
  B2C_CHECK_ARG(teacher_dtype == B2C_F32 || teacher_dtype == B2C_BF16 || teacher_dtype == B2C_F16,
                "bad teacher dtype %d (B2C_F32, B2C_BF16 or B2C_F16)", teacher_dtype);
  const B2CDropout dr{0.f, 0, nullptr};
  const EvalOut ev{teacher_logits, teacher_dtype, targets, temperature, row_kl, row_ce, argmax_out};
  return decoder_forward_impl<bf16>(*shape, *params, (const bf16*)feats, captions, (bf16*)nullptr, (bf16*)hidden_top, attn_w, workspace, ws_bytes, dr,
                                    (cudaStream_t)stream, false, &ev);
}

int b2c_decoder_prepare(const B2CShape* shape, const B2CParams* params, const int64_t* captions, void* workspace, size_t ws_bytes,
                        int dtype, void* stream) {
  B2C_TRY(check_shape(shape)); B2C_TRY(check_device());
  B2C_CHECK_ARG(params && captions && workspace, "NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B2C_F32) return decoder_prepare_impl<float>(*shape, *params, captions, workspace, ws_bytes, st);
  if (dtype == B2C_BF16) return decoder_prepare_impl<bf16>(*shape, *params, captions, workspace, ws_bytes, st);
  return set_err(B2C_EINVAL, "bad dtype %d", dtype);
}

int b2c_decoder_set_initial_state(const B2CShape* shape, const float* h0, const float* c0, void* workspace, size_t ws_bytes,
                                  int dtype, void* stream) {
  B2C_TRY(check_shape(shape)); B2C_TRY(check_device());
  B2C_CHECK_ARG(h0 && c0 && workspace, "NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B2C_F32) return set_initial_state_impl<float>(*shape, h0, c0, workspace, ws_bytes, st);
  if (dtype == B2C_BF16) return set_initial_state_impl<bf16>(*shape, h0, c0, workspace, ws_bytes, st);
  return set_err(B2C_EINVAL, "bad dtype %d", dtype);
}

int b2c_decoder_backward(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                         const void* hidden_top, const float* attn_w, const void* dlogits, const void* dhidden_top,
                         const B2CGrads* grads, float* dfeats, void* workspace, size_t ws_bytes,
                         int dtype, const B2CDropout* dropout, int flags, void* stream) {
  B2C_TRY(check_shape(shape)); B2C_TRY(check_device());
  B2C_CHECK_ARG(params && feats && captions && hidden_top && attn_w && dlogits && grads && workspace, "NULL argument");
  const B2CDropout dr = dropout ? *dropout : B2CDropout{0.f, 0, nullptr};
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B2C_F32) return decoder_backward_impl<float>(*shape, *params, (const float*)feats, captions, (const float*)hidden_top, attn_w, (const float*)dlogits, (const float*)dhidden_top, *grads, dfeats, workspace, ws_bytes, dr, st, flags);
  if (dtype == B2C_BF16) return decoder_backward_impl<bf16>(*shape, *params, (const bf16*)feats, captions, (const bf16*)hidden_top, attn_w, (const bf16*)dlogits, (const bf16*)dhidden_top, *grads, dfeats, workspace, ws_bytes, dr, st, flags);
  return set_err(B2C_EINVAL, "bad dtype %d", dtype);
}

int b2c_decoder_backward_pitched(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                                 const void* hidden_top, const float* attn_w, const void* dlogits, int64_t ld_dlogits, const void* dhidden_top,
                                 const B2CGrads* grads, float* dfeats, void* workspace, size_t ws_bytes,
                                 int dtype, const B2CDropout* dropout, int flags, void* stream) {
  B2C_TRY(check_shape(shape)); B2C_TRY(check_device());
  B2C_CHECK_ARG(params && feats && captions && hidden_top && attn_w && dlogits && grads && workspace, "NULL argument");
  B2C_CHECK_ARG(ld_dlogits >= shape->V, "ld_dlogits=%ld < V=%d", (long)ld_dlogits, shape->V);
  const B2CDropout dr = dropout ? *dropout : B2CDropout{0.f, 0, nullptr};
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B2C_F32) return decoder_backward_impl<float>(*shape, *params, (const float*)feats, captions, (const float*)hidden_top, attn_w, (const float*)dlogits, (const float*)dhidden_top, *grads, dfeats, workspace, ws_bytes, dr, st, flags, (long)ld_dlogits);
  if (dtype == B2C_BF16) return decoder_backward_impl<bf16>(*shape, *params, (const bf16*)feats, captions, (const bf16*)hidden_top, attn_w, (const bf16*)dlogits, (const bf16*)dhidden_top, *grads, dfeats, workspace, ws_bytes, dr, st, flags, (long)ld_dlogits);
  return set_err(B2C_EINVAL, "bad dtype %d", dtype);
}

int b2c_decoder_backward_steps(const B2CShape* shape, const B2CParams* params, const void* feats, const int64_t* captions,
                               const void* hidden_top, const float* attn_w, const void* dlogits, int64_t ld_dlogits, const void* dhidden_top,
                               const B2CGrads* grads, float* dfeats, void* workspace, size_t ws_bytes,
                               int dtype, const B2CDropout* dropout, int flags, const int32_t* steps, void* stream) {
  B2C_TRY(check_shape(shape)); B2C_TRY(check_device());
  B2C_CHECK_ARG(params && feats && captions && hidden_top && attn_w && dlogits && grads && workspace, "NULL argument");
  B2C_CHECK_ARG(ld_dlogits >= shape->V, "ld_dlogits=%ld < V=%d", (long)ld_dlogits, shape->V);
  const B2CDropout dr = dropout ? *dropout : B2CDropout{0.f, 0, nullptr};
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B2C_F32) return decoder_backward_impl<float>(*shape, *params, (const float*)feats, captions, (const float*)hidden_top, attn_w, (const float*)dlogits, (const float*)dhidden_top, *grads, dfeats, workspace, ws_bytes, dr, st, flags, (long)ld_dlogits, steps);
  if (dtype == B2C_BF16) return decoder_backward_impl<bf16>(*shape, *params, (const bf16*)feats, captions, (const bf16*)hidden_top, attn_w, (const bf16*)dlogits, (const bf16*)dhidden_top, *grads, dfeats, workspace, ws_bytes, dr, st, flags, (long)ld_dlogits, steps);
  return set_err(B2C_EINVAL, "bad dtype %d", dtype);
}

int b2c_debug_recur_trace(uint64_t* out_host, int64_t n, int32_t* grid_out, int32_t* steps_out) {
  RecurTrace& t = recur_trace_state();
  B2C_CHECK_ARG(t.dev != nullptr && out_host && n > 0, "no trace recorded (set B2C_RECUR_TRACE=1 before the first forward)");
  B2C_CUDA(cudaDeviceSynchronize());
  const size_t m = (size_t)n < t.n ? (size_t)n : t.n;
  B2C_CUDA(cudaMemcpy(out_host, t.dev, m * 8, cudaMemcpyDeviceToHost));
  if (grid_out) *grid_out = t.grid;
  if (steps_out) *steps_out = t.T;
  return 0;
}

int b2c_bump_counter(uint64_t* counter, void* stream) {
  B2C_TRY(check_device());
  B2C_CHECK_ARG(counter != nullptr, "NULL counter");
  bump_counter_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(reinterpret_cast<unsigned long long*>(counter));
  B2C_LAUNCH_CHECK("bump_counter_kernel");
  return 0;
}

int b2c_set_gemm_cta_limit(int32_t max_ctas) {
  B2C_CHECK_ARG(max_ctas >= 0, "max_ctas=%d must be >= 0", max_ctas);
  gemm_cta_cap() = max_ctas;
  return 0;
}

int b2c_join_side_work(void* stream) {
  B2C_TRY(check_device());
  SubStreams* hs = nullptr;
  B2C_TRY(get_substreams(&hs));
  B2C_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, hs->join[MAX_SUB - 1], 0));
  return 0;
}

int b2c_greedy_decode(const B2CShape* shape, const B2CParams* params, const void* feats, int64_t start_id, int64_t end_id,
                      int64_t* tokens, int32_t* lengths, void* workspace, size_t ws_bytes, int dtype, void* stream) {
  B2C_TRY(check_shape(shape)); B2C_TRY(check_device());
  B2C_CHECK_ARG(params && feats && tokens && lengths && workspace, "NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B2C_F32) return greedy_decode_impl<float>(*shape, *params, (const float*)feats, start_id, end_id, tokens, lengths, workspace, ws_bytes, st);
  if (dtype == B2C_BF16) return greedy_decode_impl<bf16>(*shape, *params, (const bf16*)feats, start_id, end_id, tokens, lengths, workspace, ws_bytes, st);
  return set_err(B2C_EINVAL, "bad dtype %d", dtype);
}

int b2c_attention_step(const B2CShape* shape, const float* attn_w, const float* attn_b, const void* hidden, const void* feats,
                       void* context, float* weights, void* workspace, size_t ws_bytes, int dtype, void* stream) {
  B2C_TRY(check_shape(shape)); B2C_TRY(check_device());
  B2C_CHECK_ARG(attn_w && attn_b && hidden && feats && context && weights && workspace, "NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B2C_F32) return attention_step_impl<float>(*shape, attn_w, attn_b, (const float*)hidden, (const float*)feats, (float*)context, weights, workspace, ws_bytes, st);
  if (dtype == B2C_BF16) return attention_step_impl<bf16>(*shape, attn_w, attn_b, (const bf16*)hidden, (const bf16*)feats, (bf16*)context, weights, workspace, ws_bytes, st);
  return set_err(B2C_EINVAL, "bad dtype %d", dtype);
}

int b2c_refinement_forward(const B2CShape* shape, const B2CRefineParams* params, const float* x, float* out,
                           void* workspace, size_t ws_bytes, int dtype, const B2CDropout* dropout, void* stream) {
  B2C_TRY(check_refine_shape(shape)); B2C_TRY(check_device());
  B2C_CHECK_ARG(params && x && out && workspace, "NULL argument");
  const B2CDropout dr = dropout ? *dropout : B2CDropout{0.f, 0, nullptr};
  B2C_CHECK_ARG(dr.p >= 0.f && dr.p < 1.f, "dropout p=%f outside [0,1)", dr.p);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B2C_F32) return refinement_forward_impl<float>(*shape, *params, x, out, workspace, ws_bytes, dr, st);
  if (dtype == B2C_BF16) return refinement_forward_impl<bf16>(*shape, *params, x, out, workspace, ws_bytes, dr, st);
  return set_err(B2C_EINVAL, "bad dtype %d", dtype);
}

int b2c_refinement_forward_dual(const B2CShape* shape, const B2CRefineParams* params, const float* x, float* out, void* out_compute,
                                void* workspace, size_t ws_bytes, int dtype, const B2CDropout* dropout, void* stream) {
  B2C_TRY(check_refine_shape(shape)); B2C_TRY(check_device());
  B2C_CHECK_ARG(params && x && out && workspace, "NULL argument");
  const B2CDropout dr = dropout ? *dropout : B2CDropout{0.f, 0, nullptr};
  B2C_CHECK_ARG(dr.p >= 0.f && dr.p < 1.f, "dropout p=%f outside [0,1)", dr.p);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B2C_F32) return refinement_forward_impl<float>(*shape, *params, x, out, workspace, ws_bytes, dr, st, (float*)nullptr);   // fp32: `out` is the compute copy
  if (dtype == B2C_BF16) return refinement_forward_impl<bf16>(*shape, *params, x, out, workspace, ws_bytes, dr, st, (bf16*)out_compute);
  return set_err(B2C_EINVAL, "bad dtype %d", dtype);
}

int b2c_refinement_backward(const B2CShape* shape, const B2CRefineParams* params, const float* x, const float* dout, const B2CRefineGrads* grads,
                            float* dx, void* workspace, size_t ws_bytes, int dtype, const B2CDropout* dropout, void* stream) {
  B2C_TRY(check_refine_shape(shape)); B2C_TRY(check_device());
  B2C_CHECK_ARG(params && x && dout && grads && dx && workspace, "NULL argument");
  const B2CDropout dr = dropout ? *dropout : B2CDropout{0.f, 0, nullptr};
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B2C_F32) return refinement_backward_impl<float>(*shape, *params, x, dout, *grads, dx, workspace, ws_bytes, dr, st);
  if (dtype == B2C_BF16) return refinement_backward_impl<bf16>(*shape, *params, x, dout, *grads, dx, workspace, ws_bytes, dr, st);
  return set_err(B2C_EINVAL, "bad dtype %d", dtype);
}

int b2c_projector_forward(const B2CShape* shape, const B2CProjParams* params, const float* x, float* out,
                          void* workspace, size_t ws_bytes, int dtype, const B2CDropout* dropout, void* stream) {
  return b2c_projector_forward_teacher(shape, params, x, B2C_F32, out, workspace, ws_bytes, dtype, dropout, stream);
}
int b2c_projector_forward_teacher(const B2CShape* shape, const B2CProjParams* params, const void* x, int teacher_dtype, float* out,
                                  void* workspace, size_t ws_bytes, int dtype, const B2CDropout* dropout, void* stream) {
  B2C_TRY(check_proj_shape(shape)); B2C_TRY(check_device());
  B2C_CHECK_ARG(params && x && out && workspace, "NULL argument");
  const B2CDropout dr = dropout ? *dropout : B2CDropout{0.f, 0, nullptr};
  B2C_CHECK_ARG(dr.p >= 0.f && dr.p < 1.f, "dropout p=%f outside [0,1)", dr.p);
  cudaStream_t st = (cudaStream_t)stream;
  return with_teacher(x, teacher_dtype, [&](auto xt) {
    if (dtype == B2C_F32) return projector_forward_impl<float>(*shape, *params, xt, out, workspace, ws_bytes, dr, st);
    if (dtype == B2C_BF16) return projector_forward_impl<bf16>(*shape, *params, xt, out, workspace, ws_bytes, dr, st);
    return set_err(B2C_EINVAL, "bad dtype %d", dtype);
  });
}

int b2c_projector_backward(const B2CShape* shape, const B2CProjParams* params, const float* dout, const B2CProjGrads* grads,
                           void* workspace, size_t ws_bytes, int dtype, const B2CDropout* dropout, void* stream) {
  B2C_TRY(check_proj_shape(shape)); B2C_TRY(check_device());
  B2C_CHECK_ARG(params && dout && grads && workspace, "NULL argument");
  const B2CDropout dr = dropout ? *dropout : B2CDropout{0.f, 0, nullptr};
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B2C_F32) return projector_backward_impl<float>(*shape, *params, dout, *grads, workspace, ws_bytes, dr, st);
  if (dtype == B2C_BF16) return projector_backward_impl<bf16>(*shape, *params, dout, *grads, workspace, ws_bytes, dr, st);
  return set_err(B2C_EINVAL, "bad dtype %d", dtype);
}

int b2c_count_valid(const int64_t* targets, int64_t n, int32_t V, int32_t* n_valid_out, void* stream) {
  B2C_TRY(check_device());
  B2C_CHECK_ARG(targets && n_valid_out && n > 0, "bad argument");
  count_valid_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(targets, (long)n, V, n_valid_out);
  B2C_LAUNCH_CHECK("count_valid_kernel");
  return 0;
}

int b2c_kd_token_loss(const void* student_logits, const float* teacher_logits, const int64_t* targets,
                      int64_t N, int32_t V, float temperature, float alpha, float w_ce, float ce_mult,
                      const int32_t* n_valid, void* dlogits, float* row_kl, float* row_ce, int dtype, void* stream) {
  return b2c_kd_token_loss_teacher(student_logits, teacher_logits, B2C_F32, targets, N, V, temperature, alpha, w_ce, ce_mult, n_valid,
                                   dlogits, V, row_kl, row_ce, dtype, nullptr, 0, stream);
}

int b2c_kd_token_loss_pitched(const void* student_logits, const float* teacher_logits, const int64_t* targets,
                              int64_t N, int32_t V, float temperature, float alpha, float w_ce, float ce_mult,
                              const int32_t* n_valid, void* dlogits, int64_t ld_dlogits, float* row_kl, float* row_ce, int dtype, void* stream) {
  return b2c_kd_token_loss_teacher(student_logits, teacher_logits, B2C_F32, targets, N, V, temperature, alpha, w_ce, ce_mult, n_valid,
                                   dlogits, ld_dlogits, row_kl, row_ce, dtype, nullptr, 0, stream);
}

int b2c_kd_token_loss_steps(const void* student_logits, const float* teacher_logits, const int64_t* targets,
                            int64_t N, int32_t V, float temperature, float alpha, float w_ce, float ce_mult,
                            const int32_t* n_valid, void* dlogits, int64_t ld_dlogits, float* row_kl, float* row_ce, int dtype,
                            const int32_t* steps, int64_t rows_per_step, void* stream) {
  return b2c_kd_token_loss_teacher(student_logits, teacher_logits, B2C_F32, targets, N, V, temperature, alpha, w_ce, ce_mult, n_valid,
                                   dlogits, ld_dlogits, row_kl, row_ce, dtype, steps, rows_per_step, stream);
}

int b2c_kd_token_loss_teacher(const void* student_logits, const void* teacher_logits, int teacher_dtype, const int64_t* targets,
                              int64_t N, int32_t V, float temperature, float alpha, float w_ce, float ce_mult,
                              const int32_t* n_valid, void* dlogits, int64_t ld_dlogits, float* row_kl, float* row_ce, int dtype,
                              const int32_t* steps, int64_t rows_per_step, void* stream) {
  B2C_TRY(check_device());
  B2C_CHECK_ARG(student_logits && teacher_logits && targets && n_valid && dlogits && row_kl && row_ce, "NULL argument");
  B2C_CHECK_ARG(N > 0 && N < 2147483647L && V > 1 && temperature > 0.f, "bad N=%ld V=%d temperature=%f", (long)N, V, temperature);
  B2C_CHECK_ARG(ld_dlogits >= V, "ld_dlogits=%ld < V=%d", (long)ld_dlogits, V);
  B2C_CHECK_ARG(steps == nullptr || (rows_per_step > 0 && N % rows_per_step == 0), "rows_per_step=%ld must divide N=%ld", (long)rows_per_step, (long)N);
  cudaStream_t st = (cudaStream_t)stream;
  return with_teacher(teacher_logits, teacher_dtype, [&](auto z) {
    if (dtype == B2C_F32) return kd_token_loss_impl<float>((const float*)student_logits, z, targets, (long)N, V, temperature, alpha, w_ce * ce_mult, n_valid, (float*)dlogits, row_kl, row_ce, st, nullptr, (long)ld_dlogits, steps, (long)rows_per_step);
    if (dtype == B2C_BF16) return kd_token_loss_impl<bf16>((const bf16*)student_logits, z, targets, (long)N, V, temperature, alpha, w_ce * ce_mult, n_valid, (bf16*)dlogits, row_kl, row_ce, st, nullptr, (long)ld_dlogits, steps, (long)rows_per_step);
    return set_err(B2C_EINVAL, "bad dtype %d", dtype);
  });
}

int b2c_kd_token_eval(const void* student_logits, const float* teacher_logits, const int64_t* targets, int64_t N, int32_t V,
                      float temperature, const int32_t* n_valid, float* row_kl, float* row_ce, int32_t* argmax_out, int dtype, void* stream) {
  return b2c_kd_token_eval_teacher(student_logits, teacher_logits, B2C_F32, targets, N, V, temperature, n_valid, row_kl, row_ce, argmax_out,
                                   dtype, stream);
}

int b2c_kd_token_eval_teacher(const void* student_logits, const void* teacher_logits, int teacher_dtype, const int64_t* targets, int64_t N,
                              int32_t V, float temperature, const int32_t* n_valid, float* row_kl, float* row_ce, int32_t* argmax_out,
                              int dtype, void* stream) {
  B2C_TRY(check_device());
  B2C_CHECK_ARG(student_logits && teacher_logits && targets && n_valid && row_kl && row_ce, "NULL argument");
  B2C_CHECK_ARG(N > 0 && N < 2147483647L && V > 1 && temperature > 0.f, "bad N=%ld V=%d temperature=%f", (long)N, V, temperature);
  cudaStream_t st = (cudaStream_t)stream;
  return with_teacher(teacher_logits, teacher_dtype, [&](auto z) {
    if (dtype == B2C_F32) return kd_token_loss_impl<float>((const float*)student_logits, z, targets, (long)N, V, temperature, 0.f, 0.f, n_valid, (float*)nullptr, row_kl, row_ce, st, argmax_out);
    if (dtype == B2C_BF16) return kd_token_loss_impl<bf16>((const bf16*)student_logits, z, targets, (long)N, V, temperature, 0.f, 0.f, n_valid, (bf16*)nullptr, row_kl, row_ce, st, argmax_out);
    return set_err(B2C_EINVAL, "bad dtype %d", dtype);
  });
}

int b2c_bleu1(const int32_t* predicted, const int64_t* targets, int32_t T, int32_t B, float* bleu_out, void* stream) {
  B2C_TRY(check_device());
  B2C_CHECK_ARG(predicted && targets && bleu_out && T > 0 && B > 0, "bad argument");
  bleu1_kernel<<<cdiv(B, 4), 128, 0, (cudaStream_t)stream>>>(predicted, targets, T, B, bleu_out);
  B2C_LAUNCH_CHECK("bleu1_kernel");
  return 0;
}

int b2c_aux_loss(const void* feats_s, const float* feats_t, int32_t B, int32_t Ss, int32_t St, int32_t E,
                 const void* hid_s, const float* hid_t, int32_t T, int32_t Th, int32_t H,
                 float beta, float gamma, float* dfeats_s, float* dfeats_t, void* dhid_s,
                 float* feat_part, float* hid_part, int dtype, int feat_dtype, void* stream) {
  return b2c_aux_loss_teacher(feats_s, feats_t, B, Ss, St, E, hid_s, hid_t, B2C_F32, T, Th, H, beta, gamma, dfeats_s, dfeats_t, dhid_s,
                              feat_part, hid_part, dtype, feat_dtype, nullptr, stream);
}

int b2c_aux_loss_steps(const void* feats_s, const float* feats_t, int32_t B, int32_t Ss, int32_t St, int32_t E,
                       const void* hid_s, const float* hid_t, int32_t T, int32_t Th, int32_t H,
                       float beta, float gamma, float* dfeats_s, float* dfeats_t, void* dhid_s,
                       float* feat_part, float* hid_part, int dtype, int feat_dtype, const int32_t* steps, void* stream) {
  return b2c_aux_loss_teacher(feats_s, feats_t, B, Ss, St, E, hid_s, hid_t, B2C_F32, T, Th, H, beta, gamma, dfeats_s, dfeats_t, dhid_s,
                              feat_part, hid_part, dtype, feat_dtype, steps, stream);
}

int b2c_aux_loss_teacher(const void* feats_s, const float* feats_t, int32_t B, int32_t Ss, int32_t St, int32_t E,
                         const void* hid_s, const void* hid_t, int hid_t_dtype, int32_t T, int32_t Th, int32_t H,
                         float beta, float gamma, float* dfeats_s, float* dfeats_t, void* dhid_s,
                         float* feat_part, float* hid_part, int dtype, int feat_dtype, const int32_t* steps, void* stream) {
  B2C_TRY(check_device());
  B2C_CHECK_ARG(B > 0, "B=%d", B);
  if (feats_s) B2C_CHECK_ARG(feats_t && feat_part && Ss > 0 && St > 0 && E > 0 && E % 8 == 0, "feature KD needs feats_t, feat_part, positive Ss/St and E a positive multiple of 8 (E=%d)", E);
  if (hid_s) B2C_CHECK_ARG(hid_t && hid_part && T > 0 && Th > 0 && Th <= T && H > 0 && H % 8 == 0, "hidden KD needs hid_t, hid_part, 0 < Th <= T and H a positive multiple of 8 (H=%d)", H);
  cudaStream_t st = (cudaStream_t)stream;
  return with_teacher(hid_t, hid_t_dtype, [&](auto ht) {
    if (dtype == B2C_F32 && feat_dtype == B2C_F32) return aux_loss_impl<float, float>((const float*)feats_s, feats_t, B, Ss, St, E, (const float*)hid_s, ht, T, Th, H, beta, gamma, dfeats_s, dfeats_t, (float*)dhid_s, feat_part, hid_part, st, steps);
    if (dtype == B2C_BF16 && feat_dtype == B2C_BF16) return aux_loss_impl<bf16, bf16>((const bf16*)feats_s, feats_t, B, Ss, St, E, (const bf16*)hid_s, ht, T, Th, H, beta, gamma, dfeats_s, dfeats_t, (bf16*)dhid_s, feat_part, hid_part, st, steps);
    if (dtype == B2C_BF16 && feat_dtype == B2C_F32) return aux_loss_impl<float, bf16>((const float*)feats_s, feats_t, B, Ss, St, E, (const bf16*)hid_s, ht, T, Th, H, beta, gamma, dfeats_s, dfeats_t, (bf16*)dhid_s, feat_part, hid_part, st, steps);
    return set_err(B2C_EINVAL, "bad dtype %d / feature dtype %d", dtype, feat_dtype);
  });
}

int b2c_loss_finalize(const float* row_kl, const float* row_ce, int64_t N, const int32_t* n_valid, float ce_mult,
                      const float* feat_part, int32_t B, int32_t E, const float* hid_part, int32_t Th, int32_t H,
                      float temperature, float alpha, float beta, float gamma, float w_ce, float* out5, void* stream) {
  B2C_TRY(check_device());
  B2C_CHECK_ARG(row_kl && row_ce && n_valid && out5 && N > 0 && B > 0, "bad argument");
  loss_finalize_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(row_kl, row_ce, (long)N, n_valid, feat_part, B, E, feat_part ? 1 : 0,
                                                            hid_part, (long)Th * B, H, Th, hid_part ? 1 : 0,
                                                            temperature, alpha, beta, gamma, w_ce, ce_mult, out5, (const int*)nullptr);
  B2C_LAUNCH_CHECK("loss_finalize_kernel");
  return 0;
}

int b2c_loss_finalize_steps(const float* row_kl, const float* row_ce, int64_t N, const int32_t* n_valid, float ce_mult,
                            const float* feat_part, int32_t B, int32_t E, const float* hid_part, int32_t Th, int32_t H,
                            float temperature, float alpha, float beta, float gamma, float w_ce, float* out5, const int32_t* steps, void* stream) {
  B2C_TRY(check_device());
  B2C_CHECK_ARG(row_kl && row_ce && n_valid && out5 && N > 0 && B > 0, "bad argument");
  loss_finalize_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(row_kl, row_ce, (long)N, n_valid, feat_part, B, E, feat_part ? 1 : 0,
                                                            hid_part, (long)Th * B, H, Th, hid_part ? 1 : 0,
                                                            temperature, alpha, beta, gamma, w_ce, ce_mult, out5, steps);
  B2C_LAUNCH_CHECK("loss_finalize_kernel");
  return 0;
}

int b2c_scale_inplace(void* p, int64_t n, int dtype, const float* scale, void* stream) {
  B2C_TRY(check_device());
  B2C_CHECK_ARG(p && scale && n >= 0, "bad argument");
  if (n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == B2C_F32) scale_inplace_kernel<float><<<ew_grid(n), 256, 0, st>>>((float*)p, (long)n, scale);
  else if (dtype == B2C_BF16) scale_inplace_kernel<bf16><<<ew_grid(n), 256, 0, st>>>((bf16*)p, (long)n, scale);
  else return set_err(B2C_EINVAL, "bad dtype %d", dtype);
  B2C_LAUNCH_CHECK("scale_inplace_kernel");
  return 0;
}

int b2c_optimizer_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                       const B2COptSegment* segments_host, int32_t n_segments, const B2COptHyper* hyper_host,
                       const float* lr, int32_t n_lr, int32_t* step, float* loss_scale, int32_t* growth_tracker,
                       float* stats, void* scratch, void* stream) {
  B2C_TRY(check_device());
  B2C_CHECK_ARG(param && grad && exp_avg && exp_avg_sq && segments_host && hyper_host && lr && step && stats && scratch, "null argument");
  B2C_CHECK_ARG(n_segments >= 1 && n_segments <= B2C_OPT_MAX_SEG, "n_segments %d outside 1..%d", n_segments, B2C_OPT_MAX_SEG);
  B2C_CHECK_ARG(((uintptr_t)param | (uintptr_t)grad | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) % 16 == 0, "flat buffers must be 16-byte aligned");
  B2C_CHECK_ARG(hyper_host->beta1 >= 0. && hyper_host->beta1 < 1. && hyper_host->beta2 >= 0. && hyper_host->beta2 < 1. && hyper_host->eps >= 0.,
                "bad AdamW hyper-parameters");
  B2C_CHECK_ARG(hyper_host->grad_scale > 0.f, "grad_scale must be positive (1 when unused)");
  OptSegs segs; memset(&segs, 0, sizeof(segs));
  segs.nseg = n_segments;
  for (int i = 0; i < n_segments; ++i) {
    const B2COptSegment& s = segments_host[i];
    B2C_CHECK_ARG(s.begin >= 0 && s.end >= s.begin && (s.begin & 3) == 0, "segment %d: bad range [%lld, %lld)", i, (long long)s.begin, (long long)s.end);
    B2C_CHECK_ARG(s.lr_index >= 0 && s.lr_index < n_lr, "segment %d: lr_index %d outside 0..%d", i, s.lr_index, n_lr - 1);
    B2C_CHECK_ARG(s.clip_group >= -1 && s.clip_group < B2C_OPT_MAX_CLIP, "segment %d: clip_group %d", i, s.clip_group);
    segs.begin[i] = (long)s.begin; segs.end[i] = (long)s.end; segs.lr_index[i] = s.lr_index; segs.clip_group[i] = s.clip_group;
    segs.weight_decay[i] = s.weight_decay;
  }
  OptHyper hp{hyper_host->beta1, hyper_host->beta2, (float)hyper_host->beta2, (float)(1.0 - hyper_host->beta1), (float)(1.0 - hyper_host->beta2),
              (float)hyper_host->eps, hyper_host->max_norm, hyper_host->grad_scale, hyper_host->growth_factor, hyper_host->backoff_factor, hyper_host->growth_interval};
  cudaStream_t st = (cudaStream_t)stream;
  const int nblk = 4 * sm_count();
  static_assert(16 + 4 * 160 * 4 * OPT_NPART <= B2C_OPT_SCRATCH_BYTES, "scratch too small for the partials");
  B2C_CHECK_ARG(nblk <= 4 * 160, "unexpected SM count");
  unsigned int* ticket = reinterpret_cast<unsigned int*>(scratch);
  float* partials = reinterpret_cast<float*>(reinterpret_cast<char*>(scratch) + 16);
  grad_sqnorm_kernel<<<nblk, OPT_THREADS, 0, st>>>(grad, segs, partials);
  B2C_LAUNCH_CHECK("grad_sqnorm_kernel");
  clip_adamw_kernel<<<nblk, OPT_THREADS, 0, st>>>(param, grad, exp_avg, exp_avg_sq, segs, hp, lr, step, loss_scale, growth_tracker,
                                                  partials, nblk, stats, ticket);
  B2C_LAUNCH_CHECK("clip_adamw_kernel");
  return 0;
}

int b2c_gemm(int32_t M, int32_t N, int32_t K, float alpha, const void* A, int64_t lda, int a_mn,
             const void* B, int64_t ldb, int b_mn, float beta, void* C, int64_t ldc, const float* bias, int relu,
             int dtype, int c_dtype, int impl, void* stream) {
  B2C_TRY(check_device());
  B2C_CHECK_ARG(M > 0 && N > 0 && K > 0 && A && B && C, "bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  GemmArgs g{M, N, K, alpha, beta, A, (long)lda, a_mn, B, (long)ldb, b_mn, C, (long)ldc, bias, relu};
  if (dtype == B2C_F32) {
    B2C_CHECK_ARG(c_dtype == B2C_F32, "fp32 operands produce fp32 output");
    return gemm_simt<float, float, float>(g, st);
  }
  if (dtype == B2C_BF16) {
    if (impl == 1) return c_dtype == B2C_F32 ? gemm_simt<bf16, bf16, float>(g, st) : gemm_simt<bf16, bf16, bf16>(g, st);
    return c_dtype == B2C_F32 ? Gemm<bf16, float>::run(g, st) : Gemm<bf16, bf16>::run(g, st);
  }
  return set_err(B2C_EINVAL, "bad dtype %d", dtype);
}

}  // extern "C"
