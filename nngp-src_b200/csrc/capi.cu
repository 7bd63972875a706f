// capi.cu -- host side of the C ABI declared in include/nngp_b200.h.
//
// Everything here is orchestration: device buffers, TMA tensor maps, the blocked Cholesky /
// triangular-solve schedules, and per-stage CUDA-event accounting.  All arithmetic runs in the
// sm_100a kernels of gemm_nt.cuh (DMMA + TMA) and dense_kernels.cuh.  There is no CPU path.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <chrono>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#include "../../include/nngp_b200.h"
#include "dense_kernels.cuh"
#include "gemm_nt.cuh"
#include "trsm_fused.cuh"
#include "potrf_panel.cuh"
#include "active_kernels.cuh"
#include "sliced_gemm.cuh"

using namespace nngp;

namespace {

thread_local std::string g_create_error;


typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  template <class T>
  T* as() const { return static_cast<T*>(p); }
};

// Device time between two events recorded on `s`, added to *dst when the call settles (end_call).  A span without an
// end or a destination is an event that only orders streams inside the call.
struct Span {
  cudaEvent_t a, b;
  cudaStream_t s;
  double* dst;
};

inline int64_t round_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

}  // namespace

struct nngp_handle {
  nngp_config cfg;
  double lsw2[NNGP_MAX_LAYERS], lsb2[NNGP_MAX_LAYERS];   // sigma_w^2 / sigma_b^2 of Dense layer l (uniform: all alike)
  ActCoef act{};         // activation of every hidden step (make_act_coef)
  double q_limit = 0.0;  // layer-0 diagonals must stay below this (row_sqnorm_kernel's range flag)
  int device = 0;
  // cfg.n_gpus > 1: replicas of the fitted state on the other GPUs (each a complete single-GPU handle with its own
  // streams and workspace; nngp_predict runs them on one host thread each).  `owner` is set on a replica.
  std::vector<nngp_handle*> peers;
  nngp_handle* owner = nullptr;
  int sm_count = 148;
  cudaStream_t stream = nullptr;        // main stream (all stage timing events live here)
  cudaStream_t panel_stream = nullptr;  // high-priority stream: Cholesky panel look-ahead
  cudaStream_t cur = nullptr;           // stream the launch helpers currently target
  cudaStream_t copy_stream = nullptr;   // H2D of test-row chunks, running ahead of the Gram launches (nngp_predict)
  PFN_encodeTiled encode = nullptr;
  std::string err;

  // fitted state
  bool fitted = false;
  int64_t N = 0, D = 0, ldx = 0, ldl = 0;
  double lambda = 0.0;
  double lml_terms[2] = {0.0, 0.0};  // {sum log diag(L), y^T (K+lambda I)^-1 y}; valid after nngp_fit
  bool have_labels = false;   // fitted from labels on this handle (nngp_fit / nngp_append_fit): y, z and lml_terms are valid
  bool have_M = false;   // NTK mode: M = L^-1 K_dd L^-T is present (nngp_fit or nngp_set_state_ntk_m)
  DevBuf X, q, L, alpha;
  DevBuf Linv;    // inv(L_JJ) of every 64 x 64 diagonal block of L (trtri_diag_kernel), operand of the solves' diagonal step
  DevBuf y;       // raw labels of the last nngp_fit (kept for nngp_append_fit)
  DevBuf app_x, app_y;  // nngp_append_fit staging: [X; X_new], [y; y_new]
  DevBuf panel_sync;   // fused panel kernel: {item counter, progress[row tiles], inv_ready[column blocks]}
  DevBuf panel_inv;  // scratch inverses of a factorisation that is not the handle's own factor (Schur block, nngp_diag_potrf)
  DevBuf zkeep;   // z = L^-1 y of the last fit (the backward substitution destroys its copy in the factor buffer)
  DevBuf Linvfull;  // latency mode: the explicit inverse factor L^-1 (N x N, lower, row-major, ld = ldl)
  bool have_inv = false;
  // cfg.variance_slices: int8 digit planes of L^-1 ([s][wq_rb][wq_ldq]) + 2^(e-6) of its rows; planes of the current
  // K_* row block, their row exponents, and the per-CTA running-sum tiles of sliced_gemm_kernel
  DevBuf Wq, wexp, Aq, aexp, slscratch, slsync;
  bool have_wq = false;
  int64_t wq_ldq = 0, wq_rb = 0;
  DevBuf L2;      // second factor buffer: target of the incremental (fixed-lambda) append, then swapped with L
  bool importing = false;   // between nngp_state_import_begin and _end
  DevBuf flags;   // int[2]: {potrf info, non-finite input}
  DevBuf lam_d;   // double[4]: {lambda, sum log diag L, z^T z, spare}

  // predict workspace
  DevBuf xt, qt, kss, blk, mean_d, var_d, ssq, sync_ints;
  // NTK mode: M = L^-1 K_dd L^-T (N x N), scratch for building it, second row block, cross / partial terms
  DevBuf Mmat, Kdd, blk2, cross, partial, mean_partial;
  // nngp_predict_cov: the T x T posterior covariance, and P = -V M ('ntk')
  DevBuf cov, covP;
  // nngp_kernel workspace
  DevBuf ka, kb, kqa, kqb, kout;
  DevBuf qtab;    // Erf, depth > 2: the per-row diagonal tables of the operands of the current Gram launch (run_gram)
  DevBuf stage;   // nngp_state_pack / _unpack with host memory on the other side: one range at a time
  // nngp_active_select workspace
  DevBuf sel_mean, sel_var, sel_score, sel_key, sel_state, sel_okey, sel_oidx, sel_max;

  std::map<std::tuple<const void*, uint64_t, uint64_t, uint64_t, uint32_t>, CUtensorMap> tmaps;

  nngp_stats_t st;
  std::vector<Span> spans;   // of the current call: settled by end_call, or discarded by the next begin_call
  std::vector<cudaEvent_t> ev_pool;
  std::vector<cudaEvent_t> rep_events;   // no-timing events of replicate_state (recorded on this handle's copy stream)
};

namespace {

int fail(nngp_handle* h, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (h) h->err = buf; else g_create_error = buf;
  return code;
}

#define CK(expr)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (expr);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(h, e_ == cudaErrorMemoryAllocation ? NNGP_ENOMEM : NNGP_ECUDA, "%s failed: %s (%s:%d)", #expr, \
                  cudaGetErrorString(e_), __FILE__, __LINE__);                                     \
  } while (0)

#define CKR(expr)                     \
  do {                                \
    int r_ = (expr);                  \
    if (r_ != NNGP_OK) return r_;     \
  } while (0)

int ensure(nngp_handle* h, DevBuf& b, size_t bytes) {
  if (bytes <= b.cap && b.p) return NNGP_OK;
  const bool regrow = b.p != nullptr;
  if (b.p) {  // every stream of the handle may still touch the old buffer (uploads run ahead on copy_stream)
    CK(cudaStreamSynchronize(h->stream));
    if (h->copy_stream) CK(cudaStreamSynchronize(h->copy_stream));
    if (h->panel_stream) CK(cudaStreamSynchronize(h->panel_stream));
    CK(cudaFree(b.p)); b.p = nullptr; b.cap = 0;
  }
  if (bytes == 0) bytes = 256;
  // A buffer that grows again (the active-learning loop: N += budget every round) gets 25 % head-room, so that
  // multi-GB cudaFree / cudaMalloc pairs do not recur every round; exact size if that does not fit.
  if (regrow && bytes >= (64u << 20)) {
    const size_t roomy = bytes + bytes / 4;
    if (cudaMalloc(&b.p, roomy) == cudaSuccess) { b.cap = roomy; h->st.device_allocs++; return NNGP_OK; }
    b.p = nullptr;
    cudaGetLastError();
  }
  cudaError_t e = cudaMalloc(&b.p, bytes);
  if (e != cudaSuccess) {
    b.p = nullptr;
    cudaGetLastError();
    return fail(h, NNGP_ENOMEM, "cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
  }
  b.cap = bytes;
  h->st.device_allocs++;
  return NNGP_OK;
}

void release(DevBuf& b) {
  if (b.p) cudaFree(b.p);
  b.p = nullptr;
  b.cap = 0;
}

bool is_device_ptr(const void* p) {
  cudaPointerAttributes at;
  cudaError_t e = cudaPointerGetAttributes(&at, p);
  if (e != cudaSuccess) { cudaGetLastError(); return false; }
  return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

// ---- events and stage timing ------------------------------------------------------------------
cudaEvent_t get_event(nngp_handle* h) {
  if (!h->ev_pool.empty()) { cudaEvent_t e = h->ev_pool.back(); h->ev_pool.pop_back(); return e; }
  cudaEvent_t e;
  cudaEventCreate(&e);
  return e;
}

// Opens a span on stream s that adds into *dst, if cfg.stats_level >= level.  Returns its index, or -1 (no span).
int span_open(nngp_handle* h, int level, cudaStream_t s, double* dst) {
  if (h->cfg.stats_level < level) return -1;
  const cudaEvent_t a = get_event(h);
  cudaEventRecord(a, s);
  h->spans.push_back({a, nullptr, s, dst});
  return (int)h->spans.size() - 1;
}

void span_close(nngp_handle* h, int i) {
  if (i < 0) return;
  Span& sp = h->spans[(size_t)i];
  sp.b = get_event(h);
  cudaEventRecord(sp.b, sp.s);
}

// An event that orders two streams inside the current call; it goes back to the pool with the call's spans.
cudaEvent_t call_event(nngp_handle* h) {
  const cudaEvent_t e = get_event(h);
  h->spans.push_back({e, nullptr, nullptr, nullptr});
  return e;
}

// After the call's synchronisation: add every closed span's time to its destination (`add`) and return all events
// to the pool.  A span whose end event has not completed adds nothing; only the predict upload's can be pending, on
// copy_stream, which the main stream waits for chunk by chunk but not to the span's end.
void settle_spans(nngp_handle* h, bool add = true) {
  for (const Span& sp : h->spans) {
    float ms = 0.f;
    if (add && sp.b && cudaEventElapsedTime(&ms, sp.a, sp.b) == cudaSuccess) *sp.dst += ms;
    h->ev_pool.push_back(sp.a);
    if (sp.b) h->ev_pool.push_back(sp.b);
  }
  h->spans.clear();
}

void discard_spans(nngp_handle* h) { settle_spans(h, false); }

// ---- tensor maps ------------------------------------------------------------------------------
// Row-major FP64 matrix [rows, cols] with leading dimension ld (elements); box = 16 x box_rows,
// SWIZZLE_128B (the layout gemm_nt_kernel's fragment loads assume).
int get_tmap(nngp_handle* h, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
             CUtensorMap* out) {
  auto key = std::make_tuple(base, rows, cols, ld, box_rows);
  auto it = h->tmaps.find(key);
  if (it != h->tmaps.end()) { *out = it->second; return NNGP_OK; }
  if ((reinterpret_cast<uintptr_t>(base) & 15) || (ld & 1))
    return fail(h, NNGP_EINVAL, "internal: TMA operand not 16-byte aligned (ld=%llu)", (unsigned long long)ld);
  CUtensorMap tm;
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {ld * sizeof(double)};
  cuuint32_t box[2] = {(cuuint32_t)GEMM_BK, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = h->encode(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(h, NNGP_ECUDA, "cuTensorMapEncodeTiled failed (CUresult %d; rows=%llu cols=%llu ld=%llu)", (int)r,
                (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld);
  if (h->tmaps.size() > 4096) h->tmaps.clear();
  h->tmaps[key] = tm;
  *out = tm;
  return NNGP_OK;
}

struct MatView {  // a whole device matrix a tensor map is built over
  const double* base;
  int64_t rows, cols, ld;
};

// ---- GEMM launches ----------------------------------------------------------------------------
template <int EPI, int ACT = ACT_RELU>
int launch_gemm(nngp_handle* h, const MatView& A, int a_row0, int a_col0, const MatView& B, int b_row0, int b_col0,
                GemmParams p, int grid_z = 1) {
  if (p.M <= 0 || p.N <= 0) return NNGP_OK;
  CUtensorMap tmA, tmB;
  CKR(get_tmap(h, A.base, A.rows, A.cols, A.ld, GEMM_BM, &tmA));
  CKR(get_tmap(h, B.base, B.rows, B.cols, B.ld, GEMM_BN, &tmB));
  p.a_row0 = a_row0; p.a_col0 = a_col0; p.b_row0 = b_row0; p.b_col0 = b_col0;
  dim3 grid((p.N + GEMM_BN - 1) / GEMM_BN, (p.M + GEMM_BM - 1) / GEMM_BM, grid_z);
  if (grid.y > 65535) return fail(h, NNGP_EINVAL, "internal: GEMM row range too large (%d rows)", p.M);
  // (ROWDOT counts as a GEMM-class launch)
  const int span = span_open(h, 2, h->cur, EPI == EPI_GRAM ? &h->st.gram_ms : &h->st.gemm_ms);
  gemm_nt_kernel<EPI, ACT><<<grid, GEMM_THREADS, GEMM_SMEM_BYTES, h->cur>>>(tmA, tmB, p);
  span_close(h, span);
  CK(cudaGetLastError());
  h->st.kernel_launches++;
  // algorithmic work: half the product for a lower-triangular range or a triangular B; the Gram's inner extent is the
  // true D (A's width), the other products count their K extent
  const double frac = p.lower || p.tri_k ? 0.5 : 1.0;
  const double k = EPI == EPI_GRAM ? (double)A.cols : (double)p.ktiles * GEMM_BK;
  const double flops = 2.0 * (double)p.M * (double)p.N * k * frac;
  if (EPI == EPI_GRAM) {
    h->st.gram_launches++;
    h->st.gram_flops += flops;
    h->st.gram_evals += (double)p.M * (double)p.N * frac * p.steps;
  } else {
    h->st.gemm_launches++;
    h->st.gemm_flops += flops;
  }
  return NNGP_OK;
}

// sigma_w^2 / sigma_b^2 of the Dense layer that follows activation step s
LayerSig layer_sig(const nngp_handle* h) {
  LayerSig sig;
  for (int i = 0; i < 16; ++i) { sig.sw2[i] = h->lsw2[std::min(i + 1, NNGP_MAX_LAYERS - 1)]; sig.sb2[i] = h->lsb2[std::min(i + 1, NNGP_MAX_LAYERS - 1)]; }
  return sig;
}

size_t act_table_bytes(const nngp_handle* h, int64_t rows);   // (device buffer sizes, below)

// K(A rows, B rows) -> out (M x N, ld ldo).  A: M x D (lda), B: N x D (ldb); qa/qb layer-0 diagonals.
// In NTK mode (cfg.kernel_type == 1) `out` receives Theta and `out2` (optional) the NNGP kernel K -- unless
// `nngp_only`: then `out` receives K in either mode.
int run_gram(nngp_handle* h, const double* A, int64_t lda, int64_t M, const double* qa, const double* B, int64_t ldb,
             int64_t N, const double* qb, int64_t D, double* out, int64_t ldo, int lower, double* out2 = nullptr,
             const double* alpha = nullptr, double* mean_partial = nullptr, bool nngp_only = false) {
  GemmParams p{};
  p.act = h->act;
  p.alpha = alpha; p.mean_partial = mean_partial;
  p.ntk = h->cfg.kernel_type == 1 && !nngp_only ? 1 : 0;
  p.C2 = out2;
  p.M = (int)M; p.N = (int)N;
  p.ktiles = (int)((D + GEMM_BK - 1) / GEMM_BK);
  p.C = out; p.ldc = ldo; p.lower = lower;
  p.q1 = qa; p.q2 = qb;
  p.scale = h->lsw2[0] / (double)D; p.sb2 = h->lsb2[0]; p.steps = h->cfg.depth - 1;
  for (int i = 0; i < GEMM_MAX_LAYERS; ++i) {      // step s is followed by Dense layer s + 1
    p.lsw2[i] = h->lsw2[std::min(i + 1, NNGP_MAX_LAYERS - 1)];
    p.lsb2[i] = h->lsb2[std::min(i + 1, NNGP_MAX_LAYERS - 1)];
  }
  MatView a{A, M, D, lda}, b{B, N, D, ldb};
  if (h->act.kind == ACT_ERF && p.steps > 1 && M > 0 && N > 0) {
    // the diagonals of layers 1..steps-1 of both operands (one table when both are the same rows), on the stream of
    // the launch that reads them
    const bool same = qa == qb && M == N;
    if (h->qtab.cap < act_table_bytes(h, same ? M : M + N))
      return fail(h, NNGP_EINVAL, "internal: diagonal tables sized for fewer than %lld rows", (long long)(same ? M : M + N));
    double* ta = h->qtab.as<double>();
    double* tb = same ? ta : ta + (int64_t)(p.steps - 1) * M;
    const LayerSig sig = layer_sig(h);
    q_final_kernel<<<(unsigned)((M + 255) / 256), 256, 0, h->cur>>>(qa, (int)M, p.steps, sig, h->act, ta, nullptr);
    h->st.kernel_launches++;
    if (!same) {
      q_final_kernel<<<(unsigned)((N + 255) / 256), 256, 0, h->cur>>>(qb, (int)N, p.steps, sig, h->act, tb, nullptr);
      h->st.kernel_launches++;
    }
    p.tab1 = ta; p.tld1 = M;
    p.tab2 = tb; p.tld2 = N;
  }
  switch (h->act.kind) {
    case ACT_ABRELU: return launch_gemm<EPI_GRAM, ACT_ABRELU>(h, a, 0, 0, b, 0, 0, p);
    case ACT_ERF: return launch_gemm<EPI_GRAM, ACT_ERF>(h, a, 0, 0, b, 0, 0, p);
    default: return launch_gemm<EPI_GRAM>(h, a, 0, 0, b, 0, 0, p);
  }
}

// C(M x N at `C`, ldc) -= Aop[a_row0:+M, a_col0:+K] * Bop[b_row0:+N, b_col0:+K]^T ; K % 16 == 0.
int run_gemm_sub(nngp_handle* h, const MatView& A, int64_t a_row0, int64_t a_col0, const MatView& B, int64_t b_row0,
                 int64_t b_col0, int64_t M, int64_t N, int64_t K, double* C, int64_t ldc, int lower) {
  if (K <= 0) return NNGP_OK;
  if (K % GEMM_BK) return fail(h, NNGP_EINVAL, "internal: GEMM K=%lld not a multiple of 16", (long long)K);
  GemmParams p{};
  p.M = (int)M; p.N = (int)N; p.ktiles = (int)(K / GEMM_BK);
  p.C = C; p.ldc = ldc; p.lower = lower;
  return launch_gemm<EPI_SUB>(h, A, (int)a_row0, (int)a_col0, B, (int)b_row0, (int)b_col0, p);
}

// partial[tile_n][r] = sum_{c in tile_n} (V M^T)[r][c] * V[r][c]   (V: rows x N at `V`, ldv; M: N x N, ldm == ldv)
int run_gemm_rowdot(nngp_handle* h, const double* V, int64_t ldv, int64_t rows, const double* Mm, int64_t N,
                    double* partial) {
  GemmParams p{};
  p.M = (int)rows; p.N = (int)N; p.ktiles = (int)((N + GEMM_BK - 1) / GEMM_BK);
  p.ldc = ldv; p.W = V; p.partial = partial;
  MatView a{V, rows, N, ldv}, b{Mm, N, N, ldv};
  return launch_gemm<EPI_ROWDOT>(h, a, 0, 0, b, 0, 0, p);
}

// ---- blocked Cholesky (lower, in place, row-major) ----------------------------------------------
// Right-looking over W-wide outer panels (trailing SYRK with K = W on the DMMA core), left-looking
// over the 64-wide sub-panels inside a panel (potrf_panel).
// Outer panel width: 256 keeps the panel chain short for small N; for larger N the trailing SYRK
// dominates and K = 512 runs closer to the DMMA peak (measured at N = 32768: 394 / 378 / 371 ms for
// W = 256 / 384 / 512; at N = 8192: 13.8 / 14.5 / 15.2 ms).
int chol_outer_width(int64_t N) {
  // (with the fused panel kernel: N = 4096 3.44 vs 3.54 ms, N = 8192 9.67 vs 9.96 ms for W = 512 vs 256;
  //  N = 32768: 356.0 / 353.9 / 352.0 ms for W = 512 / 768 / 1024)
  return N >= 24576 ? 1024 : (N >= 4096 ? 512 : 256);
}

// ---- device buffer sizes ----------------------------------------------------------------------------
// Every size passed to ensure() for a buffer of the handle comes from one function here, which both the code using the
// buffer and nngp_reserve call: a reserved handle never reallocates.

bool builds_inverse(const nngp_handle* h) { return h->cfg.latency_mode && h->cfg.kernel_type == 0; }   // L^-1
bool can_append_incrementally(const nngp_handle* h) { return h->cfg.diag_reg_absolute && h->cfg.kernel_type == 0; }

// fused panel kernel of an N-column factorisation of R rows: {item counter, progress[row tiles], inv_ready[col blocks]}
int ensure_panel_sync(nngp_handle* h, int64_t N, int64_t R) {
  return ensure(h, h->panel_sync, (size_t)(2 + (R + GEMM_BM - 1) / GEMM_BM + (chol_outer_width(N) + NB - 1) / NB) * sizeof(int));
}

// solves over `rows` rows: sums of squares per row, counters of trsm_fused (per 128-row tile) / trsv_bwd (per 64-block)
int ensure_solve_workspace(nngp_handle* h, int64_t rows) {
  CKR(ensure(h, h->ssq, (size_t)rows * sizeof(double)));
  return ensure(h, h->sync_ints, (size_t)((rows + NB - 1) / NB + 1) * sizeof(int));
}

// Rows per sub-block of run_sliced_variance: its planes fit 16 GiB, in whole waves of 37 row tiles x 4 column tiles (so
// that the static tile order stays balanced).
int64_t sliced_rows(const nngp_handle* h, int64_t N, int64_t rows) {
  const int64_t wave_rows = (int64_t)(h->sm_count / SL_SUPER) * SL_RT * SL_BM;
  const int64_t sb = ((16LL << 30) / ((int64_t)h->cfg.variance_slices * round_up(N, SL_BK))) / wave_rows * wave_rows;
  return std::min<int64_t>(std::max<int64_t>(sb, SL_RT * SL_BM), round_up(rows, SL_RT * SL_BM));
}

// launch_sliced over rows x N: CTAs 4k..4k+3 share K_* row tiles; per-CTA running-sum tiles, one counter per round
int sliced_grid(nngp_handle* h, int64_t rows, int64_t N, int* grid, int64_t* rounds) {
  const int64_t tiles = ((rows + SL_BM - 1) / SL_BM + SL_RT - 1) / SL_RT * ((N + SL_BN - 1) / SL_BN);
  *grid = (int)std::min<int64_t>((h->sm_count / SL_SUPER) * SL_SUPER, tiles);
  *rounds = (tiles + *grid - 1) / *grid;
  CKR(ensure(h, h->slscratch, (size_t)*grid * SL_RT * SL_BM * SL_BN * sizeof(double)));
  return *rounds >= 2 ? ensure(h, h->slsync, (size_t)*rounds * sizeof(int)) : NNGP_OK;
}

// h->partial of a variance over `rows` rows, whichever path runs: the 'ntk' row-dot and the widest split of
// run_inverse_variance (tri_gemv; <= 8 K chunks, only while rows x N spans < 4 tiles per SM; one per column tile), and
// run_sliced_variance.  Non-decreasing in N and rows, so the largest problem's size covers the smaller ones.
size_t partial_bytes(const nngp_handle* h, int64_t N, int64_t rows) {
  int64_t n = rows * ((N + GEMM_BN - 1) / GEMM_BN);
  if (builds_inverse(h)) {
    const int64_t chunks = std::min<int64_t>(8, ((N + GEMM_BK - 1) / GEMM_BK + 63) / 64);
    n = std::max({n, std::min<int64_t>(rows, TGV_MAXR) * N, chunks * std::min<int64_t>(rows * N, 4LL * h->sm_count * GEMM_BM * GEMM_BN)});
    if (h->cfg.variance_slices > 0) n = std::max(n, 2 * ((N + SL_BN - 1) / SL_BN) * sliced_rows(h, N, rows));
  }
  return (size_t)n * sizeof(double);
}

// run_sliced_variance over `rows` rows: K_* digit planes and row exponents of a sub-block, partials, launch workspace
int ensure_sliced_block(nngp_handle* h, int64_t N, int64_t rows) {
  const int64_t sb = sliced_rows(h, N, rows);
  int grid;
  int64_t rounds;
  CKR(ensure(h, h->Aq, (size_t)h->cfg.variance_slices * sb * round_up(N, SL_BK)));
  CKR(ensure(h, h->aexp, (size_t)sb * sizeof(int)));
  CKR(ensure(h, h->partial, partial_bytes(h, N, rows)));
  return sliced_grid(h, sb, N, &grid, &rounds);
}

// Erf, depth > 2: the diagonal tables of layers 1..depth-2 for a Gram launch over `rows` distinct operand rows
// (run_gram; every caller sizes them for its largest launch)
size_t act_table_bytes(const nngp_handle* h, int64_t rows) {
  const int64_t steps = h->cfg.depth - 1;
  return h->act.kind == ACT_ERF && steps >= 2 ? (size_t)(steps - 1) * rows * sizeof(double) : 0;
}
int ensure_act_tables(nngp_handle* h, int64_t rows) {
  const size_t bytes = act_table_bytes(h, rows);
  return bytes ? ensure(h, h->qtab, bytes) : NNGP_OK;
}

// the training rows X and their layer-0 diagonals q
int ensure_inputs(nngp_handle* h, int64_t N, int64_t D) {
  CKR(ensure(h, h->X, (size_t)N * round_up(D, 2) * sizeof(double)));
  return ensure(h, h->q, (size_t)N * sizeof(double));
}

// A fitted state of N x D, on every handle that holds one (replicas too): X, q, L (+1 row: y^T rides through the
// factorisation), alpha, inv(L_JJ); M ('ntk'); in latency mode L^-1 and, with variance_slices, its digit planes.
int ensure_model(nngp_handle* h, int64_t N, int64_t D) {
  const int64_t ldl = round_up(N, 16), ldq = round_up(N, SL_BK);
  const int s = h->cfg.variance_slices;
  CKR(ensure_inputs(h, N, D));
  CKR(ensure_act_tables(h, N));
  CKR(ensure(h, h->L, (size_t)(N + 1) * ldl * sizeof(double)));
  CKR(ensure(h, h->alpha, (size_t)ldl * sizeof(double)));
  CKR(ensure(h, h->Linv, (size_t)round_up(N, NB) * NB * sizeof(double)));
  if (h->cfg.kernel_type == 1) CKR(ensure(h, h->Mmat, (size_t)N * ldl * sizeof(double)));
  if (builds_inverse(h)) CKR(ensure(h, h->Linvfull, (size_t)N * ldl * sizeof(double)));
  if (s <= 0) return NNGP_OK;
  if ((int64_t)s * 4096 * ldq >= (1LL << 31))
    return fail(h, NNGP_EINVAL, "variance_slices = %d: int32 plane sums need N <= %lld (N = %lld)", s,
                (long long)((1LL << 19) / s), (long long)N);
  CKR(ensure(h, h->Wq, (size_t)s * round_up(N, SL_BN) * ldq));
  return ensure(h, h->wexp, (size_t)N * sizeof(int));
}

// Only the handle that fits N rows: y, z = L^-1 y, the panel counters of the (N + 1)-row factorisation, K_dd ('ntk')
// or the scratch of L^-T (latency mode), and the solves over N rows ('ntk' M, build_inverse, the alpha solve).
int ensure_fit_workspace(nngp_handle* h, int64_t N) {
  CKR(ensure(h, h->y, (size_t)N * sizeof(double)));
  CKR(ensure(h, h->zkeep, (size_t)N * sizeof(double)));
  CKR(ensure_panel_sync(h, N, N + 1));
  if (h->cfg.kernel_type == 1 || builds_inverse(h)) CKR(ensure(h, h->Kdd, (size_t)N * round_up(N, 16) * sizeof(double)));
  return ensure_solve_workspace(h, N);
}

// nngp_append_fit up to N x D: the staging [X; X_new], [y; y_new]; for the incremental append the second factor and
// the inverses of the Schur block (at most N rows)
int ensure_append_workspace(nngp_handle* h, int64_t N, int64_t D) {
  CKR(ensure(h, h->app_x, (size_t)N * D * sizeof(double)));
  CKR(ensure(h, h->app_y, (size_t)N * sizeof(double)));
  CKR(ensure_act_tables(h, N));   // (the incremental append's K21: the M new rows against the N - M old ones)
  if (!can_append_incrementally(h)) return NNGP_OK;
  CKR(ensure(h, h->L2, (size_t)(N + 1) * round_up(N, 16) * sizeof(double)));
  return ensure(h, h->panel_inv, (size_t)round_up(N, NB) * NB * sizeof(double));
}

// Rows per block of nngp_predict: what fits cfg.max_block_bytes (the 'ntk' variance holds two blocks), in equal blocks
// of whole 128-row tiles -- the persistent solve keeps every SM busy with any tile count, what hurts is a last block
// with too few row tiles to fill the GPU.
int64_t predict_block_rows(const nngp_handle* h, int64_t N, int64_t T, bool want_var) {
  int64_t cap_rows = h->cfg.max_block_bytes / (round_up(N, 16) * 8) / (h->cfg.kernel_type == 1 && want_var ? 2 : 1);
  cap_rows = std::min<int64_t>(std::max<int64_t>(cap_rows, GEMM_BM), 65535LL * GEMM_BM);
  const int64_t nblocks = (T + cap_rows - 1) / cap_rows;
  return std::min<int64_t>(round_up(T, 2), round_up((T + nblocks - 1) / nblocks, GEMM_BM));
}

// nngp_predict of T rows against N x D training rows
int ensure_predict_workspace(nngp_handle* h, int64_t N, int64_t D, int64_t T, bool want_var) {
  const int64_t TB = predict_block_rows(h, N, T, want_var), ldl = round_up(N, 16);
  const bool ntk = h->cfg.kernel_type == 1;
  for (DevBuf* b : {&h->qt, &h->kss}) CKR(ensure(h, *b, (size_t)TB * sizeof(double)));
  CKR(ensure(h, h->xt, (size_t)TB * round_up(D, 2) * sizeof(double)));
  CKR(ensure(h, h->blk, (size_t)TB * ldl * sizeof(double)));
  CKR(ensure(h, h->mean_partial, (size_t)TB * 2 * ((N + GEMM_BN - 1) / GEMM_BN) * sizeof(double)));  // per 32 columns
  CKR(ensure(h, h->mean_d, (size_t)T * sizeof(double)));
  CKR(ensure_act_tables(h, TB + N));   // (a chunk of the block against the training rows; the covariance: TB rows)
  if (!want_var) return NNGP_OK;
  CKR(ensure(h, h->var_d, (size_t)T * sizeof(double)));
  CKR(ensure_solve_workspace(h, TB));
  if (ntk) CKR(ensure(h, h->blk2, (size_t)TB * ldl * sizeof(double)));
  if (ntk) CKR(ensure(h, h->cross, (size_t)TB * sizeof(double)));
  if (ntk || builds_inverse(h)) CKR(ensure(h, h->partial, partial_bytes(h, N, TB)));
  return h->cfg.variance_slices > 0 ? ensure_sliced_block(h, N, TB) : NNGP_OK;
}

// nngp_predict_cov: the largest batch whose V ('ntk': V, U and P = -V M) fits cfg.max_block_bytes -- the whole batch is
// one prediction block (T <= this keeps predict_block_rows at one block of T rows, so V and U are blk and blk2)
int64_t cov_max_rows(const nngp_handle* h, int64_t N) {
  const int64_t per_row = round_up(N, 16) * 8 * (h->cfg.kernel_type == 1 ? 3 : 1);
  return std::min<int64_t>(h->cfg.max_block_bytes / per_row, 65535LL * GEMM_BM);
}

// nngp_predict_cov of T rows (on top of ensure_predict_workspace): the T x T result, leading dimension round_up(T, 2)
// (the GEMM epilogues store pairs of columns), and P = -V M ('ntk', T x round_up(N, 16))
int ensure_cov_workspace(nngp_handle* h, int64_t N, int64_t T) {
  CKR(ensure(h, h->cov, (size_t)T * round_up(T, 2) * sizeof(double)));
  return h->cfg.kernel_type == 1 ? ensure(h, h->covP, (size_t)T * round_up(N, 16) * sizeof(double)) : NNGP_OK;
}

// nngp_active_select of k out of T pool rows
int ensure_select_workspace(nngp_handle* h, int64_t T, int64_t k) {
  for (DevBuf* b : {&h->sel_mean, &h->sel_var, &h->sel_score, &h->sel_key}) CKR(ensure(h, *b, (size_t)T * 8));
  CKR(ensure(h, h->sel_okey, (size_t)k * 8));
  CKR(ensure(h, h->sel_oidx, (size_t)k * 4));
  CKR(ensure(h, h->sel_state, sizeof(SelectState)));
  return ensure(h, h->sel_max, 8);
}

// One outer panel, columns [j0, j0 + w) of the rows from j0 down to `R` = N + extra rows riding along below the
// matrix (see run_potrf), as one persistent kernel (potrf_panel.cuh).  Per 64-wide sub-panel: the left-looking
// update from the panel's earlier columns, potf2_64_block (Cholesky of the diagonal block AND its inverse
// W = inv(L_JJ)), and the block column below it, X L_JJ^T = B  ->  X = B W^T, as a K = 64 product on the tensor pipe.
// `Winv` receives the inverses, block J at rows [64 J, 64 J + 64) of a 64-wide matrix.
int potrf_panel(nngp_handle* h, double* A, int64_t ld, int64_t N, int64_t R, int64_t j0, int64_t w, double* Winv) {
  PanelParams p{};
  p.A = A; p.ld = ld; p.j0 = (int)j0; p.rows = (int)(R - j0); p.ncols = (int)w;
  p.row_tiles = (int)((R - j0 + GEMM_BM - 1) / GEMM_BM);
  p.col_blocks = (int)((w + NB - 1) / NB);
  p.info = h->flags.as<int>();
  p.Winv = Winv;
  const size_t nints = (size_t)1 + p.row_tiles + p.col_blocks;
  CK(cudaMemsetAsync(h->panel_sync.p, 0, nints * sizeof(int), h->cur));   // (sized by run_potrf)
  p.counter = h->panel_sync.as<int>();
  p.progress = p.counter + 1;
  p.inv_ready = p.progress + p.row_tiles;
  CUtensorMap tmA, tmL, tmW;
  CKR(get_tmap(h, A, R, N, ld, GEMM_BM, &tmA));
  CKR(get_tmap(h, A, R, N, ld, GEMM_BN, &tmL));
  CKR(get_tmap(h, Winv, round_up(N, NB), NB, NB, GEMM_BN, &tmW));
  // Grid: a few CTAs per row tile, but no more than a quarter of the GPU's CTA slots.  The kernel's CTAs spend most of
  // their life waiting for the owner's potf2; every slot they hold is a slot the trailing update running beside
  // them (look-ahead) cannot use -- with 2 x #SMs spinning CTAs the overlap was gone (measured: 11.0 ms at N = 8192,
  // no better than the launch-per-step chain this kernel replaced).
  const long long total = (long long)p.row_tiles * p.col_blocks;
  // (3 CTAs per row tile: the extra ones claim the row tile's NEXT column blocks early and work through the k-tiles
  //  that already exist while the owner is still factoring -- N = 4096: 3.45 -> 3.28 ms, 8192: 9.65 -> 9.50 ms)
  int grid = (int)std::min<long long>((long long)p.row_tiles * 3, h->sm_count / 2);
  grid = (int)std::max<long long>(1, std::min<long long>(grid, total));
  // NNGP_PANEL_TRACE=1 (diagnostics): time stamps of the owner items of every panel -> stderr (synchronises!)
#ifdef NNGP_PANEL_TRACE
  static const bool trace = [] { const char* e = getenv("NNGP_PANEL_TRACE"); return e && atoi(e) > 0; }();
#else
  const bool trace = false;   // (the stamps are compiled into the kernel only by build.sh -DNNGP_PANEL_TRACE)
#endif
  unsigned long long* tr_d = nullptr;
  if (trace) {
    CK(cudaMalloc(&tr_d, (size_t)p.col_blocks * 18 * sizeof(unsigned long long)));
    CK(cudaMemsetAsync(tr_d, 0, (size_t)p.col_blocks * 18 * sizeof(unsigned long long), h->cur));
    p.trace = tr_d;
  }
  potrf_panel_kernel<<<grid, GEMM_THREADS, TF_SMEM_BYTES, h->cur>>>(tmA, tmL, tmW, p);
  CK(cudaGetLastError());
  h->st.kernel_launches++;
  if (trace) {
    std::vector<unsigned long long> tr((size_t)p.col_blocks * 18);
    CK(cudaStreamSynchronize(h->cur));
    CK(cudaMemcpy(tr.data(), tr_d, tr.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    cudaFree(tr_d);
    const unsigned long long t00 = tr[0];
    fprintf(stderr, "panel j0=%lld rows=%d grid=%d: per owner item [claimed, update done, R stored, factor done, inverse stored, flag+reload, W+R staged, diag done, published] us since the panel's first claim\n",
            (long long)j0, p.rows, grid);
    for (int J = 0; J < p.col_blocks; ++J) {
      fprintf(stderr, "  J=%d:", J);
      for (int k = 0; k < 9; ++k) fprintf(stderr, " %8.2f", tr[(size_t)J * 10 + k] ? (double)(tr[(size_t)J * 10 + k] - t00) / 1e3 : -1.0);
      const unsigned long long* pt = tr.data() + (size_t)p.col_blocks * 10 + (size_t)J * 8;   // inside potf2_64_block
      fprintf(stderr, "   | potf2: loaded %.2f; micro-panel 8: A %.2f B %.2f C %.2f; 9: A %.2f B %.2f C %.2f; factor done %.2f",
              (double)(pt[1] - t00) / 1e3, (double)(pt[2] - t00) / 1e3, (double)(pt[3] - t00) / 1e3, (double)(pt[4] - t00) / 1e3,
              (double)(pt[5] - t00) / 1e3, (double)(pt[6] - t00) / 1e3, (double)(pt[7] - t00) / 1e3, (double)(pt[0] - t00) / 1e3);
      fprintf(stderr, "\n");
    }
  }
  return NNGP_OK;
}

// Blocked right-looking Cholesky.  The trailing update of outer step j is split into (A) the columns of the NEXT
// panel and (B) the rest.
// Look-ahead (on by default, NNGP_CHOL_LOOKAHEAD=0 disables it): as soon as (A) is done the next panel is factored
// on a high-priority stream while (B) keeps the tensor pipes busy on the main stream (-6 % fit time at N = 32768,
// -30 % at N = 8192).  The two streams touch disjoint column ranges, so the factor is bitwise the same with and
// without it (tests/test_gpu_parity.py, tools/determinism_check.py).
// `extra` rows stored below the matrix (rows N..N+extra-1, N columns each) are carried through every
// panel solve and trailing update: on exit they hold  E L^-T.  The fit puts y^T there, so the forward
// substitution z = L^-1 y of the alpha solve costs nothing extra (one more row in GEMMs already running).
int run_potrf(nngp_handle* h, double* A, int64_t ld, int64_t N, int64_t extra, double* Winv) {
  const int W = chol_outer_width(N);
  const int64_t R = N + extra;
  MatView Av{A, R, N, ld};
  CKR(ensure_panel_sync(h, N, R));
  const bool lookahead = h->panel_stream != nullptr && N > 2 * W;
  cudaEvent_t ev_cols = get_event(h), ev_panel = get_event(h);
  auto edge = [&](cudaEvent_t e, cudaStream_t from, cudaStream_t to) -> cudaError_t {
    cudaError_t r = cudaEventRecord(e, from);
    if (r == cudaSuccess) r = cudaStreamWaitEvent(to, e, 0);
    return r;
  };
  int rc = NNGP_OK;
  cudaError_t ce = cudaSuccess;
  // NNGP_CHOL_TRACE=1 (diagnostics): device time line of every panel / (A) / (B) launch -> stderr (synchronises)
  static const bool tl_on = [] { const char* e = getenv("NNGP_CHOL_TRACE"); return e && atoi(e) > 0; }();
  struct Span { const char* what; int64_t j0; cudaEvent_t a, b; };
  std::vector<Span> spans;
  auto span_begin = [&](const char* what, int64_t j) { if (tl_on) { Span sp{what, j, nullptr, nullptr}; cudaEventCreate(&sp.a); cudaEventCreate(&sp.b); cudaEventRecord(sp.a, h->cur); spans.push_back(sp); } };
  auto span_end = [&]() { if (tl_on) cudaEventRecord(spans.back().b, h->cur); };
  if (lookahead) ce = edge(ev_cols, h->stream, h->panel_stream);  // panel stream starts after the work queued so far
  for (int64_t j0 = 0; j0 < N && rc == NNGP_OK && ce == cudaSuccess; j0 += W) {
    const int64_t w = std::min<int64_t>(W, N - j0);
    const int64_t t0 = j0 + w;
    h->cur = lookahead ? h->panel_stream : h->stream;
    span_begin("panel", j0);
    rc = potrf_panel(h, A, ld, N, R, j0, w, Winv);
    span_end();
    if (rc != NNGP_OK || t0 >= N) break;
    if (lookahead) ce = edge(ev_panel, h->panel_stream, h->stream);
    h->cur = h->stream;
    const int64_t w2 = std::min<int64_t>(W, N - t0);
    const int64_t t1 = t0 + w2;
    // (A) next panel's columns: A[t0:R, t0:t1] (lower tiles) -= A[t0:R, j0:t0] * A[t0:t1, j0:t0]^T
    span_begin("A", j0);
    rc = run_gemm_sub(h, Av, t0, j0, Av, t0, j0, R - t0, w2, w, A + t0 * ld + t0, ld, 1);
    span_end();
    if (rc != NNGP_OK) break;
    if (lookahead && ce == cudaSuccess) ce = edge(ev_cols, h->stream, h->panel_stream);
    // (B) the rest of the trailing matrix: A[t1:R, t1:N] (lower) -= A[t1:R, j0:t0] * A[t1:N, j0:t0]^T
    span_begin("B", j0);
    if (t1 < N) rc = run_gemm_sub(h, Av, t1, j0, Av, t1, j0, R - t1, N - t1, w, A + t1 * ld + t1, ld, 1);
    span_end();
  }
  if (lookahead && ce == cudaSuccess) ce = edge(ev_panel, h->panel_stream, h->stream);  // join
  h->cur = h->stream;
  if (tl_on && !spans.empty()) {
    cudaStreamSynchronize(h->stream);
    if (h->panel_stream) cudaStreamSynchronize(h->panel_stream);
    fprintf(stderr, "cholesky time line N=%lld W=%d (ms since the first panel's start): what j0 start end\n", (long long)N, W);
    for (auto& sp : spans) {
      float t0 = 0.f, t1 = 0.f;
      cudaEventElapsedTime(&t0, spans[0].a, sp.a);
      cudaEventElapsedTime(&t1, spans[0].a, sp.b);
      fprintf(stderr, "  %-5s %6lld %8.3f %8.3f  (%.3f)\n", sp.what, (long long)sp.j0, t0, t1, t1 - t0);
    }
    for (auto& sp : spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); }
    cudaGetLastError();
  }
  h->ev_pool.push_back(ev_cols);
  h->ev_pool.push_back(ev_panel);
  if (ce != cudaSuccess) rc = fail(h, NNGP_ECUDA, "look-ahead event plumbing failed: %s", cudaGetErrorString(ce));
  CKR(rc);
  CK(cudaGetLastError());
  return NNGP_OK;
}

// B (rows x N, ldb) <- B * L^-T  (solve X L^T = B; L lower N x N row-major) plus, optionally, the posterior
// variance of every row, as ONE persistent kernel (trsm_fused.cuh).
int run_trsm_fused(nngp_handle* h, double* B, int64_t ldb, int64_t rows, const double* L, int64_t ldl, int64_t N,
                   const double* Linv, const double* kss, double* var, int upper_start = 0) {
  TrsmFusedParams p{};
  p.upper_start = upper_start;
  p.B = B; p.ldb = ldb; p.rows = (int)rows; p.L = L; p.ldl = ldl; p.N = (int)N;
  p.row_tiles = (int)((rows + GEMM_BM - 1) / GEMM_BM);
  p.col_blocks = (int)((N + NB - 1) / NB);
  CKR(ensure_solve_workspace(h, rows));
  CK(cudaMemsetAsync(h->sync_ints.p, 0, (size_t)(p.row_tiles + 1) * sizeof(int), h->stream));
  p.counter = h->sync_ints.as<int>();
  p.progress = h->sync_ints.as<int>() + 1;
  p.ssq = h->ssq.as<double>(); p.kss = kss; p.var = var;
  CUtensorMap tmB, tmL, tmW;
  CKR(get_tmap(h, B, rows, N, ldb, GEMM_BM, &tmB));
  CKR(get_tmap(h, L, N, N, ldl, GEMM_BN, &tmL));
  CKR(get_tmap(h, Linv, round_up(N, NB), NB, NB, GEMM_BN, &tmW));
  const long long total = (long long)p.row_tiles * p.col_blocks;
  // Fewer row tiles than CTA slots: several CTAs work on the same row tile at different J, each consuming the
  // column blocks of V as their producers publish them (software pipeline along J, see the gate in the kernel).
  const int grid = (int)std::min<long long>(total, 2LL * h->sm_count);
  p.static_sched = (p.row_tiles % grid == 0) ? 1 : 0;
  const int span = span_open(h, 2, h->cur, &h->st.gemm_ms);
  // Plenty of row tiles (or exactly one static round of them): dependencies are practically always met when an item
  // starts, and the ungated kernel is 0.5 % faster (34.8 vs 34.6 TFLOP/s at C2).  Measured at N = 8192: 296 tiles
  // 81 ms ungated / 83 gated; 313 tiles 92 ms ungated / 86 gated.
  if (p.static_sched || p.row_tiles >= grid + grid / 4)
    trsm_fused_kernel<false><<<grid, GEMM_THREADS, TF_SMEM_BYTES, h->stream>>>(tmB, tmL, tmW, p);
  else                       // several CTAs per row tile: pipeline along J
    trsm_fused_kernel<true><<<grid, GEMM_THREADS, TF_SMEM_BYTES, h->stream>>>(tmB, tmL, tmW, p);
  span_close(h, span);
  CK(cudaGetLastError());
  h->st.kernel_launches++;
  h->st.gemm_launches++;
  h->st.gemm_flops += (double)rows * (double)N * (double)N * (upper_start ? 1.0 / 3.0 : 1.0);  // N^2 flop per test row (SURVEY 8d)
  return NNGP_OK;
}

// Small-batch variant of the same solve (identical arithmetic: every element sees the same FMA chain in ascending
// k, the same diagonal step and epilogue, see diag_epilogue): right-looking over OW-wide outer blocks, so every
// trailing update exposes (N - j)/64 column tiles of parallelism even when there is a single row tile -- the
// persistent left-looking kernel would walk the N/64 blocks of a row tile sequentially on one SM.  Inside an outer
// block the 64-wide column blocks are solved left-looking (update with the block's own earlier columns, then the
// diagonal step).  OW = 256 instead of 64 cuts the read-modify-write traffic of the trailing updates 4x (at 4096
// rows x N = 8192: 34 GB -> 8.5 GB) and gives them K = 256.  Used when the block has few row tiles (serving a
// handful of queries, the forest workload).
int run_trsm_right(nngp_handle* h, double* B, int64_t ldb, int64_t rows, const double* L, int64_t ldl, int64_t N,
                   const double* Linv, const double* kss, double* var) {
  MatView Bv{B, rows, N, ldb}, Lv{L, N, N, ldl}, Wv{Linv, round_up(N, NB), NB, NB};
  const int col_blocks = (int)((N + NB - 1) / NB);
  // one or two row tiles are launch-latency bound: keep the plain 64-wide sweep (2 launches per column block)
  const int64_t OW = rows <= 2 * GEMM_BM ? NB : 4 * NB;
  CKR(ensure_solve_workspace(h, rows));
  for (int64_t o0 = 0; o0 < N; o0 += OW) {
    const int64_t o1 = std::min<int64_t>(o0 + OW, N);
    for (int64_t j0 = o0; j0 < o1; j0 += NB) {
      const int64_t nb = std::min<int64_t>(NB, N - j0);
      const int J = (int)(j0 / NB);
      if (j0 > o0)  // B[:, J] -= V[:, o0:j0] * L[J, o0:j0]^T
        CKR(run_gemm_sub(h, Bv, 0, o0, Lv, j0, o0, rows, nb, j0 - o0, B + j0, ldb, 0));
      GemmParams p{};   // V[:, J] = R[:, J] * inv(L_JJ)^T in place (+ running sum of squares / variance)
      p.M = (int)rows; p.N = (int)nb; p.ktiles = NB / GEMM_BK;
      p.C = B + j0; p.ldc = ldb;
      p.ssq = h->ssq.as<double>(); p.kss = kss; p.var = var; p.J = J; p.col_blocks = col_blocks;
      CKR(launch_gemm<EPI_DIAG>(h, Bv, 0, (int)j0, Wv, (int)j0, 0, p));
    }
    if (o1 < N)  // B[:, o1:] -= V[:, o0:o1] * L[o1:, o0:o1]^T
      CKR(run_gemm_sub(h, Bv, 0, o0, Lv, o1, o0, rows, N - o1, o1 - o0, B + o1, ldb, 0));
  }
  CK(cudaGetLastError());
  return NNGP_OK;
}

// Row-tile count up to which the right-looking path is used: 0, i.e. never, by default.  Since the persistent kernel
// gates every operand tile on its producer's progress (several CTAs pipeline along J inside one row tile) it is
// the faster path at every batch size measured (N = 8192: 1 row 2.0 vs 2.6 ms, 1024 rows 4.0 vs 6.1, 8192 rows
// 19.2 vs 21.6, 20 000 rows 44 vs 48 ms).  The right-looking path stays as the independent implementation the
// parity tests cross-check bit for bit.  Read on every call so tests / A-B runs can flip it inside one process.
int small_batch_row_tiles(const nngp_handle* h) {
  (void)h;
  const char* e = getenv("NNGP_SMALL_BATCH_TILES");
  return e ? atoi(e) : 0;
}

// V = K_* L^-T (+ variance): the persistent fused kernel, or (on request) the right-looking steps.
int run_predict_solve(nngp_handle* h, double* B, int64_t ldb, int64_t rows, const double* L, int64_t ldl, int64_t N,
                      const double* kss, double* var) {
  const double* Linv = h->Linv.as<double>();   // L is always the handle's factor
  const int64_t row_tiles = (rows + GEMM_BM - 1) / GEMM_BM;
  if (row_tiles <= small_batch_row_tiles(h)) return run_trsm_right(h, B, ldb, rows, L, ldl, N, Linv, kss, var);
  return run_trsm_fused(h, B, ldb, rows, L, ldl, N, Linv, kss, var);
}

// ---- latency mode (cfg.latency_mode): explicit inverse factor ---------------------------------------
// Serving a handful of query lines per call (estimator.py:42-62) is latency-bound on the substitution chain of
// V = K_* L^-T: N/64 dependent steps of ~10 us.  With W = L^-1 held explicitly the same V is a plain product
// K_* W^T -- no dependencies, every column tile independent -- whose cost for a few rows is one pass over W.
// W is built once per fit on the same DMMA kernels: X L^T = I solved by the persistent kernel (upper-triangular
// right-hand side: N^3/3 flop), X = L^-T, then W = X^T.  inv(L) is as benign as inv(L_JJ) in the diagonal step:
// the error of K_* W^T is eps * cond(L) = eps * sqrt(cond(K + lambda I)) (tests/checks/illcond_report.py).
int build_w_planes(nngp_handle* h);
int build_inverse(nngp_handle* h) {
  const int64_t N = h->N, ldl = h->ldl;
  CKR(ensure_fit_workspace(h, N));                             // Kdd: scratch for L^-T; the solve workspace
  double* X = h->Kdd.as<double>();
  h->st.inverse_ms = 0.0;   // the last fit's, not a sum
  const int span = span_open(h, 0, h->stream, &h->st.inverse_ms);
  set_identity_kernel<<<4 * h->sm_count, 256, 0, h->stream>>>(X, ldl, (int)N);
  h->st.kernel_launches++;
  CKR(run_trsm_fused(h, X, ldl, N, h->L.as<double>(), ldl, N, h->Linv.as<double>(), nullptr, nullptr, 1));
  dim3 tg((unsigned)((N + 31) / 32), (unsigned)((N + 31) / 32));
  transpose_kernel<<<tg, dim3(32, 8), 0, h->stream>>>(X, h->Linvfull.as<double>(), ldl, (int)N);
  h->st.kernel_launches++;
  span_close(h, span);
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaGetLastError());
  settle_spans(h);
  h->have_inv = true;
  if (h->cfg.variance_slices > 0) CKR(build_w_planes(h));
  return NNGP_OK;
}

// Row count up to which nngp_predict uses the explicit inverse in FP64 (NNGP_LATENCY_ROWS overrides; read per call).
// With digit planes (variance_slices) the int8 product takes over as soon as the batch fills the GPU with tiles.
int64_t latency_rows(const nngp_handle* h) {
  if (!h->have_inv) return 0;
  const char* e = getenv("NNGP_LATENCY_ROWS");
  return e ? atoll(e) : (h->have_wq ? 767 : 4096);
}

// var[r] = kss[r] - |K_*[r,:] W^T|^2 through the explicit inverse: one triangular GEMM whose epilogue reduces the
// squares of each 64-column tile (V itself is never written), then a fixed-order sum over the tiles.
int run_inverse_variance(nngp_handle* h, const double* B, int64_t ldb, int64_t rows, const double* kss, double* var) {
  const int64_t N = h->N;
  const int col_tiles = (int)((N + GEMM_BN - 1) / GEMM_BN);
  GemmParams p{};
  p.M = (int)rows; p.N = (int)N; p.ktiles = (int)((N + GEMM_BK - 1) / GEMM_BK);
  p.ldc = ldb; p.W = nullptr; p.tri_k = 1;
  MatView a{B, rows, N, ldb}, b{h->Linvfull.as<double>(), N, N, h->ldl};
  const int64_t row_tiles = (rows + GEMM_BM - 1) / GEMM_BM;
  CKR(ensure(h, h->partial, partial_bytes(h, N, rows)));
  if (rows <= TGV_MAXR) {
    // A handful of queries: one streaming pass over L^-1 (tri_gemv_kernel), then the fixed-order row reduction.
    const int ngroups = (int)((N + 7) / 8);
    const dim3 tg((unsigned)((ngroups + 1) / 2));
    const double* Wf = h->Linvfull.as<double>();
    double* vp = h->partial.as<double>();
    if (rows == 1) tri_gemv_kernel<1><<<tg, 256, 0, h->stream>>>(Wf, h->ldl, (int)N, B, ldb, (int)rows, vp);
    else if (rows == 2) tri_gemv_kernel<2><<<tg, 256, 0, h->stream>>>(Wf, h->ldl, (int)N, B, ldb, (int)rows, vp);
    else if (rows <= 4) tri_gemv_kernel<4><<<tg, 256, 0, h->stream>>>(Wf, h->ldl, (int)N, B, ldb, (int)rows, vp);
    else tri_gemv_kernel<8><<<tg, 256, 0, h->stream>>>(Wf, h->ldl, (int)N, B, ldb, (int)rows, vp);
    h->st.kernel_launches++;
    var_from_split_kernel<<<(unsigned)rows, 256, 0, h->stream>>>(kss, h->partial.as<double>(), (int)rows, (int)N, p.ktiles, p.ktiles, var);
  } else if (row_tiles * col_tiles < 4LL * h->sm_count) {
    // Few rows: a column tile near the end of the triangular product is one serial loop of up to N/16 k-tiles on ONE
    // SM while most of the GPU idles.  Split K into <= 8 chunks (grid z), keep the partial products of the valid rows
    // (rows x N x chunks doubles) and square / reduce them in a second, fixed-order kernel.
    int kchunk = 64;
    while ((p.ktiles + kchunk - 1) / kchunk > 8) kchunk *= 2;
    const int nz = (p.ktiles + kchunk - 1) / kchunk;
    p.kchunk = kchunk; p.vpart = h->partial.as<double>();
    CKR(launch_gemm<EPI_ROWDOT>(h, a, 0, 0, b, 0, 0, p, nz));
    var_from_split_kernel<<<(unsigned)rows, 256, 0, h->stream>>>(kss, h->partial.as<double>(), (int)rows, (int)N, p.ktiles, kchunk, var);
  } else {
    p.partial = h->partial.as<double>();
    CKR(launch_gemm<EPI_ROWDOT>(h, a, 0, 0, b, 0, 0, p));
    var_from_partial_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, h->stream>>>(kss, h->partial.as<double>(), col_tiles, (int)rows, var);
  }
  h->st.kernel_launches++;
  CK(cudaGetLastError());
  return NNGP_OK;
}

// ---- cfg.variance_slices: the variance product on the INT8 tensor cores (sliced_gemm.cuh) ---------------------
int get_tmap_u8(nngp_handle* h, const void* base, uint64_t rows, uint64_t ldq, uint32_t box_rows, CUtensorMap* out) {
  cuuint64_t gdim[2] = {ldq, rows};
  cuuint64_t gstride[1] = {ldq};
  cuuint32_t box[2] = {(cuuint32_t)SL_BK, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = h->encode(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(h, NNGP_ECUDA, "cuTensorMapEncodeTiled (digit planes) failed (CUresult %d; rows=%llu ld=%llu)", (int)r,
                (unsigned long long)rows, (unsigned long long)ldq);
  return NNGP_OK;
}

// digit planes of `rows` rows of A (columns [0, ncols), or [0, row] when tri) -> planes[s][rpad][ldq], row exponents exps[rows]
int slice_matrix(nngp_handle* h, const double* A, int64_t lda, int64_t rows, int64_t ncols, int tri, int s, int64_t rpad,
                 int64_t ldq, int8_t* planes, int* exps) {
  slice_rows_kernel<<<(unsigned)rpad, SL_SLICE_THREADS, 0, h->stream>>>(A, lda, (int)rows, (int)ncols, tri, s, planes,
                                                                       rpad * ldq, (int)ldq, exps);
  h->st.kernel_launches++;
  CK(cudaGetLastError());
  return NNGP_OK;
}

// int8 MACs the kernel issues for this shape (every supercolumn runs the K extent of its last column tile)
double sliced_macs(int64_t row_tiles, int64_t col_tiles, int64_t K, int tri, int s, int skip_weak) {
  double macs = 0.0;
  const int64_t nsup = (col_tiles + SL_SUPER - 1) / SL_SUPER;
  for (int64_t sup = 0; sup < nsup; ++sup) {
    const int64_t width = std::min<int64_t>(SL_SUPER, col_tiles - sup * SL_SUPER);
    const int64_t kext = tri ? std::min<int64_t>(K, std::min<int64_t>((sup + 1) * SL_SUPER, col_tiles) * SL_BN) : K;
    macs += (double)row_tiles * (double)width * (double)(SL_BM * SL_BN) * (double)round_up(kext, SL_BK);
  }
  return macs * (double)(s * (s + 1) / 2 - (skip_weak && s > 1 ? 1 : 0));
}

// V = A W^T from the digit planes: vpart[2 col_tiles][rows] row sums of V^2 per 128-column half tile and/or V itself
// (ra: rows per K_* plane, a multiple of 256)
int launch_sliced(nngp_handle* h, const int8_t* qa, int64_t ra, const int* ea, const int8_t* qw, int64_t rb,
                  const int* ew, int64_t ldq, int s, int tri, int64_t rows, int64_t N, int64_t K, double* vpart, double* V,
                  int64_t ldv, int skip_weak) {
  SlicedParams p{};
  p.s = s; p.rows = (int)rows; p.N = (int)N; p.K = (int)K; p.tri = tri; p.skip_weak = skip_weak;
  p.row_tiles = (int)((rows + SL_BM - 1) / SL_BM);
  p.col_tiles = (int)((N + SL_BN - 1) / SL_BN);
  p.ra = ra; p.rb = rb; p.rexp = ea; p.cexp = ew; p.vpart = vpart; p.V = V; p.ldv = ldv;
  if ((int64_t)s * ra >= (1LL << 31) || (int64_t)s * rb >= (1LL << 31))
    return fail(h, NNGP_EINVAL, "internal: digit-plane row range too large");
  // Two row tiles per CTA tile (SL_RT): 32 KiB of operands per MMA set instead of 48.  (Single row tiles -- twice as
  // many, lighter tiles -- were measured for small batches and lose: 1024 rows at N = 8192 take 1.82 ms instead of
  // 1.55 ms, the kernel is bound by bytes per MAC even there.)
  int grid;
  int64_t rounds;
  CKR(sliced_grid(h, rows, N, &grid, &rounds));
  p.scratch = h->slscratch.as<double>();
  CUtensorMap tmA, tmB;
  CKR(get_tmap_u8(h, qa, (uint64_t)s * ra, (uint64_t)ldq, SL_RT * SL_BM, &tmA));
  CKR(get_tmap_u8(h, qw, (uint64_t)s * rb, (uint64_t)ldq, SL_BN, &tmB));
  CK(cudaFuncSetAttribute(sliced_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SL_SMEM_BYTES));   // (per device)
  cudaLaunchConfig_t lc = {};
  cudaLaunchAttribute coop;
  coop.id = cudaLaunchAttributeCooperative;
  coop.val.cooperative = 1;
  lc.gridDim = dim3((unsigned)grid); lc.blockDim = dim3(SL_THREADS); lc.dynamicSmemBytes = SL_SMEM_BYTES;
  lc.stream = h->stream;
  // The wave re-alignment (wave_barrier, one counter per round of tiles) needs every CTA resident: a cooperative
  // launch.  With a single round there is nothing to re-align, and when the grid cannot be co-scheduled (another
  // context holds SMs) the launch is refused: then the CTAs run free.
  bool launched = false;
  if (rounds >= 2) {
    CK(cudaMemsetAsync(h->slsync.p, 0, (size_t)rounds * sizeof(int), h->stream));
    p.wave_sync = h->slsync.as<int>();
    lc.attrs = &coop; lc.numAttrs = 1;
    launched = cudaLaunchKernelEx(&lc, sliced_gemm_kernel, tmA, tmB, p) == cudaSuccess;
    if (!launched) cudaGetLastError();
  }
  if (!launched) {
    p.wave_sync = nullptr;
    lc.attrs = nullptr; lc.numAttrs = 0;
    if (cudaLaunchKernelEx(&lc, sliced_gemm_kernel, tmA, tmB, p) != cudaSuccess) {
      cudaGetLastError();
      return fail(h, NNGP_ECUDA, "sliced_gemm_kernel could not be launched");
    }
  }
  CK(cudaGetLastError());
  h->st.kernel_launches++;
  h->st.sliced_macs += sliced_macs(p.row_tiles, p.col_tiles, K, tri, s, skip_weak);
  return NNGP_OK;
}

// digit planes of W = L^-1, once per fit (and on every replica after the peer-to-peer copy)
int build_w_planes(nngp_handle* h) {
  const int s = h->cfg.variance_slices;
  const int64_t N = h->N;
  const int64_t ldq = round_up(N, SL_BK), rb = round_up(N, SL_BN);   // (Wq, wexp: sized by ensure_model)
  CKR(slice_matrix(h, h->Linvfull.as<double>(), h->ldl, N, N, 1, s, rb, ldq, h->Wq.as<int8_t>(), h->wexp.as<int>()));
  CK(cudaStreamSynchronize(h->stream));
  h->wq_ldq = ldq; h->wq_rb = rb; h->have_wq = true;
  return NNGP_OK;
}

// var[r] = kss[r] - |K_*[r,:] W^T|^2 with the product on the int8 tensor cores, in row sub-blocks of sliced_rows().
// The plane pair (s-1, 0) is dropped (SlicedParams::skip_weak).
int run_sliced_variance(nngp_handle* h, const double* B, int64_t ldb, int64_t rows, const double* kss, double* var) {
  const int s = h->cfg.variance_slices;
  const int64_t N = h->N, ldq = h->wq_ldq;
  const int col_tiles = (int)((N + SL_BN - 1) / SL_BN);
  const int64_t sb = sliced_rows(h, N, rows);
  CKR(ensure_sliced_block(h, N, rows));
  const int span = span_open(h, 0, h->stream, &h->st.sliced_ms);
  for (int64_t r0 = 0; r0 < rows; r0 += sb) {
    const int64_t nr = std::min<int64_t>(sb, rows - r0), ra = round_up(nr, SL_RT * SL_BM);
    CKR(slice_matrix(h, B + r0 * ldb, ldb, nr, N, 0, s, ra, ldq, h->Aq.as<int8_t>(), h->aexp.as<int>()));
    CKR(launch_sliced(h, h->Aq.as<int8_t>(), ra, h->aexp.as<int>(), h->Wq.as<int8_t>(), h->wq_rb,
                      h->wexp.as<int>(), ldq, s, 1, nr, N, N, h->partial.as<double>(), nullptr, 0, 1));
    var_from_partial_kernel<<<(unsigned)((nr + 255) / 256), 256, 0, h->stream>>>(kss + r0, h->partial.as<double>(), 2 * col_tiles, (int)nr, var + r0);
    h->st.kernel_launches++;
  }
  span_close(h, span);
  CK(cudaGetLastError());
  return NNGP_OK;
}

// out <- L^-T z  (blocked backward substitution; z is destroyed; reads L exactly once)
// (`Winv`: the inverses of L's 64 x 64 diagonal blocks, as the factorisation / run_trtri_diag leave them in h->Linv)
int run_trsv_bwd(nngp_handle* h, const double* L, int64_t ld, int64_t N, double* z, double* out, const double* Winv) {
  const int64_t nblk = (N + NB - 1) / NB;
  // one persistent launch: column slices of SW, one CTA each, all co-resident (grid <= #SMs)
  int64_t sw = 4 * NB;
  while ((N + sw - 1) / sw > h->sm_count) sw += NB;
  const int grid = (int)((N + sw - 1) / sw);
  const size_t smem = (size_t)(NB * (NB + 1) + 2 * NB + sw) * sizeof(double);
  if (smem <= 200 * 1024) {
    CKR(ensure_solve_workspace(h, N));
    CK(cudaMemsetAsync(h->sync_ints.p, 0, (size_t)nblk * sizeof(int), h->stream));
    CK(cudaFuncSetAttribute(trsv_bwd_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // The kernel's CTAs wait on each other's flags, so they must all be resident: a cooperative launch makes the
    // driver guarantee that (it waits for room when another handle or process holds SMs) instead of relying on
    // the dispatch order; if the grid cannot be co-resident at all the stepwise kernels below take over.
    int Ni = (int)N, swi = (int)sw;
    const double* zc = z;
    int* fl = h->sync_ints.as<int>();
    void* args[] = {(void*)&L, (void*)&ld, (void*)&Ni, (void*)&swi, (void*)&zc, (void*)&out, (void*)&fl, (void*)&Winv};
    cudaError_t le = cudaLaunchCooperativeKernel((const void*)trsv_bwd_persistent_kernel, dim3((unsigned)grid),
                                                 dim3(TRSVP_THREADS), args, smem, h->stream);
    if (le == cudaSuccess) {
      h->st.kernel_launches++;
      return NNGP_OK;
    }
    cudaGetLastError();   // not co-schedulable here: fall through to one launch per block
  }
  for (int64_t jb = nblk - 1; jb >= 0; --jb) {
    const int64_t j0 = jb * NB;
    const int64_t nb = std::min<int64_t>(NB, N - j0);
    const int sgrid = (int)std::min<int64_t>(std::max<int64_t>(1, (j0 + TRSV_THREADS - 1) / TRSV_THREADS), 4 * h->sm_count);
    trsv_bwd_step_kernel<<<sgrid, TRSV_THREADS, 0, h->stream>>>(L, ld, (int)j0, (int)nb, z, out);
    h->st.kernel_launches++;
  }
  CK(cudaGetLastError());
  return NNGP_OK;
}

// copy a caller matrix (host or device, dense rows x cols) into a padded device matrix (ld), zero pad
int upload_matrix(nngp_handle* h, const double* src, int64_t rows, int64_t cols, double* dst, int64_t ld,
                  cudaStream_t stream = nullptr) {
  if (!stream) stream = h->stream;
  if (ld != cols) CK(cudaMemsetAsync(dst, 0, (size_t)rows * ld * sizeof(double), stream));
  const bool dev = is_device_ptr(src);   // (possibly memory of another GPU: the kind is resolved through UVA)
  CK(cudaMemcpy2DAsync(dst, ld * sizeof(double), src, cols * sizeof(double), cols * sizeof(double), rows,
                       cudaMemcpyDefault, stream));
  if (!dev) h->st.h2d_bytes += rows * cols * (int64_t)sizeof(double);
  return NNGP_OK;
}
int download(nngp_handle* h, const double* dsrc, int64_t rows, int64_t cols, int64_t ld, double* dst) {
  const bool dev = is_device_ptr(dst);
  CK(cudaMemcpy2DAsync(dst, cols * sizeof(double), dsrc, ld * sizeof(double), cols * sizeof(double), rows,
                       cudaMemcpyDefault, h->stream));
  if (!dev) h->st.d2h_bytes += rows * cols * (int64_t)sizeof(double);
  return NNGP_OK;
}

// flags[1] |= bit when a value of x is not finite: bit 1 for caller input, FLAG_ALPHA for the solved alpha
constexpr int FLAG_ALPHA = 4;
int check_finite_async(nngp_handle* h, const double* x, int64_t ld, int64_t rows, int64_t cols, int bit = 1) {
  const int64_t total = rows * cols;
  int grid = (int)std::min<int64_t>((total + 255) / 256, 8 * h->sm_count);
  if (grid < 1) grid = 1;
  finite_check_kernel<<<grid, 256, 0, h->stream>>>(x, ld, rows, (int)cols, h->flags.as<int>() + 1, bit);
  h->st.kernel_launches++;
  return NNGP_OK;
}

// flags[1] after check_finite_async (bit 0) and row_sqnorm_kernel with range_flag (bit 1) -> the caller's error
int input_error(nngp_handle* h, int flag, const char* who, const char* what) {
  if (flag & 1) return fail(h, NNGP_EINVAL, "%s: non-finite value in %s", who, what);
  if (h->act.kind != ACT_RELU)
    return fail(h, NNGP_EINVAL,
                "%s: %s out of range: a row's layer-0 kernel diagonal q = sigma_w^2 |x|^2 / D + sigma_b^2 must stay below "
                "%.17g (every layer's diagonal below 2^512; Erf: b^2 q below 2^508)", who, what, h->q_limit);
  return fail(h, NNGP_EINVAL,
              "%s: %s out of range: a row's layer-0 kernel diagonal sigma_w^2 |x|^2 / D + sigma_b^2 reaches 2^512 "
              "(the kernel needs q q' < 2^1024)", who, what);
}

// Every call that reads `flags` back runs between begin_call and end_call.  begin_call clears the flags and discards
// whatever spans a failed earlier call left behind, so their time is charged to no later call.  No call may run
// another begin_call inside while it has spans open.
int begin_call(nngp_handle* h) {
  discard_spans(h);
  CK(cudaMemsetAsync(h->flags.p, 0, 2 * sizeof(int), h->stream));
  return NNGP_OK;
}

// Enqueues the flags read-back (after the caller's own), waits for the main stream and settles the spans.  flags[1]
// becomes input_error(who, what); flags[0], the potrf pivot + 1 (0: none), goes to *pivot; FLAG_ALPHA of a factor
// without a failed pivot means that alpha = (K + lambda I)^-1 y overflowed (lambda near the bottom of the normal
// range against O(1) labels): an error, not a model whose means are inf or NaN.
int end_call(nngp_handle* h, const char* who, const char* what, int* pivot = nullptr) {
  int flags[2];
  CK(cudaMemcpyAsync(flags, h->flags.p, sizeof flags, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaGetLastError());
  settle_spans(h);
  if (pivot) *pivot = flags[0];
  if (flags[1] & ~FLAG_ALPHA) return input_error(h, flags[1], who, what);
  if ((flags[1] & FLAG_ALPHA) && !flags[0])
    return fail(h, NNGP_EINVAL, "%s: alpha = (K + lambda I)^-1 y overflows the double range (lambda = %.6g): scale y "
                "down or raise diag_reg", who, h->lambda);
  return NNGP_OK;
}

// Rows [new0, rows) of X are new input: check them finite, and derive q of all `rows` rows with the range flag.
// Both report in flags[1], which the caller reads back and turns into input_error.
int derive_q(nngp_handle* h, int64_t rows, int64_t new0) {
  const double* X = h->X.as<double>();
  CKR(check_finite_async(h, X + new0 * h->ldx, h->ldx, rows - new0, h->D));
  row_sqnorm_kernel<<<(unsigned)((rows * 32 + 255) / 256), 256, 0, h->stream>>>(X, h->ldx, (int)rows, (int)h->D, h->lsw2[0], h->lsb2[0], h->q.as<double>(), h->flags.as<int>() + 1, h->q_limit);
  h->st.kernel_launches++;
  return NNGP_OK;
}

int bind_device(nngp_handle* h) {
  CK(cudaSetDevice(h->device));
  return NNGP_OK;
}

void drop_fit(nngp_handle* h) { h->importing = false; h->have_inv = false; h->have_wq = false; h->fitted = false; h->have_labels = false; h->have_M = false; }

// Start installing a fitted state of N x D on h: bind its device, drop the fitted state of h and its replicas, size
// the model buffers.
int begin_state(nngp_handle* h, int64_t N, int64_t D) {
  CKR(bind_device(h));
  drop_fit(h);
  for (auto* p : h->peers) drop_fit(p);
  h->N = N; h->D = D;
  h->ldx = round_up(D, 2);
  h->ldl = round_up(N, 16);
  return ensure_model(h, N, D);
}

// inv(L_JJ) for all diagonal blocks of the factor in h->L (after a factorisation or an imported state)
int run_trtri_diag(nngp_handle* h) {
  const int nblk = (int)((h->N + NB - 1) / NB);
  trtri_diag_kernel<<<nblk, POTF2_THREADS, 0, h->stream>>>(h->L.as<double>(), h->ldl, (int)h->N, h->Linv.as<double>());
  h->st.kernel_launches++;
  CK(cudaGetLastError());
  return NNGP_OK;
}


// ---- replicas (cfg.n_gpus > 1) ------------------------------------------------------------------
// After every successful fit / append / import the fitted state {X, q, alpha, inv(L_JJ), lower triangle of L
// (+ M in 'ntk' mode)} is copied to the replicas, device to device over NVLink (peer access is enabled at
// nngp_create), as a pipelined chain  d0 -> d1 -> ... -> d(G-1):  the factor travels in row panels
// [r0, r1) x [0, r1) -- only the lower trapezoid, half the bytes of the square -- and hop g forwards panel c as soon
// as it has arrived (event), so every link carries a different panel at the same time and the whole replication
// costs about one transfer of the packed factor, independent of G (NVSwitch gives every hop full bandwidth).
// Copies are pushed from the source GPU's copy stream.  No host staging, no extra device buffers.
int replicate_state(nngp_handle* h) {
  if (h->peers.empty() || !h->fitted) return NNGP_OK;
  const int64_t N = h->N, D = h->D, ldx = h->ldx, ldl = h->ldl;
  const auto t_begin = std::chrono::steady_clock::now();
  std::vector<nngp_handle*> chain;
  chain.push_back(h);
  for (auto* p : h->peers) chain.push_back(p);
  const int G = (int)chain.size();
  for (int g = 1; g < G; ++g) {
    nngp_handle* p = chain[g];
    const int rc = begin_state(p, N, D);
    if (rc != NNGP_OK) { h->err = "replica on device " + std::to_string(p->device) + ": " + p->err; cudaSetDevice(h->device); return rc; }
  }
  const int64_t RP = 512;                       // rows per panel
  const int npanel = (int)((N + RP - 1) / RP);
  // items in chain order: 0 = small vectors (X, q, alpha, Linv), 1..npanel = factor panels, then M panels
  const int nM = h->have_M ? npanel : 0;
  const int nI = h->have_inv ? npanel : 0;          // latency mode: the explicit inverse (lower trapezoids, like L)
  const int nitems = 1 + npanel + nM + nI;
  std::vector<std::vector<cudaEvent_t>> ev((size_t)G);   // ev[g][i]: item i has arrived on chain[g]
  cudaError_t ce = cudaSuccess;
  auto copy_item = [&](nngp_handle* src, nngp_handle* dst, int item, cudaStream_t st) -> cudaError_t {
    cudaError_t e = cudaSuccess;
    if (item == 0) {
      e = cudaMemcpyAsync(dst->X.p, src->X.p, (size_t)N * ldx * 8, cudaMemcpyDefault, st);
      if (e == cudaSuccess) e = cudaMemcpyAsync(dst->q.p, src->q.p, (size_t)N * 8, cudaMemcpyDefault, st);
      if (e == cudaSuccess) e = cudaMemcpyAsync(dst->alpha.p, src->alpha.p, (size_t)N * 8, cudaMemcpyDefault, st);
      if (e == cudaSuccess) e = cudaMemcpyAsync(dst->Linv.p, src->Linv.p, (size_t)round_up(N, NB) * NB * 8, cudaMemcpyDefault, st);
      return e;
    }
    const int which = item <= npanel ? 0 : (item <= npanel + nM ? 1 : 2);     // 0: L, 1: M, 2: L^-1
    const bool isM = which == 1;
    const int64_t r0 = (int64_t)((item - 1) % npanel) * RP;
    const int64_t r1 = std::min<int64_t>(r0 + RP, N);
    const DevBuf& sb = which == 0 ? src->L : (which == 1 ? src->Mmat : src->Linvfull);
    const DevBuf& db = which == 0 ? dst->L : (which == 1 ? dst->Mmat : dst->Linvfull);
    const double* sp = sb.as<double>() + r0 * ldl;
    double* dp = db.as<double>() + r0 * ldl;
    const int64_t width = isM ? N : r1;        // the factors: columns [0, r1) of these rows; M: whole rows
    return cudaMemcpy2DAsync(dp, ldl * 8, sp, ldl * 8, (size_t)width * 8, (size_t)(r1 - r0), cudaMemcpyDefault, st);
  };
  for (int g = 0; g + 1 < G && ce == cudaSuccess; ++g) {
    nngp_handle* src = chain[g];
    nngp_handle* dst = chain[g + 1];
    ce = cudaSetDevice(src->device);
    cudaStream_t st = src->copy_stream;
    ev[(size_t)g + 1].resize((size_t)nitems);
    for (int i = 0; i < nitems && ce == cudaSuccess; ++i) {
      if (g > 0) ce = cudaStreamWaitEvent(st, ev[(size_t)g][(size_t)i], 0);   // item i has reached src
      if (ce == cudaSuccess) ce = copy_item(src, dst, i, st);
      cudaEvent_t e = nullptr;
      if (ce == cudaSuccess) {   // events are kept on the source handle and reused by the next replication
        if (!src->rep_events.empty()) { e = src->rep_events.back(); src->rep_events.pop_back(); }
        else ce = cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
      }
      if (ce == cudaSuccess) { ev[(size_t)g + 1][(size_t)i] = e; ce = cudaEventRecord(e, st); }
    }
  }
  for (int g = 0; g + 1 < G; ++g) {
    cudaSetDevice(chain[g]->device);
    cudaError_t e2 = cudaStreamSynchronize(chain[g]->copy_stream);
    if (ce == cudaSuccess) ce = e2;
  }
  for (size_t g = 1; g < ev.size(); ++g)       // ev[g] was recorded on chain[g - 1]'s stream (same device)
    for (auto e : ev[g]) if (e) chain[g - 1]->rep_events.push_back(e);
  cudaSetDevice(h->device);
  if (ce != cudaSuccess) return fail(h, NNGP_ECUDA, "replicating the fitted state to the other GPUs failed: %s", cudaGetErrorString(ce));
  for (int g = 1; g < G; ++g) {
    nngp_handle* p = chain[g];
    p->lambda = h->lambda; p->fitted = true; p->have_M = h->have_M; p->have_inv = h->have_inv;
    if (h->have_wq) {          // each replica splits its own copy of L^-1 (a few ms) instead of receiving s more planes
      cudaSetDevice(p->device);
      const int rc = build_w_planes(p);
      cudaSetDevice(h->device);
      if (rc != NNGP_OK) { h->err = "replica on device " + std::to_string(p->device) + ": " + p->err; return rc; }
    }
  }
  h->st.replicate_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
  int64_t bytes = (int64_t)N * ldx * 8 + 2 * N * 8 + round_up(N, NB) * NB * 8;
  int64_t bytes_tri = 0;
  for (int c = 0; c < npanel; ++c) {
    const int64_t r0 = (int64_t)c * RP, r1 = std::min<int64_t>(r0 + RP, N);
    bytes_tri += (r1 - r0) * r1 * 8;
  }
  bytes += bytes_tri;
  if (nM) bytes += N * N * 8;
  if (nI) bytes += bytes_tri;
  h->st.replicate_bytes = bytes;
  return NNGP_OK;
}

// The common tail of every call that installs a fitted state (the factor, alpha, inv(L_JJ) and, as `have_M` says, M
// are on the device and the flags have been read back): mark it fitted, build the explicit inverse in latency mode and
// copy the state to the replicas.  `labels`: the state was fitted from labels on this handle.
int publish_state(nngp_handle* h, bool labels, bool have_M) {
  h->fitted = true;
  h->have_labels = labels;
  h->have_M = have_M;
  if (builds_inverse(h)) CKR(build_inverse(h));
  return replicate_state(h);
}

// ---- posterior variance and covariance of a prediction block ---------------------------------------------------
// The posterior variance of one block of `rows` rows of a T-row batch (blk: K_*, 'ntk': Theta_*; blk2: K_* ('ntk');
// kss: K(x,x)), by the path chosen for that T.  nngp_predict and nngp_predict_cov both take it, so the covariance's
// diagonal is bitwise the variance.  *solved: blk now holds V = blk L^-T ('ntk': also blk2 holds U = K_* L^-T) --
// the latency-mode and digit-plane paths never write V.
int block_variance(nngp_handle* h, int64_t T, int64_t rows, double* var, bool* solved) {
  const int64_t N = h->N, ldl = h->ldl;
  double* blk = h->blk.as<double>();
  const double* L = h->L.as<double>();
  const double* kss = h->kss.as<double>();
  *solved = true;
  const int trsm = span_open(h, 1, h->stream, &h->st.pred_trsm_ms);
  if (h->cfg.kernel_type == 1) {
    // var_i = K_ii + v_i^T M v_i - 2 v_i . u_i,  v_i = L^-1 theta_i, u_i = L^-1 k_i, M = L^-1 K_dd L^-T
    double* blk2 = h->blk2.as<double>();
    CKR(run_predict_solve(h, blk, ldl, rows, L, ldl, N, nullptr, nullptr));    // V
    CKR(run_predict_solve(h, blk2, ldl, rows, L, ldl, N, nullptr, nullptr));   // U
    span_close(h, trsm);
    const int vs = span_open(h, 1, h->stream, &h->st.pred_var_ms);
    rowdot_kernel<<<(unsigned)((rows * 32 + 255) / 256), 256, 0, h->stream>>>(blk, blk2, ldl, (int)rows, (int)N, h->cross.as<double>());
    CKR(run_gemm_rowdot(h, blk, ldl, rows, h->Mmat.as<double>(), N, h->partial.as<double>()));
    ntk_var_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, h->stream>>>(kss, h->partial.as<double>(), (int)((N + GEMM_BN - 1) / GEMM_BN), (int)rows, h->cross.as<double>(), var);
    h->st.kernel_launches += 2;
    span_close(h, vs);
    return NNGP_OK;
  }
  if (T <= latency_rows(h)) {                      // latency mode, small batch: dependency-free product with L^-1
    *solved = false;
    CKR(run_inverse_variance(h, blk, ldl, rows, kss, var));
  } else if (h->have_wq) {                         // variance_slices: the same product on the int8 tensor cores
    *solved = false;
    CKR(run_sliced_variance(h, blk, ldl, rows, kss, var));
  } else {                                         // solve + variance in one persistent kernel
    CKR(run_predict_solve(h, blk, ldl, rows, L, ldl, N, kss, var));
  }
  span_close(h, trsm);
  return NNGP_OK;
}

// The T x T posterior covariance of a batch that is one prediction block, after block_variance (var: its variance):
// xt / qt hold the batch, blk (blk2) V (U) unless !solved.  Lower tiles only (the full square below 4 row tiles, as
// nngp_kernel), then one kernel mirrors them and installs `var` on the diagonal.  Every product is an EPI_SUB launch
// of the DMMA core with K = round_up(N, 16); the columns past N are the tensor maps' zero fill (MatView cols = N).
//   'nngp': C = K(X*,X*) - V V^T
//   'ntk' : P = -V M (M symmetric: P -= V M^T on P = 0), C = K(X*,X*) - P V^T - U V^T - V U^T
int block_covariance(nngp_handle* h, int64_t T, bool solved, const double* var, double* C, int64_t ldc) {
  const int64_t N = h->N, D = h->D, ldl = h->ldl, K = round_up(N, GEMM_BK);
  double* blk = h->blk.as<double>();
  double* xt = h->xt.as<double>();
  const double* qt = h->qt.as<double>();
  if (!solved) {
    const int trsm = span_open(h, 1, h->stream, &h->st.pred_trsm_ms);
    CKR(run_predict_solve(h, blk, ldl, T, h->L.as<double>(), ldl, N, nullptr, nullptr));
    span_close(h, trsm);
  }
  const int lower = T >= 4 * GEMM_BM ? 1 : 0;
  const int gram = span_open(h, 1, h->stream, &h->st.pred_gram_ms);
  CKR(run_gram(h, xt, h->ldx, T, qt, xt, h->ldx, T, qt, D, C, ldc, lower, nullptr, nullptr, nullptr, true));
  span_close(h, gram);
  const int vs = span_open(h, 1, h->stream, &h->st.pred_var_ms);
  const MatView Vv{blk, T, N, ldl};
  if (h->cfg.kernel_type == 1) {
    double* P = h->covP.as<double>();
    const MatView Uv{h->blk2.as<double>(), T, N, ldl}, Pv{P, T, N, ldl}, Mv{h->Mmat.as<double>(), N, N, ldl};
    CK(cudaMemsetAsync(P, 0, (size_t)T * ldl * sizeof(double), h->stream));
    CKR(run_gemm_sub(h, Vv, 0, 0, Mv, 0, 0, T, N, K, P, ldl, 0));
    CKR(run_gemm_sub(h, Pv, 0, 0, Vv, 0, 0, T, T, K, C, ldc, 1));
    CKR(run_gemm_sub(h, Uv, 0, 0, Vv, 0, 0, T, T, K, C, ldc, 1));
    CKR(run_gemm_sub(h, Vv, 0, 0, Uv, 0, 0, T, T, K, C, ldc, 1));
  } else {
    CKR(run_gemm_sub(h, Vv, 0, 0, Vv, 0, 0, T, T, K, C, ldc, 1));
  }
  const dim3 mg((unsigned)((T + 31) / 32), (unsigned)((T + 31) / 32));
  mirror_lower_kernel<<<mg, dim3(32, 8), 0, h->stream>>>(C, ldc, (int)T, var);
  h->st.kernel_launches++;
  span_close(h, vs);
  CK(cudaGetLastError());
  return NNGP_OK;
}

}  // namespace

// =================================================================================================
extern "C" {

int nngp_abi_version(void) { return NNGP_B200_ABI_VERSION; }

void nngp_default_config(nngp_config* cfg) {
  if (!cfg) return;
  memset(cfg, 0, sizeof *cfg);
  cfg->depth = 2;
  cfg->sigma_w = 1.0;
  cfg->sigma_b = 0.0;
  cfg->diag_reg = 1e-3;
  cfg->diag_reg_absolute = 0;
  cfg->device = -1;
  cfg->max_block_bytes = 0;
  cfg->stats_level = 1;
  cfg->kernel_type = 0;
}

const char* nngp_last_error(const nngp_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

// Checks the activation of a new handle (cfg already checked) and derives its step coefficients and the limit of the
// layer-0 diagonals (nngp_activation in the header).  NULL / NNGP_ACT_RELU: ReLU, the limit 2^512.
static int make_act_coef(const nngp_config* cfg, const nngp_activation* act, ActCoef* c, double* q_limit) {
  const double inv_2pi = 0.15915494309189533577, two_over_pi = 0.63661977236758134308;
  *c = ActCoef{};
  c->kind = ACT_RELU; c->c0 = 0.5; c->c1 = inv_2pi;
  *q_limit = Q_LIMIT;
  if (!act || act->kind == NNGP_ACT_RELU) return NNGP_OK;
  const char* who = "nngp_create_with_activation";
  if (act->kind != NNGP_ACT_ABRELU && act->kind != NNGP_ACT_ERF)
    return fail(nullptr, NNGP_EINVAL, "%s: unknown activation kind %d (NNGP_ACT_RELU, _ABRELU or _ERF)", who, act->kind);
  const double a = act->a, b = act->b, cc = act->c;
  if (!std::isfinite(a) || !std::isfinite(b) || !std::isfinite(cc))
    return fail(nullptr, NNGP_EINVAL, "%s: a, b and c must be finite (got %g, %g, %g)", who, a, b, cc);
  if (act->kind == NNGP_ACT_ABRELU) {
    c->kind = ACT_ABRELU;
    c->c0 = (a * a + b * b) * 0.5;
    c->c1 = (a - b) * (a - b) * inv_2pi;
    if (!std::isfinite(c->c0) || !std::isfinite(c->c1))
      return fail(nullptr, NNGP_EINVAL, "%s: ABRelu(%g, %g): a^2 + b^2 overflows", who, a, b);
    // Every step forms q q', so the diagonal entering each step must stay below 2^512 like the layer-0 one.  Later
    // diagonals are q_l = sigma_w_l^2 c0 q_(l-1) + sigma_b_l^2: carry that bound back to a limit on the layer-0 q.
    double lim = Q_LIMIT;
    for (int l = cfg->depth - 1; l >= 1; --l) {
      const double w = cfg->per_layer ? cfg->sigma_w_layers[l] : cfg->sigma_w;
      const double sb = cfg->per_layer ? cfg->sigma_b_layers[l] : cfg->sigma_b;
      lim = std::min(Q_LIMIT, (lim - sb * sb) / (w * w * c->c0));
      if (!(lim > 0.0))
        return fail(nullptr, NNGP_EINVAL, "%s: ABRelu(%g, %g): the diagonal of Dense layer %d reaches 2^512 for every "
                    "input", who, a, b, l);
    }
    *q_limit = lim;
    return NNGP_OK;
  }
  const double b2 = b * b;
  if (!(b2 >= DBL_MIN) || !std::isfinite(b2))
    return fail(nullptr, NNGP_EINVAL, "%s: Erf needs b != 0 with b^2 a finite normal double (got b = %g)", who, b);
  c->kind = ACT_ERF;
  c->b2x2 = 2.0 * b2;
  c->e = a * a * two_over_pi;
  c->c2 = cc * cc;
  c->kd = a * a * b2 * (2.0 * two_over_pi);
  if (!std::isfinite(c->e) || !std::isfinite(c->c2) || !std::isfinite(c->kd))
    return fail(nullptr, NNGP_EINVAL, "%s: Erf(%g, %g, %g): a^2, c^2 or a^2 b^2 overflows", who, a, b, cc);
  *q_limit = std::min(Q_LIMIT, ERF_Q_LIMIT / b2);
  // the diagonal entering every later step is sigma_w^2 E[phi^2] + sigma_b^2 <= sigma_w^2 (a^2 + c^2) + sigma_b^2
  for (int l = 1; l < std::min(cfg->depth, NNGP_MAX_LAYERS); ++l) {
    const double w = cfg->per_layer ? cfg->sigma_w_layers[l] : cfg->sigma_w;
    const double sb = cfg->per_layer ? cfg->sigma_b_layers[l] : cfg->sigma_b;
    const double bound = w * w * (a * a + cc * cc) + sb * sb;
    if (!(bound < Q_LIMIT) || !(b2 * bound < ERF_Q_LIMIT))
      return fail(nullptr, NNGP_EINVAL, "%s: Erf(%g, %g, %g): the diagonal of Dense layer %d can reach %g; it needs "
                  "b^2 q < 2^508", who, a, b, cc, l, bound);
  }
  return NNGP_OK;
}

static int create_single(const nngp_config* cfg, const nngp_activation* act, nngp_handle** out) {
  nngp_handle* h = nullptr;
  if (!cfg || !out) return fail(h, NNGP_EINVAL, "nngp_create: null argument");
  *out = nullptr;
  if (cfg->depth < 1) return fail(h, NNGP_EINVAL, "nngp_create: depth must be >= 1 (got %d)", cfg->depth);
  if (cfg->kernel_type != 0 && cfg->kernel_type != 1)
    return fail(h, NNGP_EINVAL, "nngp_create: kernel_type must be 0 (nngp) or 1 (ntk)");
  if (!(cfg->sigma_w > 0.0) || !(cfg->sigma_b >= 0.0) || !(cfg->diag_reg >= 0.0))
    return fail(h, NNGP_EINVAL, "nngp_create: need sigma_w > 0, sigma_b >= 0, diag_reg >= 0");
  if (cfg->per_layer) {
    if (cfg->depth > NNGP_MAX_LAYERS)
      return fail(h, NNGP_EINVAL, "nngp_create: per-layer sigmas support at most %d Dense layers (depth=%d)", NNGP_MAX_LAYERS, cfg->depth);
    for (int l = 0; l < cfg->depth; ++l)
      if (!(cfg->sigma_w_layers[l] > 0.0) || !(cfg->sigma_b_layers[l] >= 0.0))
        return fail(h, NNGP_EINVAL, "nngp_create: layer %d needs sigma_w > 0, sigma_b >= 0", l);
  }
  ActCoef coef;
  double q_limit;
  CKR(make_act_coef(cfg, act, &coef, &q_limit));
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(h, NNGP_ENODEV, "nngp_create: no CUDA device visible (this library has no CPU path)");
  }
  int dev = cfg->device;
  if (dev < 0) { if (cudaGetDevice(&dev) != cudaSuccess) dev = 0; }
  if (dev >= ndev) return fail(h, NNGP_ENODEV, "nngp_create: device %d out of range (%d visible)", dev, ndev);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess)
    return fail(h, NNGP_ECUDA, "nngp_create: cudaGetDeviceProperties failed");
  if (prop.major != 10)
    return fail(h, NNGP_ENODEV, "nngp_create: device %d is sm_%d%d; this library is built for sm_100a only", dev,
                prop.major, prop.minor);
  if (cfg->variance_slices != 0 && (cfg->variance_slices < 5 || cfg->variance_slices > SL_MAX_SLICES))
    return fail(h, NNGP_EINVAL, "nngp_create: variance_slices must be 0 (off) or 5..%d (got %d)", SL_MAX_SLICES,
                cfg->variance_slices);
  if (cfg->variance_slices != 0 && cfg->kernel_type != 0)
    return fail(h, NNGP_EINVAL, "nngp_create: variance_slices applies to kernel_type 0 ('nngp') only");
  nngp_handle* nh = new nngp_handle();
  nh->cfg = *cfg;
  nh->act = coef;
  nh->q_limit = q_limit;
  if (nh->cfg.variance_slices > 0) nh->cfg.latency_mode = 1;   // the digit planes are those of the explicit inverse
  for (int l = 0; l < NNGP_MAX_LAYERS; ++l) {
    const int ll = std::min(l, std::max(cfg->depth - 1, 0));
    const double w = cfg->per_layer ? cfg->sigma_w_layers[ll] : cfg->sigma_w;
    const double b = cfg->per_layer ? cfg->sigma_b_layers[ll] : cfg->sigma_b;
    nh->lsw2[l] = w * w;
    nh->lsb2[l] = b * b;
  }
  if (nh->cfg.max_block_bytes <= 0) nh->cfg.max_block_bytes = (int64_t)32 << 30;
  nh->device = dev;
  nh->sm_count = prop.multiProcessorCount;
  memset(&nh->st, 0, sizeof nh->st);
  h = nh;
  auto bail = [&](int code) { std::string m = h->err; nngp_destroy(h); g_create_error = m; return code; };
  if (cudaSetDevice(dev) != cudaSuccess) { fail(h, NNGP_ECUDA, "cudaSetDevice(%d) failed", dev); return bail(NNGP_ECUDA); }
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  if (cudaStreamCreateWithPriority(&h->stream, cudaStreamNonBlocking, prio_lo) != cudaSuccess ||
      cudaStreamCreateWithPriority(&h->panel_stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) {
    fail(h, NNGP_ECUDA, "cudaStreamCreate failed");
    return bail(NNGP_ECUDA);
  }
  h->cur = h->stream;
  if (cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking) != cudaSuccess) {
    fail(h, NNGP_ECUDA, "cudaStreamCreate failed");
    return bail(NNGP_ECUDA);
  }
  // Look-ahead can be switched off (see run_potrf): with NNGP_CHOL_LOOKAHEAD=0 the panel stream is not kept.
  {
    const char* e = getenv("NNGP_CHOL_LOOKAHEAD");
    if (e && !strcmp(e, "0")) { cudaStreamDestroy(h->panel_stream); h->panel_stream = nullptr; }
  }
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn ||
      qres != cudaDriverEntryPointSuccess) {
    fail(h, NNGP_ECUDA, "cuTensorMapEncodeTiled not available from the driver");
    return bail(NNGP_ECUDA);
  }
  h->encode = reinterpret_cast<PFN_encodeTiled>(fn);
  cudaError_t e1 = cudaFuncSetAttribute(gemm_nt_kernel<EPI_GRAM>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES);
  if (e1 == cudaSuccess) e1 = cudaFuncSetAttribute(gemm_nt_kernel<EPI_GRAM, ACT_ABRELU>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES);
  if (e1 == cudaSuccess) e1 = cudaFuncSetAttribute(gemm_nt_kernel<EPI_GRAM, ACT_ERF>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES);
  cudaError_t e2 = cudaFuncSetAttribute(gemm_nt_kernel<EPI_SUB>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES);
  if (e2 == cudaSuccess) e2 = cudaFuncSetAttribute(gemm_nt_kernel<EPI_ROWDOT>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES);
  cudaError_t e3 = cudaFuncSetAttribute(trsm_fused_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TF_SMEM_BYTES);
  if (e3 == cudaSuccess) e3 = cudaFuncSetAttribute(trsm_fused_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TF_SMEM_BYTES);
  if (e3 == cudaSuccess) e3 = cudaFuncSetAttribute(gemm_nt_kernel<EPI_DIAG>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES);
  if (e3 == cudaSuccess) e3 = cudaFuncSetAttribute(potrf_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TF_SMEM_BYTES);
  if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) {
    fail(h, NNGP_ECUDA, "cudaFuncSetAttribute(max dynamic smem) failed: %s",
         cudaGetErrorString(e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3)));
    return bail(NNGP_ECUDA);
  }
  if (ensure(h, h->flags, 2 * sizeof(int)) != NNGP_OK || ensure(h, h->lam_d, 4 * sizeof(double)) != NNGP_OK)
    return bail(NNGP_ENOMEM);
  cudaMemsetAsync(h->flags.p, 0, 2 * sizeof(int), h->stream);
  cudaStreamSynchronize(h->stream);
  *out = h;
  return NNGP_OK;
}

int nngp_create(const nngp_config* cfg, nngp_handle** out) { return nngp_create_with_activation(cfg, nullptr, out); }

int nngp_create_with_activation(const nngp_config* cfg, const nngp_activation* act, nngp_handle** out) {
  nngp_handle* h = nullptr;
  if (!cfg || !out) return fail(h, NNGP_EINVAL, "nngp_create: null argument");
  *out = nullptr;
  const int G = cfg->n_gpus <= 1 ? 1 : cfg->n_gpus;
  if (G > NNGP_MAX_GPUS) return fail(h, NNGP_EINVAL, "nngp_create: n_gpus=%d exceeds NNGP_MAX_GPUS=%d", G, NNGP_MAX_GPUS);
  nngp_config c0 = *cfg;
  c0.n_gpus = 1;
  if (G == 1) return create_single(&c0, act, out);
  int ids[NNGP_MAX_GPUS];
  bool any = false;
  for (int g = 0; g < G; ++g) any = any || cfg->device_ids[g] >= 0;
  for (int g = 0; g < G; ++g) ids[g] = any ? cfg->device_ids[g] : g;
  for (int g = 0; g < G; ++g)
    for (int k = 0; k < g; ++k)
      if (ids[g] == ids[k] || ids[g] < 0)
        return fail(h, NNGP_EINVAL, "nngp_create: device_ids must be %d distinct CUDA ordinals", G);
  c0.device = ids[0];
  CKR(create_single(&c0, act, &h));
  for (int g = 1; g < G; ++g) {
    nngp_config cg = c0;
    cg.device = ids[g];
    nngp_handle* p = nullptr;
    const int rc = create_single(&cg, act, &p);
    if (rc != NNGP_OK) { nngp_destroy(h); return rc; }   // g_create_error holds the message
    p->owner = h;
    h->peers.push_back(p);
  }
  h->cfg.n_gpus = G;
  for (int g = 0; g < G; ++g) h->cfg.device_ids[g] = ids[g];
  // peer access both ways between every pair: the replication chain pushes over NVLink, and a replica may read test
  // rows from / write results to device memory of the first GPU
  for (int a = 0; a < G; ++a) {
    for (int b = 0; b < G; ++b) {
      if (a == b) continue;
      int can = 0;
      cudaDeviceCanAccessPeer(&can, ids[a], ids[b]);
      if (!can) {
        fail(nullptr, NNGP_ENODEV, "nngp_create: GPU %d cannot access GPU %d peer-to-peer", ids[a], ids[b]);
        nngp_destroy(h);
        return NNGP_ENODEV;
      }
      cudaSetDevice(ids[a]);
      cudaError_t e = cudaDeviceEnablePeerAccess(ids[b], 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
        fail(nullptr, NNGP_ECUDA, "cudaDeviceEnablePeerAccess(%d -> %d) failed: %s", ids[a], ids[b], cudaGetErrorString(e));
        nngp_destroy(h);
        return NNGP_ECUDA;
      }
      cudaGetLastError();
    }
  }
  cudaSetDevice(ids[0]);
  *out = h;
  return NNGP_OK;
}

int nngp_num_gpus(const nngp_handle* h) { return h ? 1 + (int)h->peers.size() : 0; }

// sum_t partial[t][r] in tile order (the order the variance uses)
static __global__ void rowsq_from_partial_kernel(const double* __restrict__ partial, int tiles, int rows, double* __restrict__ out) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  double q = 0.0;
  for (int t = 0; t < tiles; ++t) q += partial[(long long)t * rows + r];
  out[r] = q;
}

int nngp_sliced_product(nngp_handle* h, const double* a, int64_t M, int64_t K, const double* b, int64_t N, int32_t lower,
                        int32_t slices, double* v_out, double* rowsq_out) {
  if (!h) return NNGP_EINVAL;
  if (!a || !b || (!v_out && !rowsq_out) || M <= 0 || K <= 0 || N <= 0)
    return fail(h, NNGP_EINVAL, "nngp_sliced_product: bad argument (M=%lld K=%lld N=%lld)", (long long)M, (long long)K, (long long)N);
  if (slices < 1 || slices > SL_MAX_SLICES) return fail(h, NNGP_EINVAL, "nngp_sliced_product: slices must be 1..%d", SL_MAX_SLICES);
  if (lower && N != K) return fail(h, NNGP_EINVAL, "nngp_sliced_product: a triangular B must be square (N=%lld K=%lld)", (long long)N, (long long)K);
  const int64_t ldq = round_up(K, SL_BK), ra = round_up(M, SL_RT * SL_BM), rb = round_up(N, SL_BN);
  if ((int64_t)slices * 4096 * ldq >= (1LL << 31)) return fail(h, NNGP_EINVAL, "nngp_sliced_product: K too large for int32 plane sums");
  CKR(bind_device(h));
  const int col_tiles = (int)(rb / SL_BN);
  DevBuf dA, dB, qa, qb, sa, sb, dV, vp, rs;
  auto cleanup = [&]() { for (DevBuf* x : {&dA, &dB, &qa, &qb, &sa, &sb, &dV, &vp, &rs}) release(*x); };
  int rc = ensure(h, dA, (size_t)M * K * 8);
  if (rc == NNGP_OK) rc = ensure(h, dB, (size_t)N * K * 8);
  if (rc == NNGP_OK) rc = ensure(h, qa, (size_t)slices * ra * ldq);
  if (rc == NNGP_OK) rc = ensure(h, qb, (size_t)slices * rb * ldq);
  if (rc == NNGP_OK) rc = ensure(h, sa, (size_t)M * sizeof(int));
  if (rc == NNGP_OK) rc = ensure(h, sb, (size_t)N * sizeof(int));
  if (rc == NNGP_OK && v_out) rc = ensure(h, dV, (size_t)M * N * 8);
  if (rc == NNGP_OK) rc = ensure(h, vp, (size_t)2 * col_tiles * M * 8);
  if (rc == NNGP_OK) rc = ensure(h, rs, (size_t)M * 8);
  auto run = [&]() -> int {
    CK(cudaMemcpyAsync(dA.p, a, (size_t)M * K * 8, cudaMemcpyDefault, h->stream));
    CK(cudaMemcpyAsync(dB.p, b, (size_t)N * K * 8, cudaMemcpyDefault, h->stream));
    CKR(slice_matrix(h, dA.as<double>(), K, M, K, 0, slices, ra, ldq, qa.as<int8_t>(), sa.as<int>()));
    CKR(slice_matrix(h, dB.as<double>(), K, N, K, lower ? 1 : 0, slices, rb, ldq, qb.as<int8_t>(), sb.as<int>()));
    CKR(launch_sliced(h, qa.as<int8_t>(), ra, sa.as<int>(), qb.as<int8_t>(), rb, sb.as<int>(), ldq, slices, lower ? 1 : 0,
                      M, N, K, vp.as<double>(), v_out ? dV.as<double>() : nullptr, N, lower == 2 ? 1 : 0));
    if (v_out) CK(cudaMemcpyAsync(v_out, dV.p, (size_t)M * N * 8, cudaMemcpyDefault, h->stream));
    if (rowsq_out) {
      rowsq_from_partial_kernel<<<(unsigned)((M + 255) / 256), 256, 0, h->stream>>>(vp.as<double>(), 2 * col_tiles, (int)M, rs.as<double>());
      CK(cudaMemcpyAsync(rowsq_out, rs.p, (size_t)M * 8, cudaMemcpyDefault, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    return NNGP_OK;
  };
  if (rc == NNGP_OK) rc = run();
  cleanup();
  return rc;
}

#ifndef NNGP_BUILD_ID
#define NNGP_BUILD_ID "unknown"
#endif
// "nngp-build-id:<16 hex>" is also what the Python loader scans the file for before loading it
static const char g_build_marker[] = "nngp-build-id:" NNGP_BUILD_ID;
const char* nngp_build_id(void) { return g_build_marker + 14; }

void nngp_destroy(nngp_handle* h) {
  if (!h) return;
  for (auto* p : h->peers) nngp_destroy(p);
  h->peers.clear();
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  for (DevBuf* b : {&h->X, &h->q, &h->L, &h->alpha, &h->flags, &h->lam_d, &h->xt, &h->qt, &h->kss,
                    &h->blk, &h->mean_d, &h->var_d, &h->ssq, &h->sync_ints, &h->Mmat, &h->Kdd, &h->blk2, &h->cov, &h->covP, &h->cross, &h->partial, &h->mean_partial, &h->ka, &h->kb, &h->kqa, &h->kqb, &h->kout, &h->qtab, &h->stage, &h->Linv, &h->Linvfull, &h->panel_inv, &h->panel_sync, &h->zkeep, &h->L2, &h->y, &h->app_x, &h->app_y, &h->sel_mean, &h->sel_var, &h->sel_score, &h->sel_key,
                    &h->sel_state, &h->sel_okey, &h->sel_oidx, &h->sel_max, &h->Wq, &h->wexp, &h->Aq, &h->aexp, &h->slscratch, &h->slsync})
    release(*b);
  discard_spans(h);
  for (auto e : h->ev_pool) cudaEventDestroy(e);
  for (auto e : h->rep_events) cudaEventDestroy(e);
  if (h->panel_stream) cudaStreamDestroy(h->panel_stream);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

void* nngp_get_stream(nngp_handle* h) { return h ? (void*)h->stream : nullptr; }

int nngp_stats(nngp_handle* h, nngp_stats_t* out) {
  if (!h || !out) return NNGP_EINVAL;
  *out = h->st;   // stage / kernel-class times: the first GPU's; counters: summed over the handle's GPUs
  for (auto* p : h->peers) {
    out->kernel_launches += p->st.kernel_launches;
    out->h2d_bytes += p->st.h2d_bytes;
    out->d2h_bytes += p->st.d2h_bytes;
    out->gemm_launches += p->st.gemm_launches;
    out->gram_launches += p->st.gram_launches;
    out->device_allocs += p->st.device_allocs;
  }
  return NNGP_OK;
}
int nngp_stats_reset(nngp_handle* h) {
  if (!h) return NNGP_EINVAL;
  memset(&h->st, 0, sizeof h->st);
  for (auto* p : h->peers) memset(&p->st, 0, sizeof p->st);
  return NNGP_OK;
}

// -------------------------------------------------------------------------------------------------
int nngp_kernel(nngp_handle* h, const double* x1, int64_t M, const double* x2, int64_t N2, int64_t D, double* k_out) {
  if (!h) return NNGP_EINVAL;
  if (!x1 || !k_out || M <= 0 || D <= 0 || (x2 && N2 <= 0))
    return fail(h, NNGP_EINVAL, "nngp_kernel: bad argument (M=%lld N2=%lld D=%lld)", (long long)M, (long long)N2, (long long)D);
  CKR(bind_device(h));
  const int64_t Nn = x2 ? N2 : M;
  if (M > 65535LL * GEMM_BM || Nn > 0x7fffffffLL || D > 0x7fffffffLL)
    return fail(h, NNGP_EINVAL, "nngp_kernel: shape too large for one call");
  const int64_t ldx = round_up(D, 2), ldo = round_up(Nn, 2);
  const double sw2 = h->lsw2[0], sb2 = h->lsb2[0];   // first Dense layer
  CKR(ensure(h, h->ka, (size_t)M * ldx * 8));
  CKR(ensure(h, h->kqa, (size_t)M * 8));
  CKR(ensure(h, h->kout, (size_t)M * ldo * 8));
  CKR(ensure_act_tables(h, x2 ? M + Nn : M));
  CKR(begin_call(h));
  CKR(upload_matrix(h, x1, M, D, h->ka.as<double>(), ldx));
  CKR(check_finite_async(h, h->ka.as<double>(), ldx, M, D));
  row_sqnorm_kernel<<<(unsigned)((M * 32 + 255) / 256), 256, 0, h->stream>>>(h->ka.as<double>(), ldx, (int)M, (int)D, sw2, sb2, h->kqa.as<double>(), h->flags.as<int>() + 1, h->q_limit);
  h->st.kernel_launches++;
  const double* bptr = h->ka.as<double>();
  const double* qb = h->kqa.as<double>();
  if (x2) {
    CKR(ensure(h, h->kb, (size_t)Nn * ldx * 8));
    CKR(ensure(h, h->kqb, (size_t)Nn * 8));
    CKR(upload_matrix(h, x2, Nn, D, h->kb.as<double>(), ldx));
    CKR(check_finite_async(h, h->kb.as<double>(), ldx, Nn, D));
    row_sqnorm_kernel<<<(unsigned)((Nn * 32 + 255) / 256), 256, 0, h->stream>>>(h->kb.as<double>(), ldx, (int)Nn, (int)D, sw2, sb2, h->kqb.as<double>(), h->flags.as<int>() + 1, h->q_limit);
    h->st.kernel_launches++;
    bptr = h->kb.as<double>();
    qb = h->kqb.as<double>();
  }
  // kernel_fn(x, None) is symmetric: compute the tiles at / below the diagonal only and mirror them (NNGP mode; the
  // entries are bitwise symmetric anyway -- same products, same summation order).  'ntk' keeps the full square.
  const bool sym = !x2 && h->cfg.kernel_type == 0 && M >= 4 * GEMM_BM;
  CKR(run_gram(h, h->ka.as<double>(), ldx, M, h->kqa.as<double>(), bptr, ldx, Nn, qb, D, h->kout.as<double>(), ldo, sym ? 1 : 0));
  if (sym) {
    dim3 mg((unsigned)((M + 31) / 32), (unsigned)((M + 31) / 32));
    mirror_lower_kernel<<<mg, dim3(32, 8), 0, h->stream>>>(h->kout.as<double>(), ldo, (int)M, nullptr);
    h->st.kernel_launches++;
  }
  CKR(download(h, h->kout.as<double>(), M, Nn, ldo, k_out));
  return end_call(h, "nngp_kernel", "the inputs");
}

// -------------------------------------------------------------------------------------------------
static int fit_impl(nngp_handle* h, const double* x_train, const double* y_train, int64_t N, int64_t D);
int nngp_fit(nngp_handle* h, const double* x_train, const double* y_train, int64_t N, int64_t D) {
  if (!h) return NNGP_EINVAL;
  CKR(fit_impl(h, x_train, y_train, N, D));
  return publish_state(h, true, h->cfg.kernel_type == 1);
}

static int fit_impl(nngp_handle* h, const double* x_train, const double* y_train, int64_t N, int64_t D) {
  if (!x_train || !y_train || N <= 0 || D <= 0)
    return fail(h, NNGP_EINVAL, "nngp_fit: bad argument (N=%lld D=%lld)", (long long)N, (long long)D);
  if (N > 65535LL * GEMM_BM || D > 0x7fffffffLL) return fail(h, NNGP_EINVAL, "nngp_fit: N=%lld too large", (long long)N);
  CKR(begin_state(h, N, D));
  CKR(ensure_fit_workspace(h, N));
  double* X = h->X.as<double>();
  double* L = h->L.as<double>();
  double* alpha = h->alpha.as<double>();
  double* q = h->q.as<double>();

  CKR(begin_call(h));
  const int total = span_open(h, 1, h->stream, &h->st.fit_total_ms), h2d = span_open(h, 1, h->stream, &h->st.h2d_ms);
  CKR(upload_matrix(h, x_train, N, D, X, h->ldx));
  CKR(upload_matrix(h, y_train, N, 1, alpha, 1));
  CK(cudaMemcpyAsync(h->y.p, alpha, (size_t)N * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  span_close(h, h2d);
  CKR(check_finite_async(h, alpha, 1, N, 1));

  const int gram = span_open(h, 1, h->stream, &h->st.fit_gram_ms);
  CKR(derive_q(h, N, 0));
  const bool ntk = h->cfg.kernel_type == 1;
  if (!ntk) {
    CKR(run_gram(h, X, h->ldx, N, q, X, h->ldx, N, q, D, L, h->ldl, 1));
  } else {  // NTK: Theta_dd (to be factored) -> L, the full symmetric K_dd -> Kdd (for M = L^-1 K_dd L^-T)
    CKR(run_gram(h, X, h->ldx, N, q, X, h->ldx, N, q, D, L, h->ldl, 0, h->Kdd.as<double>()));
  }
  diag_reg_kernel<<<1, 1024, 0, h->stream>>>(L, h->ldl, (int)N, h->cfg.diag_reg, h->cfg.diag_reg_absolute, h->lam_d.as<double>());
  h->st.kernel_launches++;
  span_close(h, gram);

  const int chol = span_open(h, 1, h->stream, &h->st.fit_chol_ms);
  // y^T goes into row N of the factor buffer: the factorisation turns it into z^T = (L^-1 y)^T
  CK(cudaMemcpyAsync(L + N * h->ldl, alpha, (size_t)N * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  CKR(run_potrf(h, L, h->ldl, N, 1, h->Linv.as<double>()));   // also leaves inv(L_JJ) of every diagonal block in Linv
  span_close(h, chol);

  const int solve = span_open(h, 1, h->stream, &h->st.fit_solve_ms);
  lml_terms_kernel<<<1, 1024, 0, h->stream>>>(L, h->ldl, (int)N, L + N * h->ldl, h->lam_d.as<double>() + 1);
  h->st.kernel_launches++;
  CK(cudaMemcpyAsync(h->zkeep.p, L + N * h->ldl, (size_t)N * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  CKR(run_trsv_bwd(h, L, h->ldl, N, L + N * h->ldl, alpha, h->Linv.as<double>()));  // alpha = L^-T z
  CKR(check_finite_async(h, alpha, 1, N, 1, FLAG_ALPHA));
  if (ntk) {  // M = L^-1 K_dd L^-T : two row-wise solves around a transpose (M is symmetric)
    double* Kd = h->Kdd.as<double>();
    double* Mm = h->Mmat.as<double>();
    CKR(run_predict_solve(h, Kd, h->ldl, N, L, h->ldl, N, nullptr, nullptr));   // Kd <- K_dd L^-T
    dim3 tg((unsigned)((N + 31) / 32), (unsigned)((N + 31) / 32));
    transpose_kernel<<<tg, dim3(32, 8), 0, h->stream>>>(Kd, Mm, h->ldl, (int)N);
    h->st.kernel_launches++;
    CKR(run_predict_solve(h, Mm, h->ldl, N, L, h->ldl, N, nullptr, nullptr));   // Mm <- (L^-1 K_dd L^-T)^T = M
  }
  span_close(h, solve);
  span_close(h, total);

  CK(cudaMemcpyAsync(&h->lambda, h->lam_d.p, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(h->lml_terms, h->lam_d.as<double>() + 1, 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  int pivot = 0;
  CKR(end_call(h, "nngp_fit", "x_train / y_train", &pivot));
  if (pivot)
    return fail(h, NNGP_ENOTPD, "nngp_fit: K + lambda*I is not positive definite (pivot %d of %lld, lambda=%.6g)",
                pivot - 1, (long long)N, h->lambda);
  return NNGP_OK;
}

// -------------------------------------------------------------------------------------------------
// Active-learning step (SURVEY 8f-3).  Selection: active/ActiveLearner.py:43-55; merge + refit: :57-65, :76.
int nngp_active_select(nngp_handle* h, const double* x_pool, int64_t T, int64_t budget, int32_t mode, uint64_t seed,
                       int64_t* idx_out, int64_t* n_selected_out, double* score_out) {
  if (!h) return NNGP_EINVAL;
  if (!h->fitted) return fail(h, NNGP_ESTATE, "nngp_active_select: no fitted model");
  if (!x_pool || !idx_out || T <= 0 || budget <= 0 || (mode != NNGP_SELECT_TOPK && mode != NNGP_SELECT_SAMPLE))
    return fail(h, NNGP_EINVAL, "nngp_active_select: bad argument (T=%lld budget=%lld mode=%d)", (long long)T, (long long)budget, mode);
  if (T > 0xffffffffLL) return fail(h, NNGP_EINVAL, "nngp_active_select: T=%lld exceeds 2^32-1 rows", (long long)T);
  CKR(bind_device(h));
  const int64_t k = budget < T ? budget : T;   // num_select = budget if num_test > budget else num_test
  CKR(ensure_select_workspace(h, T, k));
  // posterior mean / variance of the pool, left on the device (outputs are device pointers)
  CKR(nngp_predict(h, x_pool, T, h->sel_mean.as<double>(), h->sel_var.as<double>()));

  SelectState init;
  memset(&init, 0, sizeof init);
  init.k_remaining = k;
  SelectState* st = h->sel_state.as<SelectState>();
  CK(cudaMemcpyAsync(st, &init, sizeof init, cudaMemcpyHostToDevice, h->stream));
  max_reduce_kernel<<<1, 1024, 0, h->stream>>>(h->sel_mean.as<double>(), (long long)T, h->sel_max.as<double>());
  const unsigned gridT = (unsigned)((T + 255) / 256);
  unsigned long long* key = h->sel_key.as<unsigned long long>();
  score_key_kernel<<<gridT, 256, 0, h->stream>>>(h->sel_var.as<double>(), h->sel_max.as<double>(), (long long)T, mode,
                                                 (unsigned long long)seed, h->sel_score.as<double>(), key, st);
  const int hist_grid = (int)std::min<int64_t>(gridT, 4 * h->sm_count);
  for (int pass = 0; pass < 12; ++pass) {
    select_hist_kernel<<<hist_grid, 256, 0, h->stream>>>(key, (long long)T, pass, st);
    select_pick_kernel<<<1, 1, 0, h->stream>>>(pass, st);
  }
  select_compact_kernel<<<gridT, 256, 0, h->stream>>>(key, (long long)T, st, h->sel_okey.as<unsigned long long>(),
                                                      h->sel_oidx.as<unsigned int>());
  h->st.kernel_launches += 3 + 24;
  // the k winners come back (16 B each) and are put in argsort order on the host
  std::vector<unsigned long long> okey((size_t)k);
  std::vector<unsigned int> oidx((size_t)k);
  SelectState fin;
  CK(cudaMemcpyAsync(&fin, st, sizeof fin, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(okey.data(), h->sel_okey.p, (size_t)k * 8, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(oidx.data(), h->sel_oidx.p, (size_t)k * 4, cudaMemcpyDeviceToHost, h->stream));
  if (score_out) CKR(download(h, h->sel_score.as<double>(), T, 1, 1, score_out));
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaGetLastError());
  if (fin.out_count != (unsigned int)k)
    return fail(h, NNGP_ECUDA, "nngp_active_select: internal error, selected %u of %lld rows", fin.out_count, (long long)k);
  if (mode == NNGP_SELECT_SAMPLE && fin.bad)
    return fail(h, NNGP_EINVAL, "nngp_active_select: sampling needs finite, non-negative scores std/max(mean)");
  std::vector<int64_t> order((size_t)k);
  for (int64_t i = 0; i < k; ++i) order[(size_t)i] = i;
  const bool ascending = mode == NNGP_SELECT_TOPK;   // argsort tail: ascending; Gumbel-top-k: best first
  std::sort(order.begin(), order.end(), [&](int64_t a, int64_t b) {
    const bool less = okey[(size_t)a] != okey[(size_t)b] ? okey[(size_t)a] < okey[(size_t)b] : oidx[(size_t)a] < oidx[(size_t)b];
    return ascending ? less : (a != b && !less);
  });
  std::vector<int64_t> out((size_t)k);
  for (int64_t i = 0; i < k; ++i) out[(size_t)i] = (int64_t)oidx[(size_t)order[(size_t)i]];
  CK(cudaMemcpy(idx_out, out.data(), (size_t)k * sizeof(int64_t), cudaMemcpyDefault));
  if (n_selected_out) *n_selected_out = k;
  return NNGP_OK;
}

int nngp_reserve(nngp_handle* h, int64_t n_train_max, int64_t dim, int64_t n_test_max) {
  if (!h) return NNGP_EINVAL;
  if (n_train_max <= 0 || dim <= 0 || n_test_max < 0 || n_train_max > 65535LL * GEMM_BM)
    return fail(h, NNGP_EINVAL, "nngp_reserve: bad argument (n_train_max=%lld dim=%lld n_test_max=%lld)",
                (long long)n_train_max, (long long)dim, (long long)n_test_max);
  CKR(bind_device(h));
  const int64_t N = n_train_max, D = dim, T = n_test_max;
  drop_fit(h);   // growing a buffer does not keep its contents
  CKR(ensure_fit_workspace(h, N));
  CKR(ensure_append_workspace(h, N, D));
  if (T > 0) CKR(ensure_select_workspace(h, T, T));
  // the model and the predict workspace on every GPU; a replica predicts its share of the rows (nngp_predict)
  const int G = 1 + (int)h->peers.size();
  for (int g = 0; g < G; ++g) {
    nngp_handle* p = g == 0 ? h : h->peers[(size_t)g - 1];
    const int64_t Tg = g == 0 || T == 0 ? T : (T + G - 1) / G + 1;
    CK(cudaSetDevice(p->device));
    drop_fit(p);
    int rc = ensure_model(p, N, D);
    for (bool want_var : {false, true})
      if (rc == NNGP_OK && Tg > 0) rc = ensure_predict_workspace(p, N, D, Tg, want_var);
    if (rc != NNGP_OK) {
      if (p != h) h->err = "replica on device " + std::to_string(p->device) + ": " + p->err;
      cudaSetDevice(h->device);
      return rc;
    }
  }
  if (G > 1) CK(cudaSetDevice(h->device));
  return NNGP_OK;
}

// Fixed-lambda append (cfg.diag_reg_absolute): extend the factor instead of refactoring.  With A' = [[A, K21^T],
// [K21, K22 + lambda I]] and A = L11 L11^T:   L21 = K21 L11^-T (the prediction solve),  L22 L22^T = K22 + lambda I
// - L21 L21^T (Gram + one SYRK-shaped GEMM + a Cholesky of the M x M Schur complement),  z' = [z; L22^-1 (y_new -
// L21 z)] (the y row rides through that small Cholesky as in the full fit), alpha' = L'^-T z'.  N^2 M + M^3/3 flop
// instead of (N+M)^3/3.  Exact in exact arithmetic; in FP64 it agrees with a fresh fit to rounding (tested), not
// bitwise.  Not applicable to the reference's relative diag_reg: there lambda = 1e-3 tr(K)/N moves with every row.
// On entry X/y staging holds [X; X_new], [y; y_new]; h->L, h->Linv, h->zkeep describe the old N-row model, and L2 and
// panel_inv are sized for Nn rows (ensure_append_workspace).
static int append_incremental(nngp_handle* h, int64_t M) {
  const int64_t N = h->N, D = h->D, Nn = N + M;
  const int64_t ldo = h->ldl, ldn = round_up(Nn, 16);
  drop_fit(h);   // a half-extended model is not a model (nngp_append_fit publishes the extended one)
  CKR(begin_call(h));
  const int total = span_open(h, 1, h->stream, &h->st.fit_total_ms);
  double* Ln = h->L2.as<double>();
  // old factor (lower part incl. diagonal blocks) and old z into the new pitch
  CK(cudaMemcpy2DAsync(Ln, ldn * sizeof(double), h->L.p, ldo * sizeof(double), (size_t)N * sizeof(double), N,
                       cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaMemsetAsync(Ln + Nn * ldn, 0, (size_t)ldn * sizeof(double), h->stream));
  CK(cudaMemcpyAsync(Ln + Nn * ldn, h->zkeep.p, (size_t)N * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  CK(cudaMemcpyAsync(Ln + Nn * ldn + N, h->app_y.as<double>() + N, (size_t)M * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  // X, y, q for all Nn rows (the staging buffers are contiguous).  The old X, y and z are in the staging and in Ln now,
  // so their buffers may grow; the rest of the model grows only after the L21 solve has read the old inv(L_JJ).
  CKR(ensure_fit_workspace(h, Nn));
  CKR(ensure_inputs(h, Nn, D));
  double* X = h->X.as<double>();
  double* q = h->q.as<double>();
  CKR(upload_matrix(h, h->app_x.as<double>(), Nn, D, X, h->ldx));
  CK(cudaMemcpyAsync(h->y.p, h->app_y.p, (size_t)Nn * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  CKR(derive_q(h, Nn, N));
  CKR(check_finite_async(h, h->y.as<double>() + N, 1, M, 1));

  const int gram = span_open(h, 1, h->stream, &h->st.fit_gram_ms);
  double* L21 = Ln + N * ldn;        // rows N..Nn-1, columns 0..N-1
  double* S = Ln + N * ldn + N;      // the Schur complement block
  CKR(run_gram(h, X + N * h->ldx, h->ldx, M, q + N, X, h->ldx, N, q, D, L21, ldn, 0));                     // K21
  CKR(run_gram(h, X + N * h->ldx, h->ldx, M, q + N, X + N * h->ldx, h->ldx, M, q + N, D, S, ldn, 1));       // K22 (lower)
  diag_reg_kernel<<<1, 1024, 0, h->stream>>>(S, ldn, (int)M, h->cfg.diag_reg, 1, h->lam_d.as<double>());
  h->st.kernel_launches++;
  span_close(h, gram);

  const int chol = span_open(h, 1, h->stream, &h->st.fit_chol_ms);
  CKR(run_predict_solve(h, L21, ldn, M, Ln, ldn, N, nullptr, nullptr));                                    // L21 = K21 L11^-T
  {  // [S; y_new^T] -= [L21; z^T] L21^T   (K = N, zero-filled up to a multiple of 16 by the tensor map bounds)
    MatView Av{Ln, Nn + 1, N, ldn};
    CKR(run_gemm_sub(h, Av, N, 0, Av, N, 0, M + 1, M, round_up(N, GEMM_BK), S, ldn, 1));
  }
  // (panel_inv: inverses on the Schur block's own 64-grid)
  CKR(run_potrf(h, S, ldn, M, 1, h->panel_inv.as<double>()));                                              // L22, z_new
  // from here on the handle describes the extended model
  std::swap(h->L, h->L2);
  h->N = Nn; h->ldl = ldn;
  CKR(ensure_model(h, Nn, D));   // (the old inverses are no longer needed)
  CKR(run_trtri_diag(h));
  span_close(h, chol);

  const int solve = span_open(h, 1, h->stream, &h->st.fit_solve_ms);
  double* zrow = Ln + Nn * ldn;
  lml_terms_kernel<<<1, 1024, 0, h->stream>>>(Ln, ldn, (int)Nn, zrow, h->lam_d.as<double>() + 1);
  h->st.kernel_launches++;
  CK(cudaMemcpyAsync(h->zkeep.p, zrow, (size_t)Nn * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  CKR(run_trsv_bwd(h, Ln, ldn, Nn, zrow, h->alpha.as<double>(), h->Linv.as<double>()));
  CKR(check_finite_async(h, h->alpha.as<double>(), 1, Nn, 1, FLAG_ALPHA));
  span_close(h, solve);
  span_close(h, total);

  CK(cudaMemcpyAsync(h->lml_terms, h->lam_d.as<double>() + 1, 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  int pivot = 0;
  CKR(end_call(h, "nngp_append_fit", "x_new / y_new", &pivot));
  if (pivot)
    return fail(h, NNGP_ENOTPD, "nngp_append_fit: the extended K + lambda*I is not positive definite (pivot %lld of %lld)",
                (long long)(N + pivot - 1), (long long)Nn);
  return NNGP_OK;
}

int nngp_append_fit(nngp_handle* h, const double* x_new, const double* y_new, int64_t M) {
  if (!h) return NNGP_EINVAL;
  if (!h->fitted || !h->have_labels)
    return fail(h, NNGP_ESTATE, "nngp_append_fit: needs a model fitted by nngp_fit on this handle (the labels are kept there)");
  if (!x_new || !y_new || M <= 0) return fail(h, NNGP_EINVAL, "nngp_append_fit: bad argument (M=%lld)", (long long)M);
  CKR(bind_device(h));
  const int64_t N = h->N, D = h->D;
  // [X_old; x_new], [y_old; y_new] contiguous on the device, then an ordinary fit from device pointers
  DevBuf& xc = h->app_x;
  DevBuf& yc = h->app_y;
  int rc = ensure_append_workspace(h, N + M, D);
  auto body = [&]() -> int {
    CK(cudaMemcpy2DAsync(xc.p, D * sizeof(double), h->X.p, h->ldx * sizeof(double), D * sizeof(double), N,
                         cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaMemcpyAsync(yc.p, h->y.p, (size_t)N * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    CKR(upload_matrix(h, x_new, M, D, xc.as<double>() + N * D, D));
    CKR(upload_matrix(h, y_new, M, 1, yc.as<double>() + N, 1));
    CK(cudaStreamSynchronize(h->stream));
    // fixed lambda: extend the factor (NNGP_APPEND_INCREMENTAL=0 forces the full refit, e.g. for A/B runs)
    const char* inc = getenv("NNGP_APPEND_INCREMENTAL");
    // (an odd N would put the Schur block at an 8-byte-aligned column: TMA bases and the double2 epilogues need 16)
    if (can_append_incrementally(h) && N % 2 == 0 && !(inc && !strcmp(inc, "0"))) return append_incremental(h, M);
    return fit_impl(h, xc.as<double>(), yc.as<double>(), N + M, D);
  };
  for (auto* p : h->peers) drop_fit(p);
  if (rc == NNGP_OK) rc = body();
  if (rc == NNGP_OK) rc = publish_state(h, true, h->cfg.kernel_type == 1);
  return rc;
}

// -------------------------------------------------------------------------------------------------
static int predict_impl(nngp_handle* h, const double* x_test, int64_t T, double* mean_out, double* var_out,
                        double* cov_out = nullptr);

// cfg.n_gpus > 1: rows [g*T/G, (g+1)*T/G) go to GPU g (SURVEY 8e); the replicas run on one host thread each while the
// calling thread drives the first GPU.  Rows are independent and every reduction has a fixed order, so the result
// is bitwise the single-GPU result.  Small batches (fewer than one 128-row tile per GPU) stay on the first GPU.
int nngp_predict(nngp_handle* h, const double* x_test, int64_t T, double* mean_out, double* var_out) {
  if (!h) return NNGP_EINVAL;
  const int G = 1 + (int)h->peers.size();
  if (G == 1 || T < (int64_t)G * GEMM_BM) return predict_impl(h, x_test, T, mean_out, var_out);
  if (!h->fitted) return fail(h, NNGP_ESTATE, "nngp_predict: no fitted model (call nngp_fit or nngp_set_state)");
  if (!x_test || !mean_out || T <= 0) return fail(h, NNGP_EINVAL, "nngp_predict: bad argument (T=%lld)", (long long)T);
  const int64_t D = h->D;
  std::vector<int> rcs((size_t)G, NNGP_OK);
  std::vector<std::thread> workers;
  auto shard = [&](int g) {
    nngp_handle* hg = g == 0 ? h : h->peers[(size_t)g - 1];
    const int64_t lo = (int64_t)g * T / G, hi = (int64_t)(g + 1) * T / G;
    rcs[(size_t)g] = predict_impl(hg, x_test + lo * D, hi - lo, mean_out + lo, var_out ? var_out + lo : nullptr);
  };
  int started = 1;
  try {
    for (int g = 1; g < G; ++g) { workers.emplace_back(shard, g); started = g + 1; }
  } catch (...) {   // (no exception may cross the C ABI) a worker thread could not be created: its shard runs here
  }
  shard(0);
  for (int g = started; g < G; ++g) shard(g);
  for (auto& w : workers) w.join();
  cudaSetDevice(h->device);
  for (int g = 1; g < G; ++g)
    if (rcs[(size_t)g] != NNGP_OK) {
      h->err = "GPU " + std::to_string(h->peers[(size_t)g - 1]->device) + ": " + h->peers[(size_t)g - 1]->err;
      return rcs[(size_t)g];
    }
  if (rcs[0] != NNGP_OK) return rcs[0];
  for (auto* p : h->peers) { h->st.queries += p->st.queries; p->st.queries = 0; }
  return NNGP_OK;
}

// cov_out (nngp_predict_cov, which has checked that T rows are one block): also the T x T posterior covariance.
static int predict_impl(nngp_handle* h, const double* x_test, int64_t T, double* mean_out, double* var_out,
                        double* cov_out) {
  if (!h->fitted) return fail(h, NNGP_ESTATE, "nngp_predict: no fitted model (call nngp_fit or nngp_set_state)");
  if (!x_test || !mean_out || T <= 0) return fail(h, NNGP_EINVAL, "nngp_predict: bad argument (T=%lld)", (long long)T);
  const bool want_var = var_out != nullptr || cov_out != nullptr;
  if (h->cfg.kernel_type == 1 && want_var && !h->have_M)
    return fail(h, NNGP_ESTATE, "nngp_predict: this imported 'ntk' state has no M yet (nngp_set_state_ntk_m) -- the variance needs it");
  CKR(bind_device(h));
  const int64_t N = h->N, D = h->D, ldx = h->ldx, ldl = h->ldl;
  const double sw2 = h->lsw2[0], sb2 = h->lsb2[0];   // first Dense layer

  const bool ntk = h->cfg.kernel_type == 1;
  const int64_t TB = predict_block_rows(h, N, T, want_var);
  const int col_tiles = (int)((N + GEMM_BN - 1) / GEMM_BN);
  CKR(ensure_predict_workspace(h, N, D, T, want_var));
  if (cov_out) CKR(ensure_cov_workspace(h, N, T));
  CKR(begin_call(h));

  double* xt = h->xt.as<double>();
  double* blk = h->blk.as<double>();
  const int total = span_open(h, 1, h->stream, &h->st.pred_total_ms);
  // ev_landed: a chunk is on the device (one event serves every chunk: a stream wait binds the record before it)
  cudaEvent_t ev_landed = call_event(h), ev_xt_free = nullptr;
  for (int64_t t0 = 0; t0 < T; t0 += TB) {
    const int64_t rows = std::min<int64_t>(TB, T - t0);
    // Upload and Gram are pipelined in chunks of CH rows: the copy stream runs ahead, the main stream starts the
    // Gram of a chunk as soon as that chunk has landed -- H2D (and, for pageable host memory, the driver's staging
    // memcpy, which blocks this thread, not the GPU) hides behind the Gram of the previous chunk.  Rows are
    // independent, so chunking does not change a bit of the result.
    const int64_t CH = 16384;
    const int nchunks = (int)((rows + CH - 1) / CH);
    if (ev_xt_free) CK(cudaStreamWaitEvent(h->copy_stream, ev_xt_free, 0));   // previous block's Gram has read xt
    const int h2d = span_open(h, 1, h->copy_stream, &h->st.h2d_ms);
    const int gram = span_open(h, 1, h->stream, &h->st.pred_gram_ms);
    for (int c = 0; c < nchunks; ++c) {
      const int64_t c0 = (int64_t)c * CH, cr = std::min<int64_t>(CH, rows - c0);
      CKR(upload_matrix(h, x_test + (t0 + c0) * D, cr, D, xt + c0 * ldx, ldx, h->copy_stream));
      CK(cudaEventRecord(ev_landed, h->copy_stream));
      CK(cudaStreamWaitEvent(h->stream, ev_landed, 0));
      CKR(check_finite_async(h, xt + c0 * ldx, ldx, cr, D));
      double* qt_c = h->qt.as<double>() + c0;
      double* mp_c = h->mean_partial.as<double>() + c0 * 2 * col_tiles;
      row_sqnorm_kernel<<<(unsigned)((cr * 32 + 255) / 256), 256, 0, h->stream>>>(xt + c0 * ldx, ldx, (int)cr, (int)D, sw2, sb2, qt_c, h->flags.as<int>() + 1, h->q_limit);
      h->st.kernel_launches++;
      CKR(run_gram(h, xt + c0 * ldx, ldx, cr, qt_c, h->X.as<double>(), ldx, N, h->q.as<double>(), D, blk + c0 * ldl, ldl, 0,
                   (ntk && want_var) ? h->blk2.as<double>() + c0 * ldl : nullptr, h->alpha.as<double>(), mp_c));
      mean_reduce_kernel<<<(unsigned)((cr + 255) / 256), 256, 0, h->stream>>>(mp_c, 2 * col_tiles, (int)cr, h->mean_d.as<double>() + t0 + c0);
      h->st.kernel_launches++;
    }
    span_close(h, gram);
    span_close(h, h2d);
    if (!ev_xt_free) ev_xt_free = call_event(h);
    CK(cudaEventRecord(ev_xt_free, h->stream));   // the next block's upload may overlap this block's solve

    if (want_var) {
      q_final_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, h->stream>>>(h->qt.as<double>(), (int)rows, h->cfg.depth - 1, layer_sig(h), h->act, nullptr, h->kss.as<double>());
      h->st.kernel_launches++;
      bool solved = false;
      CKR(block_variance(h, T, rows, h->var_d.as<double>() + t0, &solved));
      if (cov_out) CKR(block_covariance(h, T, solved, h->var_d.as<double>(), h->cov.as<double>(), round_up(T, 2)));
    }
  }
  const int d2h = span_open(h, 1, h->stream, &h->st.d2h_ms);
  CKR(download(h, h->mean_d.as<double>(), T, 1, 1, mean_out));
  if (var_out) CKR(download(h, h->var_d.as<double>(), T, 1, 1, var_out));
  if (cov_out) CKR(download(h, h->cov.as<double>(), T, T, round_up(T, 2), cov_out));
  span_close(h, d2h);
  span_close(h, total);
  CKR(end_call(h, cov_out ? "nngp_predict_cov" : "nngp_predict", "x_test"));
  h->st.queries += T;
  return NNGP_OK;
}

// The covariance couples every pair of rows, so it is not sharded: on a handle with replicas it runs on the fit GPU,
// which makes it bitwise the single-GPU result.
int nngp_predict_cov(nngp_handle* h, const double* x_test, int64_t T, double* mean_out, double* cov_out) {
  if (!h) return NNGP_EINVAL;
  if (!h->fitted) return fail(h, NNGP_ESTATE, "nngp_predict_cov: no fitted model (call nngp_fit or nngp_set_state)");
  if (!x_test || !mean_out || !cov_out || T <= 0)
    return fail(h, NNGP_EINVAL, "nngp_predict_cov: bad argument (T=%lld)", (long long)T);
  if (h->cfg.kernel_type == 1 && !h->have_M)
    return fail(h, NNGP_ESTATE, "nngp_predict_cov: this imported 'ntk' state has no M yet (nngp_set_state_ntk_m) -- the covariance needs it");
  const int64_t cap = cov_max_rows(h, h->N);
  if (T > cap)
    return fail(h, NNGP_EINVAL, "nngp_predict_cov: T=%lld rows do not fit one prediction block: %s of the batch must fit "
                "max_block_bytes=%lld at N=%lld, which allows T <= %lld", (long long)T,
                h->cfg.kernel_type == 1 ? "V, U and V M" : "V", (long long)h->cfg.max_block_bytes, (long long)h->N,
                (long long)cap);
  return predict_impl(h, x_test, T, mean_out, nullptr, cov_out);
}

// -------------------------------------------------------------------------------------------------
int nngp_get_dims(nngp_handle* h, int64_t* N, int64_t* D, double* lambda_out) {
  if (!h) return NNGP_EINVAL;
  if (!h->fitted) return fail(h, NNGP_ESTATE, "nngp_get_dims: no fitted model");
  if (N) *N = h->N;
  if (D) *D = h->D;
  if (lambda_out) *lambda_out = h->lambda;
  return NNGP_OK;
}

int nngp_log_marginal_likelihood(nngp_handle* h, double* lml_out) {
  if (!h || !lml_out) return NNGP_EINVAL;
  if (!h->fitted || !h->have_labels)
    return fail(h, NNGP_ESTATE, "nngp_log_marginal_likelihood: needs a model fitted by nngp_fit on this handle");
  const double two_pi = 6.283185307179586476925;
  *lml_out = -0.5 * h->lml_terms[1] - h->lml_terms[0] - 0.5 * (double)h->N * log(two_pi);
  return NNGP_OK;
}

int nngp_get_state(nngp_handle* h, double* x_out, double* l_out, double* alpha_out) {
  if (!h) return NNGP_EINVAL;
  if (!h->fitted) return fail(h, NNGP_ESTATE, "nngp_get_state: no fitted model");
  CKR(bind_device(h));
  if (x_out) CKR(download(h, h->X.as<double>(), h->N, h->D, h->ldx, x_out));
  if (l_out) {
    dim3 grid((unsigned)((h->N + 255) / 256), (unsigned)std::min<int64_t>(h->N, 4096));
    zero_upper_kernel<<<grid, 256, 0, h->stream>>>(h->L.as<double>(), h->ldl, (int)h->N);
    h->st.kernel_launches++;
    CKR(download(h, h->L.as<double>(), h->N, h->N, h->ldl, l_out));
  }
  if (alpha_out) CKR(download(h, h->alpha.as<double>(), h->N, 1, 1, alpha_out));
  CK(cudaStreamSynchronize(h->stream));
  return NNGP_OK;
}

// The tail of nngp_set_state / nngp_state_import_end: X, L and alpha are on the device.  X gets the checks of a fit
// (the handle stays unfitted if it fails them); q and inv(L_JJ) are derived, then the state is published.
static int finish_import(nngp_handle* h, double lambda, bool have_M, const char* who) {
  CKR(begin_call(h));
  CKR(derive_q(h, h->N, 0));
  CKR(run_trtri_diag(h));
  CKR(end_call(h, who, "x"));
  h->lambda = lambda;
  return publish_state(h, false, have_M);
}

int nngp_set_state(nngp_handle* h, const double* x, const double* l, const double* alpha, int64_t N, int64_t D,
                   double lambda) {
  if (!h) return NNGP_EINVAL;
  if (!x || !l || !alpha || N <= 0 || D <= 0) return fail(h, NNGP_EINVAL, "nngp_set_state: bad argument");
  CKR(begin_state(h, N, D));
  CKR(upload_matrix(h, x, N, D, h->X.as<double>(), h->ldx));
  CKR(upload_matrix(h, l, N, N, h->L.as<double>(), h->ldl));
  CKR(upload_matrix(h, alpha, N, 1, h->alpha.as<double>(), 1));
  return finish_import(h, lambda, false, "nngp_set_state");
}

// NTK mode: the fitted state also holds M = L^-1 K_dd L^-T (N x N, symmetric, dense), needed by the posterior variance.
int nngp_get_state_ntk_m(nngp_handle* h, double* m_out) {
  if (!h || !m_out) return NNGP_EINVAL;
  if (!h->fitted || h->cfg.kernel_type != 1 || !h->have_M)
    return fail(h, NNGP_ESTATE, "nngp_get_state_ntk_m: needs a fitted 'ntk' model that holds M");
  CKR(bind_device(h));
  CKR(download(h, h->Mmat.as<double>(), h->N, h->N, h->ldl, m_out));
  CK(cudaStreamSynchronize(h->stream));
  return NNGP_OK;
}

int nngp_set_state_ntk_m(nngp_handle* h, const double* m) {
  if (!h || !m) return NNGP_EINVAL;
  if (!h->fitted || h->cfg.kernel_type != 1)
    return fail(h, NNGP_ESTATE, "nngp_set_state_ntk_m: call nngp_set_state on an 'ntk' handle first");
  CKR(bind_device(h));
  CKR(upload_matrix(h, m, h->N, h->N, h->Mmat.as<double>(), h->ldl));   // (Mmat: sized by ensure_model)
  CK(cudaStreamSynchronize(h->stream));
  return publish_state(h, h->have_labels, true);
}

// -------------------------------------------------------------------------------------------------
// Packed state (see the header): [ X (N*D) | alpha (N) | tril(L) by rows (N(N+1)/2) | ntk: M (N*N) ]
static int64_t packed_size(const nngp_handle* h) {
  const int64_t N = h->N, D = h->D;
  return N * D + N + N * (N + 1) / 2 + ((h->cfg.kernel_type == 1) ? N * N : 0);
}
static StatePackView pack_view(nngp_handle* h) {
  StatePackView v;
  v.X = h->X.as<double>(); v.alpha = h->alpha.as<double>(); v.L = h->L.as<double>(); v.M = h->Mmat.as<double>();
  v.N = h->N; v.D = h->D; v.ldx = h->ldx; v.ldl = h->ldl;
  return v;
}
static int pack_range(nngp_handle* h, int64_t offset, int64_t count, double* ext, bool unpack, const char* who) {
  if (!ext || offset < 0 || count <= 0 || offset + count > packed_size(h))
    return fail(h, NNGP_EINVAL, "%s: range [%lld, +%lld) outside the packed state (%lld doubles)", who,
                (long long)offset, (long long)count, (long long)packed_size(h));
  CKR(bind_device(h));
  double* dptr = ext;
  const bool dev = is_device_ptr(ext);
  if (!dev) {   // host memory on the other side: stage the range through a device buffer
    CKR(ensure(h, h->stage, (size_t)count * 8));
    dptr = h->stage.as<double>();
    if (unpack) { CK(cudaMemcpyAsync(dptr, ext, (size_t)count * 8, cudaMemcpyHostToDevice, h->stream)); h->st.h2d_bytes += count * 8; }
  }
  const int grid = (int)std::min<int64_t>((count + 255) / 256, 16LL * h->sm_count);
  if (unpack) state_pack_kernel<true><<<grid, 256, 0, h->stream>>>(pack_view(h), offset, count, dptr);
  else state_pack_kernel<false><<<grid, 256, 0, h->stream>>>(pack_view(h), offset, count, dptr);
  h->st.kernel_launches++;
  if (!dev && !unpack) { CK(cudaMemcpyAsync(ext, dptr, (size_t)count * 8, cudaMemcpyDeviceToHost, h->stream)); h->st.d2h_bytes += count * 8; }
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaGetLastError());
  return NNGP_OK;
}

int nngp_state_packed_size(nngp_handle* h, int64_t* n_doubles) {
  if (!h || !n_doubles) return NNGP_EINVAL;
  if (!h->fitted && !h->importing) return fail(h, NNGP_ESTATE, "nngp_state_packed_size: no fitted model and no import in progress");
  *n_doubles = packed_size(h);
  return NNGP_OK;
}

int nngp_state_pack(nngp_handle* h, int64_t offset, int64_t count, double* dst) {
  if (!h) return NNGP_EINVAL;
  if (!h->fitted) return fail(h, NNGP_ESTATE, "nngp_state_pack: no fitted model");
  if (h->cfg.kernel_type == 1 && !h->have_M) return fail(h, NNGP_ESTATE, "nngp_state_pack: this 'ntk' state holds no M");
  return pack_range(h, offset, count, dst, false, "nngp_state_pack");
}

int nngp_state_import_begin(nngp_handle* h, int64_t N, int64_t D) {
  if (!h) return NNGP_EINVAL;
  if (N <= 0 || D <= 0 || N > 65535LL * GEMM_BM) return fail(h, NNGP_EINVAL, "nngp_state_import_begin: bad shape (N=%lld D=%lld)", (long long)N, (long long)D);
  CKR(begin_state(h, N, D));
  if (h->ldx != D) CK(cudaMemsetAsync(h->X.p, 0, (size_t)N * h->ldx * 8, h->stream));   // the pad column stays zero
  CK(cudaStreamSynchronize(h->stream));
  h->importing = true;
  return NNGP_OK;
}

int nngp_state_unpack(nngp_handle* h, int64_t offset, int64_t count, const double* src) {
  if (!h) return NNGP_EINVAL;
  if (!h->importing) return fail(h, NNGP_ESTATE, "nngp_state_unpack: call nngp_state_import_begin first");
  return pack_range(h, offset, count, const_cast<double*>(src), true, "nngp_state_unpack");
}

int nngp_state_import_end(nngp_handle* h, double lambda) {
  if (!h) return NNGP_EINVAL;
  if (!h->importing) return fail(h, NNGP_ESTATE, "nngp_state_import_end: no import in progress");
  CKR(bind_device(h));
  h->importing = false;
  return finish_import(h, lambda, h->cfg.kernel_type == 1, "nngp_state_import_end");
}

// -------------------------------------------------------------------------------------------------
int nngp_diag_dmma_peak(nngp_handle* h, double* tflops_out) {
  if (!h || !tflops_out) return NNGP_EINVAL;
  CKR(bind_device(h));
  const int iters = 4096;
  // exactly one full wave: every SM holds its maximum number of CTAs.  (With fewer CTAs than slots the block
  // scheduler may load some SMs with 5 and others with 3 -- the probe then reads 4/5 of the peak.)
  int per_sm = 4;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, dmma_peak_kernel, 256, 0));
  if (per_sm < 1) per_sm = 1;
  const int ctas = h->sm_count * per_sm;
  cudaEvent_t a = get_event(h), b = get_event(h);
  for (int w = 0; w < 8; ++w)  // ~35 ms of warm-up so the SM clock is at its loaded value
    dmma_peak_kernel<<<ctas, 256, 0, h->stream>>>(iters, h->lam_d.as<double>());
  double best = 0.0;
  for (int rep = 0; rep < 8; ++rep) {
    cudaEventRecord(a, h->stream);
    dmma_peak_kernel<<<ctas, 256, 0, h->stream>>>(iters, h->lam_d.as<double>());
    cudaEventRecord(b, h->stream);
    CK(cudaStreamSynchronize(h->stream));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, a, b));
    const double flops = (double)ctas * 8 /*warps*/ * (double)iters * 16 * 512.0;
    best = std::max(best, flops / (ms * 1e-3) / 1e12);
  }
  h->st.kernel_launches += 16;
  h->ev_pool.push_back(a); h->ev_pool.push_back(b);
  *tflops_out = best;
  return NNGP_OK;
}

int nngp_diag_gemm_probe(nngp_handle* h, int64_t M, int64_t N, int64_t K, int32_t iters, double* ms_out) {
  if (!h || !ms_out || M <= 0 || N <= 0 || K <= 0 || K % GEMM_BK || iters <= 0)
    return fail(h, NNGP_EINVAL, "nngp_diag_gemm_probe: bad argument");
  CKR(bind_device(h));
  DevBuf A, B, C;
  const int64_t ld = round_up(K, 16), ldc = round_up(N, 16);
  int rc = ensure(h, A, (size_t)M * ld * 8);
  if (rc == NNGP_OK) rc = ensure(h, B, (size_t)N * ld * 8);
  if (rc == NNGP_OK) rc = ensure(h, C, (size_t)M * ldc * 8);
  if (rc != NNGP_OK) { release(A); release(B); release(C); return rc; }
  cudaMemsetAsync(A.p, 0, (size_t)M * ld * 8, h->stream);
  cudaMemsetAsync(B.p, 0, (size_t)N * ld * 8, h->stream);
  cudaMemsetAsync(C.p, 0, (size_t)M * ldc * 8, h->stream);
  MatView Av{A.as<double>(), M, K, ld}, Bv{B.as<double>(), N, K, ld};
  discard_spans(h);   // (spans of a failed earlier call)
  rc = run_gemm_sub(h, Av, 0, 0, Bv, 0, 0, M, N, K, C.as<double>(), ldc, 0);  // warm-up
  cudaEvent_t a = get_event(h), b = get_event(h);
  cudaEventRecord(a, h->stream);
  for (int i = 0; i < iters && rc == NNGP_OK; ++i) rc = run_gemm_sub(h, Av, 0, 0, Bv, 0, 0, M, N, K, C.as<double>(), ldc, 0);
  cudaEventRecord(b, h->stream);
  cudaError_t e = cudaStreamSynchronize(h->stream);
  float ms = 0.f;
  cudaEventElapsedTime(&ms, a, b);
  h->ev_pool.push_back(a); h->ev_pool.push_back(b);
  settle_spans(h);
  h->tmaps.clear();  // the scratch operands are about to be freed
  release(A); release(B); release(C);
  if (rc != NNGP_OK) return rc;
  if (e != cudaSuccess) return fail(h, NNGP_ECUDA, "gemm probe failed: %s", cudaGetErrorString(e));
  *ms_out = ms / iters;
  return NNGP_OK;
}

int nngp_diag_potrf(nngp_handle* h, double* a, int64_t N) {
  if (!h || !a || N <= 0) return NNGP_EINVAL;
  CKR(bind_device(h));
  const int64_t ld = round_up(N, 16);
  DevBuf A, W;   // the matrix and the inverses of its diagonal blocks
  CKR(ensure(h, A, (size_t)N * ld * 8));
  int rc = begin_call(h);
  if (rc == NNGP_OK) rc = upload_matrix(h, a, N, N, A.as<double>(), ld);
  if (rc == NNGP_OK) rc = ensure(h, W, (size_t)round_up(N, NB) * NB * sizeof(double));
  if (rc == NNGP_OK) rc = run_potrf(h, A.as<double>(), ld, N, 0, W.as<double>());
  if (rc == NNGP_OK) rc = download(h, A.as<double>(), N, N, ld, a);
  int pivot = 0;
  if (rc == NNGP_OK) rc = end_call(h, "nngp_diag_potrf", "a", &pivot);
  cudaStreamSynchronize(h->stream);   // (also after a failure: A and W are freed next)
  h->tmaps.clear();
  release(A); release(W);
  if (rc != NNGP_OK) return rc;
  if (pivot) return fail(h, NNGP_ENOTPD, "nngp_diag_potrf: not positive definite (pivot %d)", pivot - 1);
  return NNGP_OK;
}

}  // extern "C"
