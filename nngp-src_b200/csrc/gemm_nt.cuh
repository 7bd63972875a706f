// gemm_nt.cuh -- the FP64 "NT" tensor-core GEMM core every dense stage of the hot path uses:
//
//     acc(128 x 64) = A[m0:m0+128, k0:k0+K] * B[n0:n0+64, k0:k0+K]^T      (both row-major,
//                                                                         K contiguous)
//
//   * operands: TMA (cp.async.bulk.tensor.2d, SWIZZLE_128B, box 16 doubles x {128|64} rows)
//     into a 4-stage shared-memory ring with full/empty mbarriers; thread 0 is the producer: it
//     refills a stage right after all 8 warps have released it (prefetch distance 3 k-tiles);
//   * math: 8 warps (4 along M x 2 along N), each a 32 x 32 warp tile = 4 x 4
//     mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4) accumulators, 64 FP64 registers per thread;
//   * 256 threads x <= 128 registers, ~97 KB smem -> 2 CTAs per SM, so one CTA's epilogue hides
//     under the other's main loop, and no local memory (a 9-warp variant with a dedicated producer
//     warp was capped at 96 registers and spilled its output pointers to the stack);
//   * epilogues: (GRAM) the NNGP arc-cosine recursion of SURVEY Appendix A.1 applied in
//     registers -- intermediate layer kernels never touch HBM -- or (SUB) C -= acc, the
//     trailing/left-looking update of the blocked Cholesky and triangular solves.
//
// Shared-memory layout of one operand stage (what SWIZZLE_128B produces): row r occupies
// bytes [128 r, 128 r + 128); the 16-byte chunk c of that row lands at chunk c ^ (r & 7).
// A DMMA A/B fragment load (lane 4g+t reads row g, k = 8*(t>>1) + 2*s + (t&1) in step s -- a
// permutation of the k index shared by A and B, see mma_mainloop) touches, per half-warp, every
// bank exactly once => 2 wavefronts for 256 B: conflict-free.
#pragma once
#include "dense_kernels.cuh"
#include "ptx.cuh"

namespace nngp {

constexpr int GEMM_BM = 128;
constexpr int GEMM_BN = 64;
constexpr int GEMM_BK = 16;
constexpr int GEMM_MAX_LAYERS = 16;   // == NNGP_MAX_LAYERS (include/nngp_b200.h)
constexpr int GEMM_STAGES = 4;
constexpr int GEMM_CONSUMER_WARPS = 8;
constexpr int GEMM_THREADS = GEMM_CONSUMER_WARPS * 32;  // no dedicated producer warp: thread 0 issues the TMA loads
constexpr int GEMM_A_STAGE_BYTES = GEMM_BM * GEMM_BK * 8;  // 16 KiB
constexpr int GEMM_B_STAGE_BYTES = GEMM_BN * GEMM_BK * 8;  //  8 KiB
constexpr int GEMM_STAGE_TX_BYTES = GEMM_A_STAGE_BYTES + GEMM_B_STAGE_BYTES;
// ring + barriers + 1 KiB slack so the ring can be aligned to the 1024 B swizzle atom
constexpr int GEMM_SMEM_BYTES =
    GEMM_STAGES * (GEMM_A_STAGE_BYTES + GEMM_B_STAGE_BYTES) + 2 * GEMM_STAGES * 8 + 1024;

enum GemmEpilogue : int { EPI_GRAM = 0, EPI_SUB = 1, EPI_ROWDOT = 2, EPI_DIAG = 3 };

// Activation of every hidden step (== NNGP_ACT_*, include/nngp_b200.h), and the coefficients its steps use, derived
// once from (a, b, c) on the host (make_act_coef in capi.cu).
enum GramAct : int { ACT_RELU = 0, ACT_ABRELU = 1, ACT_ERF = 2 };
struct ActCoef {
  int kind;
  double c0, c1;   // ReLU / ABRelu: (a^2 + b^2) / 2 and (a - b)^2 / (2 pi)   (ReLU: 1/2 and 1/(2 pi))
  double b2x2;     // Erf: 2 b^2
  double e, c2;    // Erf: a^2 (2/pi) and c^2
  double kd;       // Erf: a^2 b^2 (4/pi)
};

struct GemmParams {
  int M, N;            // valid output extent (rows of the A range, rows of the B range)
  int ktiles;          // number of 16-wide K tiles
  int a_row0, a_col0;  // origin of the A range inside tensor map A (elements)
  int b_row0, b_col0;  // origin of the B range inside tensor map B
  double* C;           // output, already offset to the (0,0) element of the range
  long long ldc;
  int lower;           // 1: tiles strictly above the diagonal of the range are skipped
  // EPI_GRAM only
  const double* q1;    // per-row layer-0 diagonal of the A rows  (sigma_w^2 |x|^2/D + sigma_b^2)
  const double* q2;    // same for the B rows
  double scale;        // sigma_w^2 / D of the first Dense layer
  double sb2;          // sigma_b^2 of the first Dense layer
  double lsw2[GEMM_MAX_LAYERS];   // sigma_w^2 / sigma_b^2 of the Dense layer that FOLLOWS arc-cosine step s
  double lsb2[GEMM_MAX_LAYERS];   // (entry min(s, 15): a uniform network of any depth fills all entries alike)
  int steps;           // depth-1 arc-cosine steps
  int ntk;             // 1: C receives the NTK Theta, C2 (if not null) the NNGP kernel K
  double* C2;
  const double* alpha; // EPI_GRAM, optional: fused posterior-mean GEMV,
                       //   mean_partial[(2 * tile_n + wn) * M + r] = sum over that warp's 32 columns of K[r][c] alpha[c]
  double* mean_partial;
  // EPI_ROWDOT only: partial[tile_n * M + r] = sum_{c in tile} acc[r][c] * W[r][c]
  const double* W;     // M x N, leading dimension ldc (reuses ldc); nullptr: W = acc (row sums of squares)
  double* partial;
  int kchunk;          // > 0: split-K over blockIdx.z in chunks of kchunk k-tiles; the epilogue then stores the partial
  double* vpart;       //      products to vpart[(z * M + r) * N + c] instead of reducing them (few-row batches: the
                       //      column tiles near the end of a triangular product would otherwise be one long serial loop)
  int tri_k;           // 1: B is lower triangular (row j is zero beyond column j): column tile n only needs the k-tiles
                       //    up to its own last column -- the latency-mode product V = K_* L^-T against the explicit inverse
  uint32_t zero;       // always 0 (value-initialised): opaque run-time zero for mma_mainloop's release dependence
  // EPI_DIAG only (diagonal step of the row-wise triangular solve, see diag_epilogue): C <- A * Winv^T, K = 64
  double* ssq;         // [M] running sum of squares of the solved row (cross-launch carry)
  const double* kss;   // [M] K(x,x)
  double* var;         // [M] or nullptr (plain solve)
  int J, col_blocks;   // which 64-column block this launch solves, of how many
  // EPI_GRAM: the activation's coefficients (gemm_nt_kernel<EPI_GRAM, ACT>).  Erf reads the diagonals entering steps
  // 1..steps-1 from per-row tables (q_final_kernel): tab1[(s - 1) * tld1 + r] for the A rows, tab2 alike for B.
  ActCoef act;
  const double* tab1;
  const double* tab2;
  long long tld1, tld2;
};

// Epilogue of the diagonal step of  V = K_* L^-T  (shared by trsm_fused_kernel and gemm_nt_kernel<EPI_DIAG>, which
// is what makes a row's result bitwise independent of the path / blocking / GPU count): the accumulators hold the
// solved 128 x 64 block X = R * inv(L_JJ)^T; store it, add sum_c X[r][c]^2 to the row's running sum of squares and,
// with the last column block, write var = K(x,x) - sum.  Columns >= nb of X are exact zeros (zero residual,
// identity-padded inverse).  `s_part` is 256 doubles of shared memory nobody else uses until the next barrier.
struct DiagOut {
  double* B;            // block origin: element (row 0 of the buffer, column col0 of the block)
  long long ldb;
  int rows;
  double* ssq;
  const double* kss;
  double* var;
  int J, col_blocks;
};
__device__ __forceinline__ void diag_epilogue(const double (&acc)[4][4][2], const DiagOut& o, int row0, int nb, int wm,
                                              int wn, int g, int t, double* s_part) {
#pragma unroll
  for (int mi = 0; mi < 4; ++mi) {
    const int lr = wm * 32 + mi * 8 + g;
    const int row = row0 + lr;
    double part = 0.0;
#pragma unroll
    for (int ni = 0; ni < 4; ++ni) {
      const int lc = wn * 32 + ni * 8 + 2 * t;
      const double x0 = acc[mi][ni][0], x1 = acc[mi][ni][1];
      if (row < o.rows) {
        double* dst = o.B + (long long)row * o.ldb + lc;
        if (lc + 1 < nb) *reinterpret_cast<double2*>(dst) = make_double2(x0, x1);
        else if (lc < nb) dst[0] = x0;
      }
      part = fma(x0, x0, part);
      part = fma(x1, x1, part);
    }
    part += __shfl_xor_sync(0xffffffffu, part, 1);
    part += __shfl_xor_sync(0xffffffffu, part, 2);
    if (t == 0) s_part[lr * 2 + wn] = part;
  }
  __syncthreads();
  if (threadIdx.x < 128) {
    const int grow = row0 + (int)threadIdx.x;
    if (o.var != nullptr && grow < o.rows) {
      const double ss = s_part[threadIdx.x * 2] + s_part[threadIdx.x * 2 + 1];
      const double tot = ((o.J > 0) ? __ldcg(o.ssq + grow) : 0.0) + ss;
      if (o.J + 1 == o.col_blocks) o.var[grow] = o.kss[grow] - tot;
      else __stcg(o.ssq + grow, tot);
    }
  }
}

// theta = atan2(s, k) for s = sqrt(s2) >= 0 (theta in [0, pi]), pi/2 at s == k == 0 [nt: _arctan2(fill_zero = pi/2)].
// atan(t) = t P(t^2) on t = min(s,|k|)/max(s,|k|) in [0,1], P of degree 20 (interpolant of atan(sqrt u)/sqrt u at the
// Chebyshev nodes, fitted in 40-digit mpmath; FP64 evaluation error <= 2.3e-16 relative).  Two things keep the FP64
// pipe -- which this epilogue shares with the co-resident CTA's DMMAs -- and the dependency chain short:
//   * no division:  min/max = s |k| / max(s^2, k^2);  the reciprocal of max(s^2, k^2) (MUFU.RCP64H seed + two Newton
//     steps, 1 ulp) does not depend on the square root, so the two run side by side instead of back to back;
//   * P is evaluated as  Pe(w) + u Po(w),  w = u^2: two independent Horner chains of 10 instead of one of 20.
// Total error of theta <= 2 ulp (tests/test_oracle.py restates the identical algorithm in numpy against mpmath).
__device__ __forceinline__ double rcp_newton(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));   // ~20 good bits
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  return fma(r, e, r);
}

// max(x, 0) for finite x through the sign bit (integer pipe); -0 and negative rounding residue become +0
__device__ __forceinline__ double clamp_nonneg(double x) { return (__double2hiint(x) < 0) ? 0.0 : x; }

// GUARD = false: only for max(s^2, k^2) in [2^-1022, 2^1022) (see gram_epilogue), where both versions agree bitwise.
template <bool GUARD>
__device__ __forceinline__ double atan2_pos(double s, double s2, double k) {
  constexpr double C[21] = {
    1.0,
    -0.3333333333333286,
    0.19999999999929946,
    -0.14285714281592693,
    0.11111110982087126,
    -0.09090906605656898,
    0.0769227555520563,
    -0.06666371187721098,
    0.05880342002401543,
    -0.052527255573225747,
    0.04719723992321112,
    -0.042125723963855326,
    0.03651081352721035,
    -0.02970071773623423,
    0.021740213830758134,
    -0.013674139288399478,
    0.007038646202989813,
    -0.0028047655531701315,
    0.0008033604181626027,
    -0.00014617088163625013,
    1.2631178430477426e-05};
  const double half_pi = 1.57079632679489661923;
  const double pi = 3.14159265358979323846;
  // The comparisons run on the integer pipe (bit patterns of non-negative doubles order like the values; the sign of
  // k is its top bit): a DSETP would queue on the FP64 pipe this epilogue shares with the co-resident CTA's DMMAs.
  const double a = fabs(k);
  const double a2 = k * k;
  bool s_bigger = __double_as_longlong(s2) > __double_as_longlong(a2);
  double mx2 = s_bigger ? s2 : a2;
  double sa = s * a;
  // rcp.approx.ftz flushes a subnormal input (seed +inf -> NaN after Newton) and a subnormal result (t -> 0): outside
  // mx2 in [2^-1022, 2^1022) -- biased exponent field 1..2044, tested on the integer pipe -- s and |k| are first scaled
  // by 2^+-600 (t = min/max does not change), which brings max(s, |k|) from anywhere in [2^-1074, 2^1024) into
  // [2^-474, 2^424].  s2 / a2 are then also unreliable (underflow), so the larger side is decided on s, |k| themselves.
  if (GUARD && (unsigned)(__double2hiint(mx2) >> 20) - 1u >= 2044u) {
    const double f = (__double2hiint(mx2) < 0x00100000) ? 0x1p+600 : 0x1p-600;
    const double sf = s * f, af = a * f;
    s_bigger = __double_as_longlong(sf) > __double_as_longlong(af);
    mx2 = s_bigger ? sf * sf : af * af;
    sa = sf * af;
  }
  const double t = sa * rcp_newton(mx2);
  const double u = t * t;
  const double w = u * u;
  double pe = C[20], po = C[19];
#pragma unroll
  for (int i = 18; i >= 0; i -= 2) pe = fma(pe, w, C[i]);
#pragma unroll
  for (int i = 17; i >= 1; i -= 2) po = fma(po, w, C[i]);
  const double at = t * fma(u, po, pe);
  const double th0 = s_bigger ? (half_pi - at) : at;
  const double th = (__double2hiint(k) < 0) ? (pi - th0) : th0;
  // s == k == 0 on the bit patterns (s >= +0; the shift drops the sign of k): k^2 can underflow while k != 0
  return ((__double_as_longlong(s) | (__double_as_longlong(k) << 1)) == 0LL) ? half_pi : th;
}

// One ReLU arc-cosine step followed by the next Dense layer's affine map
// (SURVEY Appendix A.1; [nt 0.6.1 stax.ABRelu(a=0,b=1) nngp_ntk_fn + stax.Dense _affine]):
//   s = sqrt(max(q1 q2 - k^2, 0)); theta = atan2(s, k) (pi/2 when s == k == 0)
//   k' = sw2 * ( s/(2 pi) + (1/2 - theta/(2 pi)) k ) + sb2
template <bool GUARD>
__device__ __forceinline__ double arccos_step(double k, double q1, double q2, double sw2, double sb2) {
  const double inv_2pi = 0.15915494309189533577;
  double s2 = clamp_nonneg(q1 * q2 - k * k);
  double s = sqrt(s2);
  double theta = atan2_pos<GUARD>(s, s2, k);
  double dot_sigma = 0.5 - inv_2pi * theta;
  double r = inv_2pi * s + dot_sigma * k;
  return sw2 * r + sb2;
}


// Same step, also advancing the NTK:  ntk' = k' + sw2 * (ntk * kdot),  kdot = 1/2 - theta/(2 pi)
// (SURVEY Appendix A.5; [nt: Relu `ntk *= dot_sigma`, Dense `ntk = nngp + W_std^2 * ntk`]).
template <bool GUARD>
__device__ __forceinline__ void arccos_step_ntk(double& k, double& ntk, double q1, double q2, double sw2, double sb2) {
  const double inv_2pi = 0.15915494309189533577;
  double s2 = clamp_nonneg(q1 * q2 - k * k);
  double s = sqrt(s2);
  double theta = atan2_pos<GUARD>(s, s2, k);
  double dot_sigma = 0.5 - inv_2pi * theta;
  double r = inv_2pi * s + dot_sigma * k;
  k = sw2 * r + sb2;
  ntk = k + sw2 * (ntk * dot_sigma);
}

// ABRelu(a, b), phi(x) = a min(x, 0) + b max(x, 0) [nt 0.6.1 stax.ABRelu]: the arc-cosine step with two coefficients,
//   kdot = c0 - c1 theta,  E[phi(u) phi(v)] = c1 s + kdot k,  E[phi(u)^2] = c0 q;  c0 = (a^2+b^2)/2, c1 = (a-b)^2/(2 pi)
// (ReLU is c0 = 1/2, c1 = 1/(2 pi): arccos_step).  Same theta, same range argument as ReLU.  Returns kdot.
template <bool GUARD>
__device__ __forceinline__ double abrelu_step(double& k, double q1, double q2, double sw2, double sb2, double c0, double c1) {
  const double s2 = clamp_nonneg(q1 * q2 - k * k);
  const double s = sqrt(s2);
  const double theta = atan2_pos<GUARD>(s, s2, k);
  const double kdot = c0 - c1 * theta;
  const double r = c1 * s + kdot * k;
  k = sw2 * r + sb2;
  return kdot;
}

// Erf(a, b, c), phi(x) = a erf(b x) + c [nt 0.6.1 stax.Erf].  With Q = b^2 q, K = b^2 k and
//   P = (1 + 2 Q1)(1 + 2 Q2) - 4 K^2 = 1 + 2 (Q1 + Q2) + 4 b^4 s^2        (the second form cancels nothing)
//   E[phi(u) phi(v)] = a^2 (2/pi) arcsin(2K / sqrt((1 + 2 Q1)(1 + 2 Q2))) + c^2 = a^2 (2/pi) atan2(2K, sqrt P) + c^2
//   kdot = E[phi'(u) phi'(v)] = a^2 b^2 (4/pi) / sqrt P
// sqrt P >= 1, so nothing divides by a small number, and atan2_pos takes atan(|2K| / sqrt P) itself wherever
// |2K| < sqrt P (its t = min / max): a small kernel value keeps its relative accuracy against a small diagonal.  The
// accepted input range, b^2 q < 2^508 on every layer (row_sqnorm_kernel's limit and make_act_coef), keeps P below
// 2^1019 and 4 K^2 below 2^1018, so atan2_pos needs no range guard: there is no guarded Erf path.
__device__ __forceinline__ double erf_expect(double k2, double sp, const ActCoef& a) {   // k2 = 2K, sp = sqrt P
  const double th = atan2_pos<false>(fabs(k2), k2 * k2, sp);
  return fma(a.e, copysign(th, k2), a.c2);
}

// E[phi(u)^2] of Erf at variance q: the step above at k = q1 = q2 = q (s = 0), P = 1 + 4Q
__device__ __forceinline__ double erf_diag(double q, const ActCoef& a) {
  return erf_expect(a.b2x2 * q, sqrt(fma(a.b2x2, q + q, 1.0)), a);
}

template <bool NTK>
__device__ __forceinline__ void erf_step(double& k, double& ntk, double q1, double q2, double sw2, double sb2,
                                         const ActCoef& a) {
  const double s2 = clamp_nonneg(q1 * q2 - k * k);
  const double bs = a.b2x2 * sqrt(s2);                               // 2 b^2 s
  const double sp = sqrt(fma(bs, bs, fma(a.b2x2, q1 + q2, 1.0)));    // sqrt P
  const double kn = sw2 * erf_expect(a.b2x2 * k, sp, a) + sb2;
  if (NTK) ntk = kn + sw2 * (ntk * (a.kd * rcp_newton(sp)));
  k = kn;
}

// One hidden step of activation ACT on an entry (and its NTK when NTK), followed by the next Dense layer
template <int ACT, bool GUARD, bool NTK>
__device__ __forceinline__ void gram_step(double& k, double& ntk, double q1, double q2, double sw2, double sb2,
                                          const ActCoef& a) {
  if constexpr (ACT == ACT_ERF) {
    erf_step<NTK>(k, ntk, q1, q2, sw2, sb2, a);
  } else if constexpr (ACT == ACT_ABRELU) {
    const double kdot = abrelu_step<GUARD>(k, q1, q2, sw2, sb2, a.c0, a.c1);
    if (NTK) ntk = k + sw2 * (ntk * kdot);
  } else if constexpr (NTK) {
    arccos_step_ntk<GUARD>(k, ntk, q1, q2, sw2, sb2);
  } else {
    k = arccos_step<GUARD>(k, q1, q2, sw2, sb2);
  }
}

// The diagonal of the Dense layer that follows a step: q' = sw2 E[phi(u)^2] + sb2
template <int ACT>
__device__ __forceinline__ double next_diag(double q, const ActCoef& a, double sw2, double sb2) {
  if constexpr (ACT == ACT_ERF) return sw2 * erf_diag(q, a) + sb2;
  else if constexpr (ACT == ACT_ABRELU) return sw2 * (a.c0 * q) + sb2;
  else return sw2 * (0.5 * q) + sb2;
}

// Per row: the diagonals of the Dense layers after each of the `steps` activation steps.  tab (optional) receives those
// entering steps 1..steps-1, tab[(s - 1) * rows + r] (what the Erf Gram epilogue reads instead of evaluating E[phi^2]
// per entry), kss (optional) the one after the last step, K(x,x).
__global__ void q_final_kernel(const double* __restrict__ q, int rows, int steps, LayerSig sig, ActCoef act,
                               double* __restrict__ tab, double* __restrict__ kss) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows) return;
  double v = q[i];
  for (int s = 0; s < steps; ++s) {
    const int li = s < 16 ? s : 15;
    if (tab != nullptr && s > 0) tab[(long long)(s - 1) * rows + i] = v;
    // (ReLU: c0 = 1/2 exactly -- the same bits as next_diag<ACT_RELU>)
    v = act.kind == ACT_ERF ? next_diag<ACT_ERF>(v, act, sig.sw2[li], sig.sb2[li])
                            : next_diag<ACT_ABRELU>(v, act, sig.sw2[li], sig.sb2[li]);
  }
  if (kss != nullptr) kss[i] = v;
}

// Operand ring, producer and consumer in one loop.  Every warp: wait for a stage, run its 4 x (4 x 4) DMMAs on
// the warp's 32 x 32 tile, release the stage.  Thread 0 additionally re-arms the stage it has just finished with
// k-tile kt + STAGES once all 8 warps have released it.  `stage` / `phase` persist across calls (persistent kernels).
//
// Releasing a stage (WAR across proxies): the refill is a TMA write (async proxy); nothing orders it after a
// fragment LDS that has been *issued* but has not yet read shared memory, and ptxas does hoist the SYNCS.ARRIVE to
// right behind the last LDS of the k-tile.  With a second, shared-memory-heavy CTA on the SM that LDS can be late
// enough to read the next k-tile (observed: the mi = 3, k4 = 3 fragment of one warp, DESIGN.md 5.3).  The arrive
// therefore carries a data dependence on every fragment register of the k-tile (`seen & zero`, zero == 0 at run
// time but opaque to the compiler), so the scoreboard holds it back until all of them have landed.
struct TileSrc {  // where the A / B operand tiles of this output tile come from
  const CUtensorMap* tmA;
  const CUtensorMap* tmB;
  int a_col0, a_row, b_col0, b_row;
};

template <int STAGES>
__device__ __forceinline__ void ring_issue(const TileSrc& src, uint8_t* ringA, uint8_t* ringB, uint64_t* full_bar,
                                           int stage, int kt) {
  mbar_arrive_expect_tx(&full_bar[stage], GEMM_STAGE_TX_BYTES);
  tma_load_2d(ringA + stage * GEMM_A_STAGE_BYTES, src.tmA, src.a_col0 + kt * GEMM_BK, src.a_row, &full_bar[stage]);
  tma_load_2d(ringB + stage * GEMM_B_STAGE_BYTES, src.tmB, src.b_col0 + kt * GEMM_BK, src.b_row, &full_bar[stage]);
}

// Thread 0 only: start the first min(STAGES, ktiles) loads of a tile.  The stages are free: the previous tile's
// refills stopped at its last k-tile and every warp has passed the barrier that ends a tile.
template <int STAGES>
__device__ __forceinline__ void ring_prologue(const TileSrc& src, uint8_t* ringA, uint8_t* ringB, uint64_t* full_bar,
                                              int stage, int ktiles) {
  const int n = ktiles < STAGES ? ktiles : STAGES;
  for (int i = 0; i < n; ++i) {
    ring_issue<STAGES>(src, ringA, ringB, full_bar, stage, i);
    if (++stage == STAGES) stage = 0;
  }
}

#ifndef NNGP_RELEASE_AT
#define NNGP_RELEASE_AT 0  // 0..3: release k-tile kt-1 after the k4-th fragment loads of k-tile kt; 4: at the end of kt itself
#endif
struct NoGate {  // default refill gate: operand tiles are always ready to be loaded
  __device__ __forceinline__ void operator()(int) const {}
};
// `gate(kt)` is called by thread 0 right before it issues the TMA loads of k-tile kt (refills only; the caller
// gates its own prologue): the persistent solve uses it to wait until the producer of that k-tile's A operand
// (another CTA) has published it.  `active == false` (warp-uniform): this warp's 32-row slab lies entirely beyond
// the valid rows -- it keeps the barrier protocol going but skips its fragment loads and DMMAs, which leaves the
// FP64 pipe to the warps that have rows (a single query occupies 1 of the 4 slabs of a row tile).
template <int STAGES, class Gate = NoGate>
__device__ __forceinline__ void mma_mainloop(double (&acc)[4][4][2], const TileSrc& src, uint8_t* ringA, uint8_t* ringB,
                                             uint64_t* full_bar, uint64_t* empty_bar, int& stage, uint32_t& phase,
                                             int ktiles, int wm, int wn, int lane, uint32_t zero, Gate gate = Gate(),
                                             bool active = true) {
  const int g = lane >> 2, t = lane & 3;
  // Which k does lane (g, t) feed into DMMA step s?  Any bijection (s, t) -> 0..15 is a valid GEMM as long as the A
  // and the B fragment use the same one.  We use  k = 8*(t>>1) + 2*s + (t&1):  logical 16-byte chunk 4*(t>>1) + s,
  // half t&1.  With SWIZZLE_128B (physical chunk = logical ^ (row & 7)) the 16 lanes of a half-warp (4 rows g x 4 t)
  // then touch every (chunk, half) pair exactly once -> an LDS.64 of the warp is 2 wavefronts, conflict-free.
  // (The textbook k = 4*s + t puts rows g and g^1 on the same chunks: 2-way conflicts, 4 wavefronts -- measured
  // with ncu as 45 % of all shared-load wavefronts.)  Byte offset inside the row:
  //   (((4*(t>>1) + s) ^ g) << 4) | ((t&1) << 3)  ==  koff0 ^ (s << 4),   koff0 = (((4*(t>>1)) ^ g) << 4) | ((t&1) << 3)
  // Rows are 128 B apart and stages 1 KiB-aligned, so the XOR can be applied to the full address: two base
  // registers instead of four offsets.
  const uint32_t koff0 = ((uint32_t)((4 * (t >> 1)) ^ g) << 4) | ((uint32_t)(t & 1) << 3);
  const uint32_t a_warp = smem_u32(ringA) + (uint32_t)(wm * 32 + g) * 128u + koff0;
  const uint32_t b_warp = smem_u32(ringB) + (uint32_t)(wn * 32 + g) * 128u + koff0;
  // The release of k-tile kt-1 is issued inside k-tile kt (after its k4 == NNGP_RELEASE_AT loads): by then the
  // fragments it depends on have long landed, so the dependence never stalls the warp.
  auto release = [&](int s, uint32_t ph, uint32_t seen, int kdone) {
    __syncwarp();
    if (lane == 0) mbar_arrive_addr(smem_u32(&empty_bar[s]) + (seen & zero));
    if (threadIdx.x == 0 && kdone + STAGES < ktiles) {
      mbar_wait(&empty_bar[s], ph);  // all 8 warps are done with this stage in this round
      gate(kdone + STAGES);
      ring_issue<STAGES>(src, ringA, ringB, full_bar, s, kdone + STAGES);
    }
    __syncwarp();
  };
  uint32_t seen_prev = 0;
  for (int kt = 0; kt < ktiles; ++kt) {
    mbar_wait(&full_bar[stage], phase);
    uint32_t seen = 0;
    const uint32_t a_st = a_warp + stage * GEMM_A_STAGE_BYTES;
    const uint32_t b_st = b_warp + stage * GEMM_B_STAGE_BYTES;
#pragma unroll
    for (int k4 = 0; k4 < 4; ++k4) {
      double a[4], b[4];
      if (active) {
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) a[mi] = lds_f64((a_st ^ (uint32_t)(k4 << 4)) + mi * 1024);
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) b[ni] = lds_f64((b_st ^ (uint32_t)(k4 << 4)) + ni * 1024);
      }
      if (k4 == NNGP_RELEASE_AT && kt > 0)
        release(stage == 0 ? STAGES - 1 : stage - 1, stage == 0 ? phase ^ 1u : phase, seen_prev, kt - 1);
      if (active) {
#pragma unroll
        for (int mi = 0; mi < 4; ++mi)
#pragma unroll
          for (int ni = 0; ni < 4; ++ni) dmma_884(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
        // folded after the DMMAs that consume the same registers: the values have landed, the XORs never stall
#pragma unroll
        for (int i = 0; i < 4; ++i) seen ^= (uint32_t)__double2hiint(a[i]) ^ (uint32_t)__double2hiint(b[i]);
      }
    }
#if NNGP_RELEASE_AT >= 4
    release(stage, phase, seen, kt);
#endif
    seen_prev = seen;
    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
  }
  if (NNGP_RELEASE_AT < 4 && ktiles > 0) release(stage == 0 ? STAGES - 1 : stage - 1, stage == 0 ? phase ^ 1u : phase, seen_prev, ktiles - 1);
}

// Gram epilogue (K1 + K2 + K3 (+ K8)): k = scale * acc + sb2, depth-1 arc-cosine steps in registers, store, and
// (optionally) the fused posterior-mean GEMV partial of this warp's 32 columns.
// Two other organisations of this kernel were built and measured in round 2, and dropped (0.55 / 0.58 of the DMMA peak
// at D = 128 depth 2 / D = 256 depth 3 for one tile per CTA, 2 CTAs per SM):
//   * persistent: one CTA per SM slot walking the tiles, the next tile's TMA loads in flight during the epilogue --
//     0.41: two co-resident persistent CTAs run in lock-step, both in the main loop or both in the epilogue; with one
//     tile per CTA the hardware scheduler staggers them, and a DMMA phase overlapping an FP64-FMA phase is what fills
//     the shared FP64 pipe;
//   * warp-specialised: one 512-thread CTA per SM, 8 DMMA warps running the main loops back to back and handing the
//     accumulator tiles through shared memory to 8 epilogue warps -- 0.45 / 0.50 (0.47 / 0.52 with 8 entries in flight
//     per thread): the register file caps the CTA at 16 warps, and 8 warps cannot keep enough of the epilogue's
//     dependent FP64 chains in flight; the epilogue becomes the longer side.
// Whether atan2_pos may skip its range guard for all W entries of a group: with q1 in [2^e1, 2^(e1+1)) and q2 in
// [2^e2, 2^(e2+1)), max(s^2, k^2) lies in [q1 q2 / 2, q1 q2] (s^2 + k^2 = q1 q2, up to rounding), so
// e1 + e2 in [-1020, 1019] keeps it inside [2^-1022, 2^1022).  That needs q1 and q2 to be normal doubles: a zero or
// subnormal q (a row whose |x|^2 / D underflowed) no longer bounds k, whose own products did not underflow.
// Exponents only: integer pipe.  The guarded version costs a branch per entry, which splits the W independent chains
// the scheduler interleaves (-3..5 % Gram throughput), so it only runs for groups that need it (zero rows, inputs
// near the ends of the FP64 range).
template <int W>
__device__ __forceinline__ bool q_in_range(double q1, const double (&q2)[W]) {
  const int e1 = __double2hiint(q1) >> 20;   // biased exponent fields (q >= 0): 1..2046 for a normal double
  bool ok = (unsigned)(e1 - 1) < 2046u;
#pragma unroll
  for (int j = 0; j < W; ++j) {
    const int e2 = __double2hiint(q2[j]) >> 20;
    ok &= ((unsigned)(e2 - 1) < 2046u) & ((unsigned)(e1 + e2 - (2046 - 1020)) <= 2039u);
  }
  return ok;
}

#ifndef NNGP_GRAM_ILP
#define NNGP_GRAM_ILP 4   // entries advanced through the layers together (2, 4 or 8): independent dependency chains
#endif                    // (sqrt, reciprocal, two Horner halves each) for the scheduler to interleave; 8 spills
// The diagonals entering step s + 1 (not needed after the last step): ReLU / ABRelu advance them in registers, Erf
// loads them from the per-row tables (an arcsine per entry and step would double the epilogue's transcendental work).
template <int ACT, int W>
__device__ __forceinline__ void advance_diags(double& qa, double (&qb)[W], const GemmParams& p, int s, int r,
                                              int col_base, int n0, double sw2, double sb2) {
  if constexpr (ACT == ACT_ERF) {
    qa = __ldg(p.tab1 + s * p.tld1 + r);
#pragma unroll
    for (int j = 0; j < W / 2; ++j) {
      const int c = col_base + 8 * (n0 + j);
      qb[2 * j] = (c < p.N) ? __ldg(p.tab2 + s * p.tld2 + c) : 0.0;
      qb[2 * j + 1] = (c + 1 < p.N) ? __ldg(p.tab2 + s * p.tld2 + c + 1) : 0.0;
    }
  } else {
#pragma unroll
    for (int j = 0; j < W; ++j) qb[j] = next_diag<ACT>(qb[j], p.act, sw2, sb2);
    qa = next_diag<ACT>(qa, p.act, sw2, sb2);
  }
}

template <int ACT>
__device__ __forceinline__ void gram_epilogue(const double (&acc)[4][4][2], const GemmParams& p, int tile_n, int row_base,
                                              int col_base, int wn, int t) {
  constexpr int W = NNGP_GRAM_ILP;          // entries per group
  constexpr int NG = W / 2;                 // fragments (ni) per group
  double msum[4] = {0.0, 0.0, 0.0, 0.0};  // fused GEMV partial sums (this thread's 8 columns of 4 rows)
#pragma unroll
  for (int mi = 0; mi < 4; ++mi) {
    const int r = row_base + 8 * mi;
    if (r < p.M) {
      const double q1r = p.q1[r];
#pragma unroll
      for (int n0 = 0; n0 < 4; n0 += NG) {
        double k[W], qb[W];
#pragma unroll
        for (int j = 0; j < NG; ++j) {
          const int c = col_base + 8 * (n0 + j);
          k[2 * j] = p.scale * acc[mi][n0 + j][0] + p.sb2;
          k[2 * j + 1] = p.scale * acc[mi][n0 + j][1] + p.sb2;
          qb[2 * j] = (c < p.N) ? __ldg(p.q2 + c) : 0.0;          // re-read per row (L1 hit): keeps registers free
          qb[2 * j + 1] = (c + 1 < p.N) ? __ldg(p.q2 + c + 1) : 0.0;
        }
        double qa = q1r;
        // (Erf has no guarded variant: its input range keeps every step inside atan2_pos' unguarded domain)
        if (!p.ntk) {
          double unused = 0.0;
          for (int s = 0; s < p.steps; ++s) {
            const int li = s < GEMM_MAX_LAYERS ? s : GEMM_MAX_LAYERS - 1;
            const double sw2 = p.lsw2[li], sb2 = p.lsb2[li];
            if (ACT == ACT_ERF || q_in_range<W>(qa, qb)) {
#pragma unroll
              for (int j = 0; j < W; ++j) gram_step<ACT, false, false>(k[j], unused, qa, qb[j], sw2, sb2, p.act);
            } else {
#pragma unroll
              for (int j = 0; j < W; ++j) gram_step<ACT, true, false>(k[j], unused, qa, qb[j], sw2, sb2, p.act);
            }
            if (s + 1 < p.steps) advance_diags<ACT, W>(qa, qb, p, s, r, col_base, n0, sw2, sb2);
          }
        } else {
          double n[W];
#pragma unroll
          for (int j = 0; j < W; ++j) n[j] = k[j];
          for (int s = 0; s < p.steps; ++s) {
            const int li = s < GEMM_MAX_LAYERS ? s : GEMM_MAX_LAYERS - 1;
            const double sw2 = p.lsw2[li], sb2 = p.lsb2[li];
            if (ACT == ACT_ERF || q_in_range<W>(qa, qb)) {
#pragma unroll
              for (int j = 0; j < W; ++j) gram_step<ACT, false, true>(k[j], n[j], qa, qb[j], sw2, sb2, p.act);
            } else {
#pragma unroll
              for (int j = 0; j < W; ++j) gram_step<ACT, true, true>(k[j], n[j], qa, qb[j], sw2, sb2, p.act);
            }
            if (s + 1 < p.steps) advance_diags<ACT, W>(qa, qb, p, s, r, col_base, n0, sw2, sb2);
          }
          if (p.C2) {
#pragma unroll
            for (int j = 0; j < NG; ++j) {
              const int c = col_base + 8 * (n0 + j);
              double* dst2 = p.C2 + (long long)r * p.ldc + c;
              if (c + 1 < p.N) *reinterpret_cast<double2*>(dst2) = make_double2(k[2 * j], k[2 * j + 1]);
              else if (c < p.N) dst2[0] = k[2 * j];
            }
          }
#pragma unroll
          for (int j = 0; j < W; ++j) k[j] = n[j];
        }
#pragma unroll
        for (int j = 0; j < NG; ++j) {
          const int c = col_base + 8 * (n0 + j);
          double* dst = p.C + (long long)r * p.ldc + c;
          if (c + 1 < p.N) {
            *reinterpret_cast<double2*>(dst) = make_double2(k[2 * j], k[2 * j + 1]);
          } else if (c < p.N) {
            dst[0] = k[2 * j];
          }
          if (p.alpha != nullptr) {  // K_* alpha (Theta_* alpha in NTK mode), columns in ascending order
            if (c < p.N) msum[mi] = fma(k[2 * j], __ldg(p.alpha + c), msum[mi]);
            if (c + 1 < p.N) msum[mi] = fma(k[2 * j + 1], __ldg(p.alpha + c + 1), msum[mi]);
          }
        }
      }
    }
  }
  if (p.alpha != nullptr) {  // fixed-order reduction inside the quad, then one partial per (tile, warp column)
#pragma unroll
    for (int mi = 0; mi < 4; ++mi) {
      msum[mi] += __shfl_xor_sync(0xffffffffu, msum[mi], 1);
      msum[mi] += __shfl_xor_sync(0xffffffffu, msum[mi], 2);
      const int r = row_base + 8 * mi;
      if (t == 0 && r < p.M) p.mean_partial[(long long)(2 * tile_n + wn) * p.M + r] = msum[mi];
    }
  }
}

#ifndef NNGP_GEMM_MINBLOCKS
#define NNGP_GEMM_MINBLOCKS 2
#endif
// ACT: the activation of the EPI_GRAM epilogue (GramAct); the other epilogues only exist with the default.
template <int EPI, int ACT = ACT_RELU>
__global__ void __launch_bounds__(GEMM_THREADS, NNGP_GEMM_MINBLOCKS)
gemm_nt_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const GemmParams p) {
  const int tile_n = blockIdx.x;
  const int tile_m = blockIdx.y;
  if (p.lower && tile_n * GEMM_BN > tile_m * GEMM_BM + (GEMM_BM - 1)) return;

  extern __shared__ uint8_t smem_raw[];
  // align the ring to the 1024 B swizzle atom
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t pad = (1024u - (raw_addr & 1023u)) & 1023u;
  uint8_t* ring = smem_raw + pad;
  uint8_t* ringA = ring;
  uint8_t* ringB = ring + GEMM_STAGES * GEMM_A_STAGE_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(ringB + GEMM_STAGES * GEMM_B_STAGE_BYTES);
  uint64_t* empty_bar = full_bar + GEMM_STAGES;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < GEMM_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], GEMM_CONSUMER_WARPS);
    }
    fence_mbar_init();
  }
  __syncthreads();

  int ktiles = p.ktiles;
  int k0 = 0;
  if constexpr (EPI == EPI_ROWDOT) {
    if (p.tri_k) ktiles = min(ktiles, (tile_n + 1) * (GEMM_BN / GEMM_BK));
    if (p.kchunk > 0) {                       // split-K: this CTA owns k-tiles [k0, k0 + ktiles)
      k0 = (int)blockIdx.z * p.kchunk;
      if (k0 >= ktiles) return;               // (before any barrier: the whole CTA leaves)
      ktiles = min(p.kchunk, ktiles - k0);
    }
  }
  TileSrc src;
  src.tmA = &tmA; src.tmB = &tmB;
  src.a_col0 = p.a_col0 + k0 * GEMM_BK; src.a_row = p.a_row0 + tile_m * GEMM_BM;
  src.b_col0 = p.b_col0 + k0 * GEMM_BK; src.b_row = p.b_row0 + tile_n * GEMM_BN;
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    ring_prologue<GEMM_STAGES>(src, ringA, ringB, full_bar, 0, ktiles);  // overlaps the C / q loads below
  }

  const int wm = warp >> 1;  // 0..3 : 32-row slab
  const int wn = warp & 1;   // 0..1 : 32-col slab
  const int g = lane >> 2;   // fragment row / col group
  const int t = lane & 3;    // position inside the group

  const int row_base = tile_m * GEMM_BM + wm * 32 + g;      // + 8*mi
  const int col_base = tile_n * GEMM_BN + wn * 32 + 2 * t;  // + 8*ni (+0/1)

  double acc[4][4][2];
  if constexpr (EPI == EPI_SUB) {
    // start from -C so that the stored result -(acc) = C - A B^T needs no extra registers and
    // the C read overlaps the TMA prologue
#pragma unroll
    for (int mi = 0; mi < 4; ++mi) {
      const int r = row_base + 8 * mi;
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) {
        const int c = col_base + 8 * ni;
        double v0 = 0.0, v1 = 0.0;
        if (r < p.M) {
          const double* src = p.C + (long long)r * p.ldc + c;
          if (c + 1 < p.N) {
            const double2 v = __ldcg(reinterpret_cast<const double2*>(src));  // L2 only: C is produced by other kernels,
            v0 = v.x; v1 = v.y;                                                 // possibly on another stream
          } else if (c < p.N) {
            v0 = __ldcg(src);
          }
        }
        acc[mi][ni][0] = -v0;
        acc[mi][ni][1] = -v1;
      }
    }
  } else {
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) { acc[mi][ni][0] = 0.0; acc[mi][ni][1] = 0.0; }
  }

  int stage = 0;
  uint32_t phase = 0;
  if constexpr (EPI == EPI_ROWDOT) {
    // small batches (latency mode): a 32-row slab without a valid row skips its fragment loads and DMMAs
    const bool slab_active = tile_m * GEMM_BM + wm * 32 < p.M;
    mma_mainloop<GEMM_STAGES>(acc, src, ringA, ringB, full_bar, empty_bar, stage, phase, ktiles, wm, wn, lane, p.zero,
                              NoGate(), slab_active);
  } else {
    mma_mainloop<GEMM_STAGES>(acc, src, ringA, ringB, full_bar, empty_bar, stage, phase, ktiles, wm, wn, lane, p.zero);
  }

  // ===== epilogue (registers -> global) =====
  // The tile coordinates are laundered through an empty asm so that the compiler re-derives the output addresses
  // here instead of keeping the prologue's pointers alive (in registers or spilled) across the main loop.
  int row_base_e = row_base, col_base_e = col_base;
  asm volatile("" : "+r"(row_base_e), "+r"(col_base_e));
  if constexpr (EPI == EPI_SUB) {
#pragma unroll
    for (int mi = 0; mi < 4; ++mi) {
      const int r = row_base_e + 8 * mi;
      if (r >= p.M) continue;
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) {
        const int c = col_base_e + 8 * ni;
        double* dst = p.C + (long long)r * p.ldc + c;
        if (c + 1 < p.N) {
          *reinterpret_cast<double2*>(dst) = make_double2(-acc[mi][ni][0], -acc[mi][ni][1]);
        } else if (c < p.N) {
          dst[0] = -acc[mi][ni][0];
        }
      }
    }
  } else if constexpr (EPI == EPI_DIAG) {
    __syncthreads();  // every warp has left the ring: its first 2 KiB become the row-sum scratch
    DiagOut o;
    o.B = p.C; o.ldb = p.ldc; o.rows = p.M; o.ssq = p.ssq; o.kss = p.kss; o.var = p.var; o.J = p.J; o.col_blocks = p.col_blocks;
    diag_epilogue(acc, o, tile_m * GEMM_BM, p.N, wm, wn, g, t, reinterpret_cast<double*>(ringA));
  } else if constexpr (EPI == EPI_ROWDOT) {
    if (p.kchunk > 0) {   // split-K: hand the partial products to the reduction kernel
#pragma unroll
      for (int mi = 0; mi < 4; ++mi) {
        const int r = row_base_e + 8 * mi;
        if (r >= p.M) continue;
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) {
          const int c = col_base_e + 8 * ni;
          double* dst = p.vpart + ((long long)blockIdx.z * p.M + r) * p.N + c;
          if (c < p.N) dst[0] = acc[mi][ni][0];
          if (c + 1 < p.N) dst[1] = acc[mi][ni][1];
        }
      }
      return;
    }
    // quad[r] contribution of this 64-column tile: sum_c acc[r][c] * W[r][c]  (fixed order => deterministic)
    double part[4];
#pragma unroll
    for (int mi = 0; mi < 4; ++mi) {
      const int r = row_base_e + 8 * mi;
      double sacc = 0.0;
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) {
        const int c = col_base_e + 8 * ni;
        double w0 = 0.0, w1 = 0.0;
        if (p.W == nullptr) {                 // squares: columns beyond N hold exact zeros (zero-filled operand rows)
          w0 = acc[mi][ni][0]; w1 = acc[mi][ni][1];
        } else if (r < p.M) {
          const double* src = p.W + (long long)r * p.ldc + c;
          if (c + 1 < p.N) {
            const double2 v = *reinterpret_cast<const double2*>(src);
            w0 = v.x; w1 = v.y;
          } else if (c < p.N) {
            w0 = src[0];
          }
        }
        sacc = fma(acc[mi][ni][0], w0, sacc);
        sacc = fma(acc[mi][ni][1], w1, sacc);
      }
      sacc += __shfl_xor_sync(0xffffffffu, sacc, 1);
      sacc += __shfl_xor_sync(0xffffffffu, sacc, 2);
      part[mi] = sacc;
    }
    __syncthreads();  // every warp has left the ring
    double* red = reinterpret_cast<double*>(ringA);                              // [2][128]
    if (t == 0) {
#pragma unroll
      for (int mi = 0; mi < 4; ++mi) red[wn * GEMM_BM + wm * 32 + mi * 8 + g] = part[mi];
    }
    __syncthreads();
    if (threadIdx.x < GEMM_BM) {
      const int r = tile_m * GEMM_BM + threadIdx.x;
      if (r < p.M) p.partial[(long long)tile_n * p.M + r] = red[threadIdx.x] + red[GEMM_BM + threadIdx.x];
    }
  } else {
    gram_epilogue<ACT>(acc, p, tile_n, row_base_e, col_base_e, wn, t);
  }
}

}  // namespace nngp
