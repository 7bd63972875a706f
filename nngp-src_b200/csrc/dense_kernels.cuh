// dense_kernels.cuh -- the small kernels around the DMMA GEMM core:
//   row_sqnorm / q_final          layer-0 kernel diagonal and K(x,x)            (K2, K9)
//   diag_reg                      lambda = diag_reg * trace(K)/N ; K += lambda I (K4)
//   potf2_64_block                64x64 diagonal-block Cholesky, 4 x 4 register blocks            (K5 panel)
//   trtri_diag                    inv(L_JJ) of every diagonal block: operand of the solves' diagonal step (K10)
//   trsv_bwd_persistent / _step   backward substitution L^T alpha = z (the forward one rides through
//                                 the Cholesky as an extra row of the factor buffer)              (K6)
//   mean_reduce                   finishes mean = K_* alpha (the GEMV itself is fused into the Gram epilogue) (K8)
//   rowdot / ntk_var / transpose  NTK-mode variance pieces;  lml_terms, finite_check, zero_upper, dmma_peak
// All reductions have a fixed order: results are bitwise reproducible and independent of how
// test rows are sharded over GPUs.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace nngp {

constexpr int NB = 64;  // diagonal block size of the blocked factorisation / solves

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// q[r] = sw2 * sum_j x[r][j]^2 / D + sb2 ; one warp per row.
// range_flag (optional): |= 2 when some q >= 2^512 (or overflows): the Gram epilogue forms q q', which must stay finite.
constexpr double Q_LIMIT = 0x1p+512;
__global__ void row_sqnorm_kernel(const double* __restrict__ x, long long ldx, int rows, int D, double sw2,
                                  double sb2, double* __restrict__ q, int* __restrict__ range_flag = nullptr) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const double* xr = x + (long long)warp * ldx;
  double s = 0.0;
  for (int j = lane; j < D; j += 32) {
    const double v = xr[j];
    s = fma(v, v, s);
  }
  s = warp_sum(s);
  if (lane == 0) {
    const double v = sw2 * (s / (double)D) + sb2;
    q[warp] = v;
    if (range_flag && !(v < Q_LIMIT)) atomicOr(range_flag, 2);
  }
}

// kss[r] = layer-(depth-1) diagonal: q <- sw2_s*q/2 + sb2_s for the Dense layer that follows arc-cosine step s.
struct LayerSig {
  double sw2[16], sb2[16];   // entry min(s, 15)
};
__global__ void q_final_kernel(const double* __restrict__ q, int rows, int steps, LayerSig sig, double* __restrict__ kss) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows) return;
  double v = q[i];
  for (int s = 0; s < steps; ++s) {
    const int li = s < 16 ? s : 15;
    v = sig.sw2[li] * (0.5 * v) + sig.sb2[li];
  }
  kss[i] = v;
}

// Single CTA: lambda = reg * (absolute ? 1 : trace(K)/N); K[i][i] += lambda.  lambda -> *lambda_out.
__global__ void diag_reg_kernel(double* __restrict__ K, long long ld, int N, double reg, int absolute,
                                double* __restrict__ lambda_out) {
  __shared__ double red[32];
  __shared__ double lam_s;
  double s = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) s += K[(long long)i * ld + i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    double v = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.0;
    v = warp_sum(v);
    if (threadIdx.x == 0) {
      const double r = reg > 0.0 ? reg : 0.0;
      lam_s = absolute ? r : r * (v / (double)N);
      *lambda_out = lam_s;
    }
  }
  __syncthreads();
  const double lam = lam_s;
  for (int i = threadIdx.x; i < N; i += blockDim.x) K[(long long)i * ld + i] += lam;
}

// In-place lower Cholesky of the n x n (n <= 64) block at A (row-major, ld).  One CTA of 256 threads as a 16 x 16
// grid, thread (ty, tx) owning the 4 x 4 register block of rows 4ty.., columns 4tx...  Right-looking over 4-column
// micro-panels, two barriers per micro-panel (32 in all):
//   A  the diagonal thread factors its 4 x 4 block in registers and publishes it with the reciprocal pivots
//      (pivot column scaled by the reciprocal pivot as LAPACK dpotf2 does, one rsqrt each);
//   B  the threads below it finish their 4 columns (scale, update the later columns of the micro-panel) and publish them;
//   C  every trailing block applies the four rank-1 updates, column by column.
// Every element sees exactly the FMA sequence of the unblocked column-by-column algorithm (ascending j), so the
// factor is bitwise that of the one-column-per-step version this replaces (34 us -> 10 us per block).
// On a non-positive pivot: *info = global pivot index + 1 (first failure wins), block left as is.
constexpr int POTF2_THREADS = 256;
// In-place inverse of the lower-triangular 64 x 64 block in Ls (identity padded, zeros above the diagonal), by all 256
// threads of the CTA, as a recursive block inversion:  inv [[A, 0], [B, C]] = [[A^-1, 0], [-C^-1 B A^-1, C^-1]].
// Level 0 inverts the sixteen 4 x 4 diagonal blocks (one thread each); levels M = 4, 8, 16, 32 fill the off-diagonal
// M x M blocks of every 2M x 2M diagonal super-block with two small products (T = B A^-1 into the scratch `T`, then
// -C^-1 T over B: the region that held B is exactly where the result belongs, so no second matrix is needed).
// Each thread owns S = M/8 adjacent outputs of a row and runs the FULLY UNROLLED dense k loop (the zeros above the
// diagonals of A^-1 / C^-1 make the triangular bounds unnecessary), so the shared-memory loads pipeline instead of
// serialising behind a loop-carried bound: 9 barriers, ~2 us, against ~12 us with data-dependent trip counts and
// ~20 us for a column-wise forward substitution (a 64-step chain of divisions and shuffles) -- this sits on the
// critical path of the Cholesky panel chain.  `T`: 1024 doubles.
// The same routine serves the factorisation (potf2_64_block) and imported states (trtri_diag_kernel): same bits.
template <int M>
__device__ __forceinline__ void invert_level(double (*Ls)[NB + 1], double* __restrict__ T) {
  constexpr int S = M >= 8 ? M / 8 : 1;          // outputs per thread
  constexpr int GROUPS = M / S;                  // thread groups per output row
  constexpr int NTHR = (NB / (2 * M)) * M * GROUPS;   // 256 for M >= 8, 128 for M = 4
  const int tid = threadIdx.x;
  const int pr = tid / (M * GROUPS), rem = tid - pr * (M * GROUPS), i = rem / GROUPS, j0 = (rem - i * GROUPS) * S;
  const int a0 = pr * 2 * M, c0 = a0 + M;
  double acc[S];
  if (tid < NTHR) {     // T = B A^-1
#pragma unroll
    for (int s = 0; s < S; ++s) acc[s] = 0.0;
#pragma unroll
    for (int k = 0; k < M; ++k) {
      const double b = Ls[c0 + i][a0 + k];
#pragma unroll
      for (int s = 0; s < S; ++s) acc[s] = fma(b, Ls[a0 + k][a0 + j0 + s], acc[s]);
    }
#pragma unroll
    for (int s = 0; s < S; ++s) T[pr * M * M + i * M + j0 + s] = acc[s];
  }
  __syncthreads();
  if (tid < NTHR) {     // B <- -C^-1 T
#pragma unroll
    for (int s = 0; s < S; ++s) acc[s] = 0.0;
#pragma unroll
    for (int k = 0; k < M; ++k) {
      const double c = Ls[c0 + i][c0 + k];
#pragma unroll
      for (int s = 0; s < S; ++s) acc[s] = fma(c, T[pr * M * M + k * M + j0 + s], acc[s]);
    }
#pragma unroll
    for (int s = 0; s < S; ++s) Ls[c0 + i][a0 + j0 + s] = -acc[s];
  }
  __syncthreads();
}

__device__ __forceinline__ void invert_lower_64_inplace(double (*Ls)[NB + 1], double* __restrict__ T) {
  const int tid = threadIdx.x;
  if (tid < NB / 4) {
    const int o = 4 * tid;
    const double l10 = Ls[o + 1][o], l20 = Ls[o + 2][o], l21 = Ls[o + 2][o + 1];
    const double l30 = Ls[o + 3][o], l31 = Ls[o + 3][o + 1], l32 = Ls[o + 3][o + 2];
    const double r0 = 1.0 / Ls[o][o], r1 = 1.0 / Ls[o + 1][o + 1], r2 = 1.0 / Ls[o + 2][o + 2], r3 = 1.0 / Ls[o + 3][o + 3];
    const double w10 = -(l10 * r0) * r1;
    const double w21 = -(l21 * r1) * r2;
    const double w32 = -(l32 * r2) * r3;
    const double w20 = -fma(l21, w10, l20 * r0) * r2;
    const double w31 = -fma(l32, w21, l31 * r1) * r3;
    const double w30 = -fma(l32, w20, fma(l31, w10, l30 * r0)) * r3;
    Ls[o][o] = r0; Ls[o + 1][o + 1] = r1; Ls[o + 2][o + 2] = r2; Ls[o + 3][o + 3] = r3;
    Ls[o + 1][o] = w10; Ls[o + 2][o] = w20; Ls[o + 2][o + 1] = w21;
    Ls[o + 3][o] = w30; Ls[o + 3][o + 1] = w31; Ls[o + 3][o + 2] = w32;
  }
  __syncthreads();
  invert_level<4>(Ls, T);
  invert_level<8>(Ls, T);
  invert_level<16>(Ls, T);
  invert_level<32>(Ls, T);
}

// Ls (inverse, lower) -> global row-major 64 x 64 block (upper part written as zeros), coalesced.
__device__ __forceinline__ void store_inverse_64(const double (*Ls)[NB + 1], double* __restrict__ Wout) {
  for (int idx = threadIdx.x; idx < NB * NB; idx += blockDim.x) {
    const int r = idx >> 6, c = idx & 63;
    Wout[idx] = (c <= r) ? Ls[r][c] : 0.0;
  }
}

// Shared memory of one 64 x 64 block factorisation (45.9 KB), aliased onto the drained operand ring in the fused
// panel kernel (potrf_panel.cuh).
struct Potf2Smem {
  double Ld[2][4][4];     // factored diagonal 4 x 4 block (lower), double-buffered by micro-panel parity
  double Rinv[2][4];      // reciprocal pivots of its 4 columns
  double P[2][NB][4];     // the finished micro-panel: P[.][r][ja] = L[r][4 jb + ja]
  int s_bad[2];
  double Ls[NB][NB + 1];  // the factored block, then its inverse
  double T[16 * NB];      // scratch of the block inversion
};

// The block-wide routine (256 threads): factor, store, and -- `Winv` optional -- also write inv(L_JJ) (64 x 64 row-major,
// identity padded), the operand of the DMMA panel solve below the block and of the prediction solves' diagonal step.
// Returns 0, or the 1-based pivot index inside the block on a non-positive pivot (block-uniform; *info is set).
__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ int potf2_64_block(double* __restrict__ A, long long ld, int n, int pivot0, int* __restrict__ info,
                                              double* __restrict__ Winv, Potf2Smem& sm,
                                              unsigned long long* trace = nullptr) {
  double (&Ld)[2][4][4] = sm.Ld;
  double (&Rinv)[2][4] = sm.Rinv;
  double (&P)[2][NB][4] = sm.P;
  int (&s_bad)[2] = sm.s_bad;
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  double v[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int r = ty * 4 + a, c = tx * 4 + b;
      v[a][b] = (r < n && c <= r) ? __ldcg(A + (long long)r * ld + c) : ((r == c) ? 1.0 : 0.0);
    }
  if (tid < 2) s_bad[tid] = 0;
  __syncthreads();
#ifdef NNGP_PANEL_TRACE
  if (trace != nullptr && tid == 0) trace[1] = global_timer_ns();   // block loaded
#endif
  const int nblk = (n + 3) >> 2;
  // A(jb): the thread that owns diagonal block jb factors its 4 x 4 block in registers and publishes it (buffer jb & 1)
  auto factor_diag = [&](int jb) {
    const int buf = jb & 1;
    int badj = 0;
#pragma unroll
    for (int ja = 0; ja < 4; ++ja) {
      const double d = v[ja][ja];
      if (!(d > 0.0) && badj == 0 && jb * 4 + ja < n) badj = jb * 4 + ja + 1;  // also catches NaN
      const double rinv = rsqrt(d);
      Rinv[buf][ja] = rinv;
      double l[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) l[a] = (a > ja) ? v[a][ja] * rinv : 0.0;
      v[ja][ja] = d * rinv;
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        if (a > ja) v[a][ja] = l[a];
#pragma unroll
        for (int b = 0; b < 4; ++b) v[a][b] = fma(-l[a], l[b], v[a][b]);
      }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) Ld[buf][a][b] = v[a][b];
    if (badj) s_bad[buf] = badj;
  };
  // Schedule: A(0); then per micro-panel  B(jb) | barrier | C(jb) with A(jb+1) folded in | barrier.  The 4 x 4 factor
  // of the NEXT diagonal block -- four dependent rsqrt-scale-update steps on one thread, the longest phase -- runs
  // right after that thread's own rank-4 update, beside the other threads' updates, instead of as a phase of its own
  // (2 barriers per micro-panel as before, but a third less on the critical path).  Per element the operations and
  // their order are unchanged: same bits.
  if (ty == 0 && tx == 0) factor_diag(0);
  __syncthreads();
  for (int jb = 0; jb < nblk; ++jb) {
    const int buf = jb & 1;
#ifdef NNGP_PANEL_TRACE
    if (trace != nullptr && tid == 0 && (jb == 8 || jb == 9)) trace[2 + 3 * (jb - 8)] = global_timer_ns();      // A(jb) visible
#endif
    if (s_bad[buf]) {  // CTA-uniform exit
      if (tid == 0) atomicCAS(info, 0, pivot0 + s_bad[buf]);
      return s_bad[buf];
    }
    if (tx == jb && ty > jb) {  // B: the micro-panel below the diagonal block
#pragma unroll
      for (int ja = 0; ja < 4; ++ja) {
        const double rinv = Rinv[buf][ja];
        double l[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          l[a] = v[a][ja] * rinv;
          v[a][ja] = l[a];
        }
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const double lc = (b > ja) ? Ld[buf][b][ja] : 0.0;
#pragma unroll
          for (int a = 0; a < 4; ++a) v[a][b] = fma(-l[a], lc, v[a][b]);
        }
      }
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int ja = 0; ja < 4; ++ja) P[buf][ty * 4 + a][ja] = v[a][ja];
    }
    __syncthreads();
#ifdef NNGP_PANEL_TRACE
    if (trace != nullptr && tid == 0 && (jb == 8 || jb == 9)) trace[3 + 3 * (jb - 8)] = global_timer_ns();      // B done
#endif
    if (tx > jb && ty >= tx) {  // C: trailing blocks (lower part), four rank-1 updates in column order
#pragma unroll
      for (int ja = 0; ja < 4; ++ja) {
        double lr[4], lc[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) lr[a] = P[buf][ty * 4 + a][ja];
#pragma unroll
        for (int b = 0; b < 4; ++b) lc[b] = P[buf][tx * 4 + b][ja];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) v[a][b] = fma(-lr[a], lc[b], v[a][b]);
      }
      if (tx == jb + 1 && ty == jb + 1 && jb + 1 < nblk) factor_diag(jb + 1);   // A(jb+1), into the OTHER buffer
    }
    __syncthreads();
#ifdef NNGP_PANEL_TRACE
    if (trace != nullptr && tid == 0 && (jb == 8 || jb == 9)) trace[4 + 3 * (jb - 8)] = global_timer_ns();      // C + A(jb+1) done
#endif
  }
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int r = ty * 4 + a, c = tx * 4 + b;
      if (r < n && c <= r) A[(long long)r * ld + c] = v[a][b];
    }
#ifdef NNGP_PANEL_TRACE
  if (trace != nullptr && tid == 0) { trace[0] = global_timer_ns(); }   // factor done
#endif
  if (Winv != nullptr) {
    double (*Ls)[NB + 1] = sm.Ls;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int r = ty * 4 + a, c = tx * 4 + b;
        Ls[r][c] = (r < n && c <= r) ? v[a][b] : ((r == c) ? 1.0 : 0.0);
      }
    __syncthreads();
    invert_lower_64_inplace(Ls, sm.T);
    store_inverse_64(Ls, Winv);
  }
  return 0;
}

// W_J = inv(L_JJ) for every 64 x 64 diagonal block of the factor (identity padded when the last block is short):
// one CTA per block, the SAME routine (invert_lower_64_inplace) the factorisation's potf2_64_block runs on the block it has
// just factored -- so a state that was imported (nngp_set_state / nngp_state_import_end) predicts with bitwise the
// inverses of the handle that fitted it.  Output: row-major 64 x 64 blocks stacked along the rows (block J at rows
// [64 J, 64 J + 64)), the B operand of the diagonal step of the row-wise triangular solves.
__global__ void __launch_bounds__(POTF2_THREADS) trtri_diag_kernel(const double* __restrict__ L, long long ldl, int N,
                                                                   double* __restrict__ Winv) {
  __shared__ double Ls[NB][NB + 1];
  __shared__ double Tscratch[16 * NB];
  const int J = blockIdx.x;
  const int j0 = J * NB;
  const int n = min(NB, N - j0);
  const int c = threadIdx.x & 63, rsub = threadIdx.x >> 6;
  for (int r = rsub; r < NB; r += 4)
    Ls[r][c] = (r < n && c <= r) ? L[(long long)(j0 + r) * ldl + j0 + c] : ((r == c) ? 1.0 : 0.0);
  __syncthreads();
  invert_lower_64_inplace(Ls, Tscratch);
  store_inverse_64(Ls, Winv + (long long)j0 * NB);
}

// Shared helper: load the n x n lower block Ljj into Ls (identity padded), 8 loads in flight per thread,
// and the reciprocal diagonal into rd.  blockDim.x must be 256.
__device__ __forceinline__ void load_diag_block(const double* __restrict__ Ljj, long long ldl, int n,
                                                double (*Ls)[NB + 1], double* rd) {
  const int c = threadIdx.x & 63, rsub = threadIdx.x >> 6;  // 4 row phases
  for (int r0 = 0; r0 < NB; r0 += 32) {
    double t[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int r = r0 + 4 * u + rsub;
      t[u] = (r < n && c <= r) ? Ljj[(long long)r * ldl + c] : ((r == c) ? 1.0 : 0.0);
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) Ls[r0 + 4 * u + rsub][c] = t[u];
  }
  __syncthreads();
  if (threadIdx.x < NB) rd[threadIdx.x] = 1.0 / Ls[threadIdx.x][threadIdx.x];
}

constexpr int TRSV_THREADS = 256;

// Backward step of L^T a = z for diagonal block [j0, j0+n): every CTA solves Ljj^T a_J = z_J
// redundantly, CTA 0 publishes a_J into aout (not into z, which other CTAs may still be reading), and all CTAs apply z[c] -= sum_i L[j0+i][c] a_i to the
// columns c < j0 (one thread per column, coalesced row reads).
__global__ void __launch_bounds__(TRSV_THREADS) trsv_bwd_step_kernel(const double* __restrict__ L, long long ld,
                                                                    int j0, int n, double* __restrict__ z,
                                                                    double* __restrict__ aout) {
  __shared__ double Ls[NB][NB + 1];
  __shared__ double as[NB];
  __shared__ double rd[NB];
  load_diag_block(L + (long long)j0 * ld + j0, ld, n, Ls, rd);
  if (threadIdx.x < NB) as[threadIdx.x] = (threadIdx.x < n) ? z[j0 + threadIdx.x] : 0.0;
  __syncthreads();
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    double y0 = as[lane], y1 = as[lane + 32];
    for (int k = NB - 1; k >= 0; --k) {
      const double num = __shfl_sync(0xffffffffu, (k < 32) ? y0 : y1, k & 31);
      const double ak = num * rd[k];
      if (lane == (k & 31)) { if (k < 32) y0 = ak; else y1 = ak; }
      if (lane < k) y0 = fma(-Ls[k][lane], ak, y0);
      if (lane + 32 < k) y1 = fma(-Ls[k][lane + 32], ak, y1);
    }
    as[lane] = y0;
    as[lane + 32] = y1;
  }
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x < n) aout[j0 + threadIdx.x] = as[threadIdx.x];
  for (long long c = (long long)blockIdx.x * TRSV_THREADS + threadIdx.x; c < j0;
       c += (long long)gridDim.x * TRSV_THREADS) {
    const double* lc = L + (long long)j0 * ld + c;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    for (int i0 = 0; i0 < NB; i0 += 16) {
      double t[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) t[u] = (i0 + u < n) ? lc[(long long)(i0 + u) * ld] : 0.0;
#pragma unroll
      for (int u = 0; u < 16; u += 4) {
        s0 = fma(t[u], as[i0 + u], s0);
        s1 = fma(t[u + 1], as[i0 + u + 1], s1);
        s2 = fma(t[u + 2], as[i0 + u + 2], s2);
        s3 = fma(t[u + 3], as[i0 + u + 3], s3);
      }
    }
    z[c] -= (s0 + s1) + (s2 + s3);
  }
}

// The whole backward substitution  L^T a = z  as ONE kernel (the stepwise version above costs one launch per 64-row
// block: N/64 launches of ~15 us on a serial chain).  CTA k owns the SW-column slice [k SW, (k+1) SW) of z in shared
// memory, SW a multiple of 64 chosen so that all CTAs are co-resident (grid <= #SMs, asserted by the host).  Blocks
// J = N/64-1 ... 0 in order:  the CTA that owns block J's columns has, by then, applied every earlier update to
// them; it solves L_JJ^T a_J = z_J (the same warp-shuffle substitution as the stepwise kernel), writes a_J to `aout`
// and releases flag[J];  every CTA with columns below block J acquires the flag and applies
// z[c] -= sum_i L[64J+i][c] a_i  to its own columns (the L strip is loaded BEFORE the wait, so its latency hides
// behind the chain).  Per column the arithmetic and its order are exactly those of the stepwise kernel => same bits.
// Spins are bounded: a scheduling bug traps instead of hanging the GPU.
constexpr int TRSVP_THREADS = 256;
__global__ void __launch_bounds__(TRSVP_THREADS) trsv_bwd_persistent_kernel(const double* __restrict__ L, long long ld,
                                                                            int N, int SW, const double* __restrict__ z,
                                                                            double* __restrict__ aout, int* flags,
                                                                            const double* __restrict__ Winv) {
  extern __shared__ double sm[];
  double(*red)[NB] = reinterpret_cast<double(*)[NB]>(sm);            // [4][64] partial sums of the block solve
  double* as = sm + NB * (NB + 1);                                   // [64]
  double* rd = as + NB;                                              // [64] (unused since the block solve is a product)
  double* zs = rd + NB;                                              // [SW]
  const int tid = threadIdx.x;
  // slices are handed out back to front: the CTAs scheduled first own the blocks that are solved first, so a CTA
  // only ever waits for CTAs with a LOWER blockIdx
  const int c0 = (int)(gridDim.x - 1 - blockIdx.x) * SW;
  const int c1 = min(c0 + SW, N);
  for (int c = tid; c < SW; c += TRSVP_THREADS) zs[c] = (c0 + c < N) ? z[c0 + c] : 0.0;
  const int nblk = (N + NB - 1) / NB;
  const int my_first_blk = c0 / NB;   // the lowest block whose columns this CTA owns
  __syncthreads();
  for (int J = nblk - 1; J >= my_first_blk; --J) {
    const int j0 = J * NB;
    const int n = min(NB, N - j0);
    const bool owner = j0 >= c0 && j0 < c1;
    if (owner) {
      // L_JJ^T a_J = r_J  as  a_J = W_J^T r_J  with the block inverse the factorisation left in Winv (the operand the
      // prediction solves use): 16 multiply-adds per thread and one barrier instead of a 64-step substitution chain
      // (3 us of every block step were this solve; the chain of N/64 steps is what bounds the kernel).
      const int i = tid & 63, part = tid >> 6;
      const double* wj = Winv + (long long)j0 * NB;                  // 64 x 64 row-major, identity padded
      double w[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) w[u] = __ldcg(wj + (long long)(part * 16 + u) * NB + i);
      double acc = 0.0;
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        const int k = part * 16 + u;
        acc = fma(w[u], (k < n) ? zs[j0 - c0 + k] : 0.0, acc);       // a_i = sum_k W[k][i] r[k]   (W lower: k >= i)
      }
      red[part][i] = acc;
      __syncthreads();
      if (tid < NB) as[tid] = (red[0][tid] + red[1][tid]) + (red[2][tid] + red[3][tid]);
      __syncthreads();
      if (tid < n) aout[j0 + tid] = as[tid];
      __threadfence();
      __syncthreads();
      if (tid == 0) asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(flags + J), "r"(1) : "memory");
    }
    // columns of this CTA below block J:  [c0, min(c1, j0))
    const int ce = min(c1, j0);
    for (int cb = c0; cb < ce; cb += TRSVP_THREADS) {
      const int c = cb + tid;
      double t[NB];
      if (c < ce) {
        const double* lc = L + (long long)j0 * ld + c;
#pragma unroll
        for (int i = 0; i < NB; ++i) t[i] = (i < n) ? __ldcg(lc + (long long)i * ld) : 0.0;
      }
      if (!owner && cb == c0) {   // a_J comes from another CTA: wait for it (once per step), then stage it
        if (tid == 0) {
          int v;
          unsigned spin = 0;
          do {
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(flags + J) : "memory");
            if (v == 0) { __nanosleep(32); if (++spin > (1u << 27)) __trap(); }
          } while (v == 0);
        }
        __syncthreads();
        if (tid < NB) as[tid] = (tid < n) ? __ldcg(aout + j0 + tid) : 0.0;
        __syncthreads();
      }
      if (c < ce) {
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
        for (int i0 = 0; i0 < NB; i0 += 16) {
#pragma unroll
          for (int u = 0; u < 16; u += 4) {
            s0 = fma(t[i0 + u], as[i0 + u], s0);
            s1 = fma(t[i0 + u + 1], as[i0 + u + 1], s1);
            s2 = fma(t[i0 + u + 2], as[i0 + u + 2], s2);
            s3 = fma(t[i0 + u + 3], as[i0 + u + 3], s3);
          }
        }
        zs[c - c0] -= (s0 + s1) + (s2 + s3);
      }
    }
    __syncthreads();   // zs / as settled before the next block
  }
}

// Single CTA (1024 threads), fixed-order reductions for the log marginal likelihood:
//   out[0] = sum_i log L[i][i]     out[1] = sum_i z[i]^2  (= y^T (K + lambda I)^-1 y with z = L^-1 y)
__global__ void lml_terms_kernel(const double* __restrict__ L, long long ld, int N, const double* __restrict__ z,
                                 double* __restrict__ out) {
  __shared__ double red[2][32];
  double s0 = 0.0, s1 = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    s0 += log(L[(long long)i * ld + i]);
    const double v = z[i];
    s1 = fma(v, v, s1);
  }
  s0 = warp_sum(s0);
  s1 = warp_sum(s1);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s0; red[1][threadIdx.x >> 5] = s1; }
  __syncthreads();
  if (threadIdx.x < 32) {
    double a = (threadIdx.x < (blockDim.x >> 5)) ? red[0][threadIdx.x] : 0.0;
    double b = (threadIdx.x < (blockDim.x >> 5)) ? red[1][threadIdx.x] : 0.0;
    a = warp_sum(a);
    b = warp_sum(b);
    if (threadIdx.x == 0) { out[0] = a; out[1] = b; }
  }
}

// out[r] = sum_j A[r][j] * B[r][j]; one warp per row (NTK cross term  w_i^T k_i = v_i . u_i).
__global__ void rowdot_kernel(const double* __restrict__ A, const double* __restrict__ B, long long ld, int rows, int N,
                              double* __restrict__ out) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const double* a = A + (long long)warp * ld;
  const double* b = B + (long long)warp * ld;
  double s0 = 0.0, s1 = 0.0;
  int j = 2 * lane;
  for (; j + 65 < N; j += 128) {
    const double2 a0 = *reinterpret_cast<const double2*>(a + j), b0 = *reinterpret_cast<const double2*>(b + j);
    const double2 a1 = *reinterpret_cast<const double2*>(a + j + 64), b1 = *reinterpret_cast<const double2*>(b + j + 64);
    s0 = fma(a0.x, b0.x, s0); s0 = fma(a0.y, b0.y, s0);
    s1 = fma(a1.x, b1.x, s1); s1 = fma(a1.y, b1.y, s1);
  }
  for (; j < N; j += 64) {
    s0 = fma(a[j], b[j], s0);
    if (j + 1 < N) s0 = fma(a[j + 1], b[j + 1], s0);
  }
  const double s = warp_sum(s0 + s1);
  if (lane == 0) out[warp] = s;
}

// mean[r] = sum_t partial[t][r]: finishes the posterior-mean GEMV that the Gram epilogue fused (tiles in index order)
__global__ void mean_reduce_kernel(const double* __restrict__ partial, int tiles, int rows, double* __restrict__ mean) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  double s = 0.0;
  int t = 0;
  for (; t + 8 <= tiles; t += 8) {       // 8 loads in flight, added in tile order: the same sum, without 8 serial misses
    double b[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) b[u] = partial[(long long)(t + u) * rows + r];
#pragma unroll
    for (int u = 0; u < 8; ++u) s += b[u];
  }
  for (; t < tiles; ++t) s += partial[(long long)t * rows + r];
  mean[r] = s;
}

// NTK posterior variance: var[r] = kss[r] + sum_t partial[t][r] - 2 cross[r]   (tiles summed in index order)
__global__ void ntk_var_kernel(const double* __restrict__ kss, const double* __restrict__ partial, int tiles, int rows,
                               const double* __restrict__ cross, double* __restrict__ var) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  double q = 0.0;
  for (int t = 0; t < tiles; ++t) q += partial[(long long)t * rows + r];
  var[r] = kss[r] + q - 2.0 * cross[r];
}

// latency mode: var[r] = kss[r] - sum_t partial[t][r]   (tiles summed in index order: deterministic)
__global__ void var_from_partial_kernel(const double* __restrict__ kss, const double* __restrict__ partial, int tiles,
                                        int rows, double* __restrict__ var) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  double q = 0.0;
  for (int t = 0; t < tiles; ++t) q += partial[(long long)t * rows + r];
  var[r] = kss[r] - q;
}

// latency mode, split-K variant (few rows): var[r] = kss[r] - sum_c ( sum_z vpart[z][r][c] )^2, one CTA per row.
// Column c lies in column tile c / 64, whose triangular product spans 4 (c / 64 + 1) k-tiles, i.e.
// ceil(that / kchunk) chunks were written.  Fixed summation order: deterministic.
__global__ void __launch_bounds__(256) var_from_split_kernel(const double* __restrict__ kss, const double* __restrict__ vpart,
                                                             int rows, int N, int ktiles_total, int kchunk,
                                                             double* __restrict__ var) {
  __shared__ double red[256];
  const int r = blockIdx.x;
  double sacc = 0.0;
  if (kchunk >= ktiles_total) {          // a single chunk (tri_gemv path): plain strided sum of squares, loads batched
    const double* vr = vpart + (long long)r * N;
    int c = threadIdx.x;
    for (; c + 3 * 256 < N; c += 4 * 256) {
      const double v0 = vr[c], v1 = vr[c + 256], v2 = vr[c + 512], v3 = vr[c + 768];
      sacc = fma(v0, v0, sacc); sacc = fma(v1, v1, sacc); sacc = fma(v2, v2, sacc); sacc = fma(v3, v3, sacc);
    }
    for (; c < N; c += 256) { const double v0 = vr[c]; sacc = fma(v0, v0, sacc); }
  } else {
    for (int c = threadIdx.x; c < N; c += 256) {
      const int kt = min(ktiles_total, (c / 64 + 1) * 4);
      const int nz = (kt + kchunk - 1) / kchunk;
      double v = 0.0;
      for (int z = 0; z < nz; ++z) v += vpart[((long long)z * rows + r) * N + c];
      sacc = fma(v, v, sacc);
    }
  }
  red[threadIdx.x] = sacc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) var[r] = kss[r] - red[0];
}

// latency mode, a handful of queries (rows <= 8): v[r][j] = sum_{k <= j} W[j][k] ks[r][k] with W = L^-1 (lower, row-
// major) as a matrix-vector product that streams W exactly once -- the HBM floor of the request (4 N^2 bytes) --
// instead of pushing a 128-row DMMA tile that is 99 % padding through the tensor pipe.  A CTA takes a group of 8
// consecutive rows of W, one per warp, paired with the mirrored group from the other end of the matrix so that every
// CTA streams the same number of bytes; the query rows are staged in shared memory one k-chunk at a time and shared by
// the 8 warps.  Lane l accumulates k = 2 l, 2 l + 1 (+ 64, ...) and the warp combines with a fixed xor tree:
// deterministic.  Output: v[r * N + j] (squared and row-reduced by var_from_split_kernel with a single chunk).
constexpr int TGV_MAXR = 8;
constexpr int TGV_SMEM_DOUBLES = 4096;            // staged query values per k-chunk: R x KC, KC = 4096 / R
template <int R>
__global__ void __launch_bounds__(256, 2) tri_gemv_kernel(const double* __restrict__ W, long long ldw, int N,
                                                          const double* __restrict__ ks, long long ldk, int rows,
                                                          double* __restrict__ v) {
  constexpr int KC = TGV_SMEM_DOUBLES / R;
  constexpr int U = 4;                            // independent 16-byte loads in flight per lane (the stream is
  __shared__ __align__(16) double ks_s[R][KC];    // latency-bound otherwise: 1.5 TB/s with one load per lane)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ngroups = (N + 7) / 8;
  for (int half = 0; half < 2; ++half) {
    const int grp = half == 0 ? (int)blockIdx.x : ngroups - 1 - (int)blockIdx.x;
    if (half == 1 && grp <= (int)blockIdx.x) break;          // the middle group of an odd count is taken once
    const int j = grp * 8 + warp;
    const int jmax = min(grp * 8 + 7, N - 1);                 // longest row of the group
    double acc[R];
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r] = 0.0;
    const double* wj = W + (long long)min(j, N - 1) * ldw;
    for (int k0 = 0; k0 <= jmax; k0 += KC) {
      __syncthreads();
      for (int idx = threadIdx.x; idx < R * KC; idx += 256) {
        const int r = idx / KC, kk = idx - r * KC;
        ks_s[r][kk] = (r < rows && k0 + kk <= jmax) ? ks[(long long)r * ldk + k0 + kk] : 0.0;
      }
      __syncthreads();
      if (j < N) {
        const int kend = min(k0 + KC, j + 1);
        for (int kb = k0 + 2 * lane; kb < kend; kb += 64 * U) {
          double2 w2[U];
#pragma unroll
          for (int u = 0; u < U; ++u) {          // all U loads are issued before the first use
            const int k = kb + 64 * u;
            w2[u] = (k < kend) ? *reinterpret_cast<const double2*>(wj + k) : make_double2(0.0, 0.0);   // (ldw, k even)
            if (k + 1 >= kend) w2[u].y = 0.0;    // beyond the diagonal: not part of row j
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {          // ascending k: the order of the sums does not depend on U
            const int kk = min(kb + 64 * u, kend - 1 - ((kend - 1 - k0) & 1)) - k0;   // even: one 16-byte load per row
#pragma unroll
            for (int r = 0; r < R; ++r) {
              const double2 kv = *reinterpret_cast<const double2*>(&ks_s[r][kk]);
              acc[r] = fma(w2[u].x, kv.x, acc[r]);
              acc[r] = fma(w2[u].y, kv.y, acc[r]);
            }
          }
        }
      }
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
      double a = acc[r];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
      if (lane == 0 && j < N && r < rows) v[(long long)r * N + j] = a;
    }
  }
}

// A <- I (n x n, leading dimension ld)
__global__ void set_identity_kernel(double* __restrict__ A, long long ld, int n) {
  const long long total = (long long)n * ld;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / ld, c = i - r * ld;
    A[i] = (r == c) ? 1.0 : 0.0;
  }
}

// out = in^T for an n x n row-major matrix (both with leading dimension ld); 32 x 32 smem tiles.
__global__ void transpose_kernel(const double* __restrict__ in, double* __restrict__ out, long long ld, int n) {
  __shared__ double tile[32][33];
  const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = by + i, c = bx + threadIdx.x;
    if (r < n && c < n) tile[i][threadIdx.x] = in[(long long)r * ld + c];
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = bx + i, c = by + threadIdx.x;
    if (r < n && c < n) out[(long long)r * ld + c] = tile[threadIdx.x][i];
  }
}

// A[j][i] <- A[i][j] for i > j: fills the strict upper triangle of a symmetric matrix whose lower tiles were computed
// (kernel_fn(x, None): the Gram kernel then skips the tiles above the diagonal).  32 x 32 tiles through shared memory,
// one CTA per lower tile (bx <= by); grid (n/32, n/32), block (32, 8).
__global__ void mirror_lower_kernel(double* __restrict__ A, long long ld, int n) {
  __shared__ double tile[32][33];
  if (blockIdx.x > blockIdx.y) return;
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;     // source tile: rows r0.., columns c0.. (c0 <= r0)
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    if (r < n && c < n) tile[i][threadIdx.x] = A[(long long)r * ld + c];
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = c0 + i, c = r0 + threadIdx.x;             // destination: rows c0.., columns r0..
    if (r < n && c < n && c > r) A[(long long)r * ld + c] = tile[threadIdx.x][i];
  }
}

// zero the strict upper triangle of an N x N row-major matrix (state export)
__global__ void zero_upper_kernel(double* __restrict__ A, long long ld, int N) {
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= N) return;
  for (long long i = blockIdx.y; i < N && i < j; i += gridDim.y) A[i * ld + j] = 0.0;
}

// Packed fitted state <-> the handle's padded device buffers (include/nngp_b200.h, nngp_state_pack / _unpack):
//   [ X (N*D, row-major) | alpha (N) | lower triangle of L by rows (N(N+1)/2) | 'ntk' only: M (N*N) ]
// element g = offset + i of the packed array <-> its home; UNPACK = true stores ext[i] there, false loads it.
struct StatePackView {
  double* X; double* alpha; double* L; double* M;
  long long N, D, ldx, ldl;
};
template <bool UNPACK>
__global__ void state_pack_kernel(StatePackView v, long long offset, long long count, double* __restrict__ ext) {
  const long long nx = v.N * v.D, ntri = v.N * (v.N + 1) / 2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
    long long g = offset + i;
    double* home;
    if (g < nx) {
      const long long r = g / v.D;
      home = v.X + r * v.ldx + (g - r * v.D);
    } else if (g < nx + v.N) {
      home = v.alpha + (g - nx);
    } else if (g < nx + v.N + ntri) {
      const long long t = g - nx - v.N;                       // t = r (r + 1) / 2 + c, 0 <= c <= r
      long long r = (long long)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
      while (r * (r + 1) / 2 > t) --r;                        // the sqrt may be off by one either way
      while ((r + 1) * (r + 2) / 2 <= t) ++r;
      home = v.L + r * v.ldl + (t - r * (r + 1) / 2);
    } else {
      const long long t = g - nx - v.N - ntri;
      const long long r = t / v.N;
      home = v.M + r * v.ldl + (t - r * v.N);
    }
    if (UNPACK) *home = ext[i]; else ext[i] = *home;
  }
}

// finite check: *flag |= 1 for any non-finite in x (rows x cols, ld)
__global__ void finite_check_kernel(const double* __restrict__ x, long long ld, long long rows, int cols,
                                    int* __restrict__ flag) {
  const long long total = rows * cols;
  int bad = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cols;
    const int c = (int)(i - r * cols);
    if (!isfinite(x[r * ld + c])) bad = 1;
  }
  if (bad) atomicOr(flag, 1);
}

// Register-resident DMMA issue-rate microbenchmark: 8 warps per CTA, 16 independent accumulators.
__global__ void __launch_bounds__(256) dmma_peak_kernel(int iters, double* __restrict__ sink) {
  double c[16][2];
#pragma unroll
  for (int i = 0; i < 16; ++i) { c[i][0] = 0.0; c[i][1] = 0.0; }
  double a = 1.0 + 1e-9 * threadIdx.x, b = 1.0 - 1e-9 * threadIdx.x;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 16; ++i)
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                   : "+d"(c[i][0]), "+d"(c[i][1])
                   : "d"(a), "d"(b));
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += c[i][0] + c[i][1];
  if (s == 123.456) sink[0] = s;
}

}  // namespace nngp
