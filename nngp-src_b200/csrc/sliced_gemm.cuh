// sliced_gemm.cuh -- the variance product  V = K_* W^T  (W = L^-1, lower triangular) on the INT8 tensor cores
// (tcgen05.mma kind::i8, accumulators in TMEM), exact enough for FP64 parity.
//
// sm_100a has no FP64 tcgen05 kind; its FP64 tensor path (DMMA) peaks at 37 TFLOP/s while kind::i8 runs ~120x the
// MAC rate.  Every row of both operands is therefore written as
//        a[k] = 2^(e-6) * sum_p d_p[k] 2^(-7p),   d_p[k] integer, |d_p[k]| <= 64   (one exponent e per row)
// (slice_rows_kernel; the digits are exact: each step subtracts the rounded value and rescales by 128).  Every finite
// row is covered, down to a largest magnitude of 2^-1074: the kernel keeps the integer exponent e of each row, scales
// the row up by two power-of-two factors (2^(6-e) alone overflows for e < -1017) and the epilogue applies both rows'
// exponents at once, V = S 2^(ea+eb-12) rounded once (sl_ldexp), so no scale 2^(e-6) has to be a double.  The
// product of two digit planes is an exact int32 GEMM (|sum| <= (g+1) * 2^12 * K < 2^31 for K <= 65536), planes with
// the same p + q = g share the scale 2^(-7g), and keeping the groups g < s gives V to 2^(-7s) of
// |row a|_max |row b|_max K -- s = 7: posterior variance within 1e-8 of the FP64 path at cond 1e7
// (tools/ozaki_study.py, tests/test_gpu_sliced.py).  s (s+1) / 2 integer GEMMs replace one FP64 GEMM (the variance
// path drops the weakest pair: SlicedParams::skip_weak).
//
// Kernel: persistent, one CTA per SM, warp-specialised the Blackwell way:
//   warp 0 (one lane)  TMA producer: 128-byte-swizzled boxes of the digit planes into a 3-stage ring (mbarrier tx);
//                      a stage holds 128 bytes of K for TWO row tiles of K_* (256 rows) and one column tile of W
//   warp 1 (one lane)  MMA issuer: tcgen05.mma M=128 N=256 K=32, the two row tiles into two int32 accumulators that
//                      fill the 512 TMEM columns; tcgen05.commit releases ring stages / publishes the accumulators
//   warps 2-9          epilogue: tcgen05.ld the finished group, fold it into the FP64 running sum (Horner in 2^-7)
//                      held in an L2-resident per-CTA scratch tile; on the last group scale by the two row exponents,
//                      square, reduce along the row -> two partials per (row, column tile); V itself is never stored.
// What bounds it (DESIGN.md 5.10): with one accumulator per stage (48 KiB of operands per 128 x 256 x 128 MMA set of
// 512 clk) the L2 -> SM fabric (~43 B/clk/SM): 2.3 POP/s; sharing each W stage between two accumulators (32 KiB per
// set) moves the limit to the 1 kW power cap -- the kernel runs at ~1.4 GHz with the tensor pipe ~90 % busy, so what
// is left to gain is energy per MAC, i.e. bytes moved:
// Tile order: column tiles in groups of 4 ("supercolumns") from the widest triangular extent down, row-tile pairs
// inside, the 4 column tiles of one pair adjacent -- CTAs 4k..4k+3 stream the same K_* planes (the second to fourth
// read hit L2, sparing HBM) and all CTAs of a wave stream the same W planes.  That only holds while the CTAs stay in
// step, so the producers re-align at a grid-wide counter at every tile (wave_barrier): DRAM reads -55 %, +6.6 %.
#pragma once
#include "ptx.cuh"

namespace nngp {

constexpr int SL_BM = 128;                 // rows per MMA = TMEM lanes
constexpr int SL_RT = 2;                   // row tiles per CTA tile: two M=128 MMAs share every W stage (2 accumulators)
constexpr int SL_BN = 256;                 // rows of W (columns of V) per tile = MMA N
constexpr int SL_BK = 128;                 // bytes (= int8 elements) of K per ring stage: one swizzle row
constexpr int SL_UK = 32;                  // K of one tcgen05.mma kind::i8
constexpr int SL_STAGES = 3;
constexpr int SL_A_BYTES = SL_RT * SL_BM * SL_BK;  // 32 KiB: one TMA box of 256 rows
constexpr int SL_B_BYTES = SL_BN * SL_BK;          // 32 KiB
constexpr int SL_EPI_WARPS = 8;            // two per TMEM lane quarter, each half of the columns
constexpr int SL_THREADS = 64 + 32 * SL_EPI_WARPS;
constexpr int SL_SUPER = 4;                // column tiles per supercolumn
constexpr int SL_MAX_SLICES = 9;
constexpr int SL_SMEM_BYTES = SL_STAGES * (SL_A_BYTES + SL_B_BYTES) + 1024 /*alignment*/ + 256 /*barriers*/;
constexpr int SL_SLICE_THREADS = 256;

struct SlicedParams {
  int s;                   // digit planes per operand
  int rows;                // valid rows of K_*
  int N;                   // columns of V = rows of W
  int K;                   // inner dimension (= N for the triangular W)
  int row_tiles, col_tiles;
  int tri;                 // W lower triangular: column tile j needs K < 256 (j + 1) only
  long long ra, rb;        // rows per plane in the stacked plane arrays of K_* / W
  const int* rexp;         // [rows]  exponent e of the K_* rows (the row is 2^(e-6) times its digits)
  const int* cexp;         // [N]     exponent e of the W rows
  double* scratch;         // gridDim.x x 2 x 256 x 128 running sums
  double* vpart;           // [2 col_tiles][rows] sum over each 128-column half tile of V^2 (may be null)
  double* V;               // [rows][ldv] the product itself (diagnostics / tests)     (may be null)
  long long ldv;
  int skip_weak;           // 1 (variance path): drop the pair (A plane s-1, W plane 0).  A row of W = L^-1 is dominated by
                           // its diagonal entry, so plane 0 of W holds digits 0 / +-1 almost everywhere and this pair
                           // weighs like the first DROPPED group (tools/ozaki_pairskip_study.py): 1 / 28 of the MACs
  int* wave_sync;          // one arrival counter per tile round, zeroed before a cooperative launch: the producers
                           // re-align at every tile (wave_barrier); null: free-running CTAs
};

// ---- digit planes ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double sl_pow2(int n) {   // 2^n, n in [-1022, 1023]
  return __longlong_as_double((long long)(n + 1023) << 52);
}

// x 2^n rounded once, for the folded plane sums x (0, or |x| in [2^-56, 2^32): s <= 9 groups of int32 sums in 2^-7
// steps) and n = ea + eb - 12 anywhere in [-2158, 2036].  Inside the normal exponent range it is the one product
// x 2^n; outside, the first factor keeps the product normal and exact (|x 2^(n+k)| >= 2^-1022) and the second rounds.
// Below n = -1988 the first factor stops at 2^-1022, which only matters where |x 2^n| < 2^-1956: the result is 0
// either way.
__device__ __forceinline__ double sl_ldexp(double x, int n) {
  if (n > 1023) return (x * sl_pow2(1023)) * sl_pow2(min(n - 1023, 1023));
  if (n < -1022) {
    const int k = min(-966 - n, 1022);
    return (x * sl_pow2(max(n + k, -1022))) * sl_pow2(-k);
  }
  return x * sl_pow2(n);
}

// One CTA per (padded) row.  planes[p][row][ldq] int8, zero outside [0, ncols) and for rows >= rows; exp_out[row]
// the row's exponent e (|a| < 2^e; 0 for a zero row).
__global__ void __launch_bounds__(SL_SLICE_THREADS)
slice_rows_kernel(const double* __restrict__ A, long long lda, int rows, int ncols, int tri, int s,
                  int8_t* __restrict__ planes, long long plane_stride, int ldq, int* __restrict__ exp_out) {
  __shared__ double red[SL_SLICE_THREADS / 32];
  __shared__ int e_sh;
  const int row = blockIdx.x;
  const int nc = (row < rows) ? (tri ? min(ncols, row + 1) : ncols) : 0;
  const double* a = A + (long long)row * lda;
  double amax = 0.0;
  for (int c = threadIdx.x; c < nc; c += SL_SLICE_THREADS) amax = fmax(amax, fabs(a[c]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) amax = fmax(amax, __shfl_xor_sync(0xffffffffu, amax, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = amax;
  __syncthreads();
  if (threadIdx.x == 0) {
    double m = red[0];
#pragma unroll
    for (int w = 1; w < SL_SLICE_THREADS / 32; ++w) m = fmax(m, red[w]);
    int e = 0;
    if (m > 0.0) (void)frexp(m, &e);          // m = f 2^e, f in [0.5, 1)  =>  |a| 2^(6-e) < 64
    e_sh = e;
    if (row < rows) exp_out[row] = e;
  }
  __syncthreads();
  // |a| 2^(6-e) < 64 in two exact steps: 2^(6-e) is not a double for e < -1017 (e >= -1073, so the second is <= 2^56)
  const int k = 6 - e_sh;
  const double up = sl_pow2(min(k, 1023)), up2 = sl_pow2(max(k - 1023, 0));
  int8_t* out = planes + (long long)row * ldq;
  for (int c0 = threadIdx.x * 4; c0 < ldq; c0 += SL_SLICE_THREADS * 4) {
    double t[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) t[j] = (c0 + j < nc) ? a[c0 + j] * up * up2 : 0.0;
    for (int p = 0; p < s; ++p) {
      uint32_t w = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int d = __double2int_rn(t[j]);
        t[j] = (t[j] - (double)d) * 128.0;
        w |= (uint32_t)(d & 0xff) << (8 * j);
      }
      *reinterpret_cast<uint32_t*>(out + (long long)p * plane_stride + c0) = w;
    }
  }
}

// ---- tcgen05 wrappers -------------------------------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {   // arrives on `bar` when all MMAs issued so far are done
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T ; int8 x int8 -> int32, M = 128, N = 256, K = 32, both operands K-major
__device__ __forceinline__ void tc_mma_i8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// shared-memory matrix descriptor: K-major, 128-byte swizzle, rows 128 B apart, 8-row groups 1024 B apart
__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) /*LBO (unused)*/ | (64ull << 32) /*SBO = 1024 B*/ |
         (1ull << 46) /*descriptor version: sm_100*/ | (2ull << 61) /*SWIZZLE_128B*/;
}
// instruction descriptor: dense, no saturate, D = s32, A = B = signed int8, K-major, N = 256, M = 128
constexpr uint32_t SL_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(SL_BN >> 3) << 17) |
                              ((uint32_t)(SL_BM >> 4) << 24);

__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&r)[32]) {   // 32 lanes x 32 columns -> 32 regs/thread
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---- tile order -------------------------------------------------------------------------------------------------
struct SlicedTile { int ip, jt, nkb; };   // row-tile pair, column tile, K blocks
__device__ __forceinline__ bool sliced_tile(const SlicedParams& p, long long idx, SlicedTile& t) {
  const int row_pairs = (p.row_tiles + SL_RT - 1) / SL_RT;
  const long long total = (long long)row_pairs * p.col_tiles;
  if (idx >= total) return false;
  const int nsup = (p.col_tiles + SL_SUPER - 1) / SL_SUPER;
  const int wlast = p.col_tiles - (nsup - 1) * SL_SUPER;          // width of the last (widest-K) supercolumn
  const long long first = (long long)row_pairs * wlast;
  int sup, c;
  if (idx < first) {
    sup = nsup - 1;
    t.ip = (int)(idx / wlast); c = (int)(idx % wlast);
  } else {
    const long long r = idx - first, per = (long long)row_pairs * SL_SUPER;
    sup = nsup - 2 - (int)(r / per);
    const long long in = r % per;
    t.ip = (int)(in / SL_SUPER); c = (int)(in % SL_SUPER);
  }
  t.jt = sup * SL_SUPER + c;
  // the whole supercolumn runs the K extent of its last column tile, so that its CTAs stay in lockstep
  const int kext = p.tri ? min(p.K, min((sup + 1) * SL_SUPER, p.col_tiles) * SL_BN) : p.K;
  t.nkb = (kext + SL_BK - 1) / SL_BK;
  return true;
}

// Re-alignment of the CTAs of a wave (cooperative launch: all CTAs resident).  The tile order makes neighbouring CTAs
// stream the same operand planes at the same time; without a common clock they drift apart by more stages than L2
// holds and the shared planes are fetched from HBM again.  Only the TMA producers wait; bounded like every wait here.
__device__ __forceinline__ void wave_barrier(int* counter, int participants) {
  __threadfence();
  atomicAdd(counter, 1);
  for (uint32_t spin = 0;; ++spin) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
    if (v >= participants) break;
    if (spin > (1u << 28)) __trap();
    __nanosleep(64);
  }
}

// ---- the kernel -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SL_THREADS, 1)
sliced_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   const SlicedParams p) {
  extern __shared__ uint8_t sl_smem_raw[];
  const uint32_t raw_addr = smem_u32(sl_smem_raw);
  uint8_t* ring = sl_smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint8_t* ringA = ring;
  uint8_t* ringB = ring + SL_STAGES * SL_A_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(ringB + SL_STAGES * SL_B_BYTES);
  uint64_t* empty_bar = full_bar + SL_STAGES;
  uint64_t* acc_full = empty_bar + SL_STAGES;
  uint64_t* acc_empty = acc_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < SL_STAGES; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 32 * SL_EPI_WARPS);
    fence_mbar_init();
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1) {   // one warp allocates all 512 TMEM columns (1 CTA per SM: no contention) and frees them at the end
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);

  if (warp == 0) {
    if (lane == 0) {   // ===== TMA producer =====
      uint32_t n = 0;
      SlicedTile t;
      const long long total = (long long)((p.row_tiles + SL_RT - 1) / SL_RT) * p.col_tiles;
      int round = 0;
      for (long long idx = blockIdx.x; sliced_tile(p, idx, t); idx += gridDim.x, ++round) {
        if (p.wave_sync != nullptr)
          wave_barrier(p.wave_sync + round, (int)min((long long)gridDim.x, total - (long long)round * gridDim.x));
        for (int g = p.s - 1; g >= 0; --g) {
          const int pa_last = (p.skip_weak && g == p.s - 1 && g > 0) ? g - 1 : g;
          for (int pa = 0; pa <= pa_last; ++pa) {
            const int a_row = (int)(pa * p.ra) + t.ip * (SL_RT * SL_BM);
            const int b_row = (int)((g - pa) * p.rb) + t.jt * SL_BN;
            for (int kb = 0; kb < t.nkb; ++kb, ++n) {
              const uint32_t st = n % SL_STAGES, ph = (n / SL_STAGES) & 1u;
              mbar_wait(&empty_bar[st], ph ^ 1u);
              mbar_arrive_expect_tx(&full_bar[st], SL_A_BYTES + SL_B_BYTES);
              tma_load_2d(ringA + st * SL_A_BYTES, &tmA, kb * SL_BK, a_row, &full_bar[st]);   // both row tiles: 256 rows
              tma_load_2d(ringB + st * SL_B_BYTES, &tmB, kb * SL_BK, b_row, &full_bar[st]);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {   // ===== MMA issuer =====
      uint32_t n = 0, a = 0;
      SlicedTile t;
      for (long long idx = blockIdx.x; sliced_tile(p, idx, t); idx += gridDim.x) {
        const bool two = t.ip * 2 + 1 < p.row_tiles;     // the second row tile exists
        for (int g = p.s - 1; g >= 0; --g, ++a) {
          mbar_wait(acc_empty, (a & 1u) ^ 1u);              // the epilogue has drained both accumulators
          tc_fence_after();
          uint32_t acc = 0;
          const int pa_last = (p.skip_weak && g == p.s - 1 && g > 0) ? g - 1 : g;
          for (int pa = 0; pa <= pa_last; ++pa)
            for (int kb = 0; kb < t.nkb; ++kb, ++n) {
              const uint32_t st = n % SL_STAGES, ph = (n / SL_STAGES) & 1u;
              mbar_wait(&full_bar[st], ph);
              tc_fence_after();
              const uint64_t da0 = tc_smem_desc(smem_u32(ringA + st * SL_A_BYTES));
              const uint64_t da1 = tc_smem_desc(smem_u32(ringA + st * SL_A_BYTES + SL_BM * SL_BK));
              const uint64_t db = tc_smem_desc(smem_u32(ringB + st * SL_B_BYTES));
#pragma unroll
              for (int k = 0; k < SL_BK / SL_UK; ++k) {   // +32 bytes of K inside the swizzle row: +2 in the address field
                tc_mma_i8(tmem_base, da0 + 2u * k, db + 2u * k, SL_IDESC, acc);
                if (two) tc_mma_i8(tmem_base + SL_BN, da1 + 2u * k, db + 2u * k, SL_IDESC, acc);
                acc = 1;
              }
              tc_commit(&empty_bar[st]);                     // stage free once these MMAs have read it
            }
          tc_commit(acc_full);                           // group complete: hand the accumulators to the epilogue
        }
      }
    }
  } else {             // ===== epilogue warps =====
    const int quarter = warp & 3;                        // TMEM lanes this warp may read: 32 quarter .. +31
    const int half = (warp - 2) >> 2;                    // which 128 of the 256 columns
    const int row = quarter * 32 + lane;
    double* sc = p.scratch + (long long)blockIdx.x * (SL_RT * SL_BN * SL_BM) + row;
    uint32_t a = 0;
    SlicedTile t;
    for (long long idx = blockIdx.x; sliced_tile(p, idx, t); idx += gridDim.x) {
      const int ntile = (t.ip * 2 + 1 < p.row_tiles) ? 2 : 1;
      double sum[SL_RT] = {0.0, 0.0};
      for (int g = p.s - 1; g >= 0; --g, ++a) {
        mbar_wait(acc_full, a & 1u);
        __syncwarp();
        tc_fence_after();
        const bool first = (g == p.s - 1);
        for (int h = 0; h < ntile; ++h) {
          const int grow = (t.ip * SL_RT + h) * SL_BM + row;
          const int re = (grow < p.rows) ? p.rexp[grow] - 12 : 0;
          const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + h * SL_BN + half * (SL_BN / 2);
          double* sch = sc + (h * SL_BN + half * (SL_BN / 2)) * SL_BM;
          for (int c0 = 0; c0 < SL_BN / 2; c0 += 32) {
            uint32_t r[32];
            tc_ld32(taddr + c0, r);
            if (g > 0) {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                double* sp = sch + (c0 + j) * SL_BM;
                const double c = (double)(int)r[j];
                *sp = first ? c : fma(*sp, 0.0078125, c);   // S_g = C_g + 2^-7 S_(g+1)
              }
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const int col = t.jt * SL_BN + half * (SL_BN / 2) + c0 + j;
                const double c = (double)(int)r[j];
                const double sv = first ? c : fma(sch[(c0 + j) * SL_BM], 0.0078125, c);
                const double v = (col < p.N && grow < p.rows) ? sl_ldexp(sv, re + __ldg(p.cexp + col)) : 0.0;
                sum[h] = fma(v, v, sum[h]);
                if (p.V && grow < p.rows && col < p.N) p.V[(long long)grow * p.ldv + col] = v;
              }
            }
          }
        }
        tc_fence_before();
        mbar_arrive(acc_empty);
      }
      if (p.vpart)
        for (int h = 0; h < ntile; ++h) {
          const int grow = (t.ip * SL_RT + h) * SL_BM + row;
          if (grow < p.rows) p.vpart[((long long)t.jt * 2 + half) * p.rows + grow] = sum[h];   // two partials per column tile
        }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

}  // namespace nngp
