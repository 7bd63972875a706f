// potrf_panel.cuh -- one outer panel of the blocked Cholesky as ONE persistent kernel (K5 panel).
//
// The panel (W = 256 / 512 columns at offset j0, all rows from j0 down, including the y^T row that rides through the
// factorisation) used to be a chain of 3 launches per 64-wide sub-panel -- left-looking update (DMMA), potf2 of the
// diagonal block (one CTA), block column below it (DMMA product with inv(L_JJ)) -- each a single short wave paying
// ~8 us of launch / pipeline-fill / drain: 12 launches and ~250 us per panel, on the critical path of the whole
// factorisation (at N = 8192 the chain, not the trailing update, set the fit time).
// Here the panel is the work-item scheme of trsm_fused.cuh applied to the factor itself.  Item (r, J) = row tile r
// (128 panel rows) x column block J (64 panel columns):
//     acc = -(A[r, J] - V[r, 0:64J] V[J rows, 0:64J]^T) = -R              TMA + DMMA main loop; BOTH operands are
//                                                                         earlier results of this kernel: thread 0
//                                                                         gates every TMA issue on progress[r] (A
//                                                                         operand) and progress[J / 2] (the rows of
//                                                                         diagonal block J live in row tile J / 2)
//     owner (r == J / 2):  R -> global;  potf2_64_block on the diagonal block (factor + inverse, its shared memory
//                          aliased onto the drained ring);  publish inv_ready[J]
//     everyone:            V[r, J] = R W_J^T  on the tensor pipe (the diagonal step of trsm_fused.cuh), rows strictly
//                          below the diagonal block only;  publish progress[r] = J + 1
// Items above the diagonal are skipped.  Items are claimed in J-major order from a counter, so whatever an item waits
// for -- its own row tile's earlier blocks, the owner tile's earlier blocks, the owner's inverse -- belongs to an item
// with a SMALLER ticket, i.e. to a CTA that is already running: no deadlock and no co-residency assumption, and the
// CTAs of one row tile pipeline along J.  Waits are bounded and trap.  One launch per panel instead of 3 per sub-panel.
#pragma once
#include "dense_kernels.cuh"
#include "gemm_nt.cuh"
#include "trsm_fused.cuh"

namespace nngp {

struct PanelParams {
  double* A;            // the whole matrix (row-major, ld): element (0, 0)
  long long ld;
  int j0;               // panel origin (row and column)
  int rows;             // panel rows: R - j0 (the matrix rows from j0 down plus the extra rows riding along)
  int ncols;            // panel columns: min(W, N - j0)
  int row_tiles, col_blocks;
  int* info;            // potrf info (first failing pivot + 1)
  double* Winv;         // inverses of ALL diagonal blocks (block at global column c at rows [c, c + 64) of a 64-wide matrix)
  int* counter;         // zeroed before launch
  int* progress;        // [row_tiles], zeroed before launch
  int* inv_ready;       // [col_blocks], zeroed before launch
  uint32_t zero;        // always 0 (see mma_mainloop's release dependence)
  unsigned long long* trace;   // NNGP_PANEL_TRACE=1 (diagnostics): [col_blocks][10] globaltimer stamps of the owner items
};

static_assert(sizeof(Potf2Smem) <= TF_RING_BYTES, "the block factorisation's shared memory is aliased onto the ring");

__global__ void __launch_bounds__(GEMM_THREADS, 2)
potrf_panel_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmL,
                   const __grid_constant__ CUtensorMap tmW, const PanelParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t pad = (1024u - (raw_addr & 1023u)) & 1023u;
  uint8_t* ring = smem_raw + pad;
  uint8_t* ringA = ring;
  uint8_t* ringB = ring + TF_STAGES * GEMM_A_STAGE_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(ring + TF_RING_BYTES);
  uint64_t* empty_bar = full_bar + TF_STAGES;
  int* s_item = reinterpret_cast<int*>(empty_bar + TF_STAGES);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int tid = threadIdx.x;
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < TF_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], GEMM_CONSUMER_WARPS);
    }
    fence_mbar_init();
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmL);
    tma_prefetch_desc(&tmW);
  }

  const int total = p.row_tiles * p.col_blocks;
  int stage = 0;
  uint32_t phase = 0;
  const int wm = warp >> 1, wn = warp & 1;
  const int g = lane >> 2, t = lane & 3;
  double* const P0 = p.A + (long long)p.j0 * p.ld + p.j0;   // panel element (0, 0)

  for (;;) {
    if (tid == 0) s_item[0] = atomicAdd(p.counter, 1);
    __syncthreads();  // publishes the item; also: nobody still uses the ring / the scratch of the last item
    const int item = s_item[0];
    if (item >= total) break;
    const int J = item / p.row_tiles;
    const int r = item - J * p.row_tiles;
    const int col0 = J * NB;                      // panel-relative
    const int nb = min(NB, p.ncols - col0);
    const int row0 = r * GEMM_BM;
    // rows above diagonal block J hold upper-triangle entries: nothing to do (block-uniform; publishes nothing)
    if (row0 + GEMM_BM <= col0) { __syncthreads(); continue; }
    const int rJ = J / 2;                         // the row tile that holds the rows of diagonal block J
    const bool owner = (r == rJ);
#ifdef NNGP_PANEL_TRACE   // diagnostics build (build.sh -DNNGP_PANEL_TRACE): phase time stamps of the owner items
    unsigned long long* tr = (p.trace != nullptr && owner) ? p.trace + J * 10 : nullptr;
    auto stamp = [&](int k) { if (tr != nullptr && tid == 0) tr[k] = global_timer_ns(); };
#else
    unsigned long long* const tr = nullptr;
    auto stamp = [](int) {};
#endif
    stamp(0);
    const int ktiles = J * (NB / GEMM_BK);

    TileSrc src;
    src.tmA = &tmA; src.tmB = &tmL;
    src.a_col0 = p.j0; src.a_row = p.j0 + row0; src.b_col0 = p.j0; src.b_row = p.j0 + col0;
    int known_a = 0, known_b = 0;   // progress[r] / progress[rJ] as last seen by thread 0
    auto wait_progress = [&](const int* flag, int& known, int need) {
      if (known < need) {
        for (unsigned spin = 0; (known = ld_acquire_gpu(flag)) < need; ++spin) {
          __nanosleep(64);
          if (spin > (1u << 27)) __trap();
        }
        fence_proxy_async_all();   // written through the generic proxy by other CTAs -> read by TMA
      }
    };
    auto gate = [&](int kt) {
      const int need = kt / (NB / GEMM_BK) + 1;
      wait_progress(p.progress + r, known_a, need);
      if (owner) known_b = known_a; else wait_progress(p.progress + rJ, known_b, need);
    };
    if (tid == 0) {
      const int n0 = ktiles < TF_STAGES ? ktiles : TF_STAGES;
      int st = stage;
      for (int i = 0; i < n0; ++i) {
        gate(i);
        ring_issue<TF_STAGES>(src, ringA, ringB, full_bar, st, i);
        if (++st == TF_STAGES) st = 0;
      }
    }

    // acc = -(tile of the panel): the values the trailing update of the previous panel left there
    double acc[4][4][2];
    auto load_tile_neg = [&]() {
#pragma unroll
      for (int mi = 0; mi < 4; ++mi) {
        const int lr = wm * 32 + mi * 8 + g;
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) {
          const int lc = wn * 32 + ni * 8 + 2 * t;
          double v0 = 0.0, v1 = 0.0;
          if (row0 + lr < p.rows) {
            const double* src_c = P0 + (long long)(row0 + lr) * p.ld + col0 + lc;
            if (lc + 1 < nb) {
              const double2 v = __ldcg(reinterpret_cast<const double2*>(src_c));
              v0 = v.x; v1 = v.y;
            } else if (lc < nb) {
              v0 = __ldcg(src_c);
            }
          }
          acc[mi][ni][0] = -v0;
          acc[mi][ni][1] = -v1;
        }
      }
    };
    load_tile_neg();
    mma_mainloop<TF_STAGES>(acc, src, ringA, ringB, full_bar, empty_bar, stage, phase, ktiles, wm, wn, lane, p.zero, gate);

    __syncthreads();  // every warp has left the ring
    stamp(1);
    if (owner) {
      // R (the updated tile) -> global, factor the diagonal block there, publish its inverse, take R back
      if (ktiles > 0) {
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) {
          const int lr = wm * 32 + mi * 8 + g;
          if (row0 + lr >= p.rows) continue;
#pragma unroll
          for (int ni = 0; ni < 4; ++ni) {
            const int lc = wn * 32 + ni * 8 + 2 * t;
            double* dst = P0 + (long long)(row0 + lr) * p.ld + col0 + lc;
            if (lc + 1 < nb) *reinterpret_cast<double2*>(dst) = make_double2(-acc[mi][ni][0], -acc[mi][ni][1]);
            else if (lc < nb) dst[0] = -acc[mi][ni][0];
          }
        }
        __threadfence();
        __syncthreads();
      }
      Potf2Smem& psm = *reinterpret_cast<Potf2Smem*>(ring);
      stamp(2);
      potf2_64_block(P0 + (long long)col0 * p.ld + col0, p.ld, nb, p.j0 + col0, p.info,
                     p.Winv + (long long)(p.j0 + col0) * NB, psm,
                     tr != nullptr ? p.trace + p.col_blocks * 10 + J * 8 : nullptr);
#ifdef NNGP_PANEL_TRACE
      if (tr != nullptr && tid == 0) tr[3] = p.trace[p.col_blocks * 10 + J * 8];   // factor done
#endif
      stamp(4);
      __threadfence();            // L_JJ and W_J (generic stores) ...
      fence_proxy_async_all();    // ... before the TMA loads of the CTAs that acquire the flag
      __syncthreads();            // (also: the ring is free again)
      if (tid == 0) st_release_gpu(p.inv_ready + J, 1);
      load_tile_neg();            // rows below the diagonal block are still R; the block's own rows are not stored below
      stamp(5);
    }

    // ---- diagonal step: V[r, J] = R * W_J^T on the tensor pipe (as in trsm_fused.cuh) ---------------------
    if (tid == 0) {
      for (unsigned spin = 0; ld_acquire_gpu(p.inv_ready + J) == 0; ++spin) {
        __nanosleep(64);
        if (spin > (1u << 27)) __trap();
      }
      fence_proxy_async_all();
      int st = stage;
#pragma unroll
      for (int kt = 0; kt < TF_STAGES; ++kt) {
        mbar_arrive_expect_tx(&full_bar[st], GEMM_B_STAGE_BYTES);
        tma_load_2d(ringB + st * GEMM_B_STAGE_BYTES, &tmW, kt * GEMM_BK, p.j0 + col0, &full_bar[st]);
        if (++st == TF_STAGES) st = 0;
      }
    }
#pragma unroll
    for (int mi = 0; mi < 4; ++mi) {
      const int lr = wm * 32 + mi * 8 + g;
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) {
        int slot = stage + wn * 2 + (ni >> 1);
        if (slot >= TF_STAGES) slot -= TF_STAGES;
        const int chunk = ((ni & 1) * 4 + t) ^ g;   // lr & 7 == g
        double2* dst = reinterpret_cast<double2*>(ringA + slot * GEMM_A_STAGE_BYTES + lr * 128 + chunk * 16);
        *dst = make_double2(-acc[mi][ni][0], -acc[mi][ni][1]);
        acc[mi][ni][0] = 0.0;
        acc[mi][ni][1] = 0.0;
      }
    }
    __syncthreads();  // R is visible to every warp
    stamp(6);
    mma_mainloop<TF_STAGES>(acc, src, ringA, ringB, full_bar, empty_bar, stage, phase, TF_STAGES, wm, wn, lane, p.zero);
    stamp(7);
    // store the rows strictly below the diagonal block (its own rows hold potf2's L_JJ; rows above it are upper triangle)
#pragma unroll
    for (int mi = 0; mi < 4; ++mi) {
      const int lr = wm * 32 + mi * 8 + g;
      const int prow = row0 + lr;
      if (prow < col0 + nb || prow >= p.rows) continue;   // (a short last block has nb < 64 rows: the y^T row follows it)
#pragma unroll
      for (int ni = 0; ni < 4; ++ni) {
        const int lc = wn * 32 + ni * 8 + 2 * t;
        double* dst = P0 + (long long)prow * p.ld + col0 + lc;
        if (lc + 1 < nb) *reinterpret_cast<double2*>(dst) = make_double2(acc[mi][ni][0], acc[mi][ni][1]);
        else if (lc < nb) dst[0] = acc[mi][ni][0];
      }
    }
    fence_proxy_async_all();
    __threadfence();
    __syncthreads();
    if (tid == 0) st_release_gpu(p.progress + r, J + 1);
    stamp(8);
  }
}

}  // namespace nngp
