/*
 * nngp_b200.h -- C ABI of the B200-native NNGP estimator core.
 *
 * This is the drop-in boundary for ONE hot path of Kangfei/NNGP-src: NNGP kernel
 * construction + exact GP posterior inference.  The reference has no FFI of its own
 * (it is pure Python delegating to neural-tangents on JAX/XLA:CPU + LAPACK), so each
 * entry point below cites the reference *call site* (file:line under the reference
 * tree) whose arithmetic it replaces; the un-vendored neural-tangents 0.6.1 callee
 * is named in brackets.
 *
 * Conventions
 *   - plain C, no torch / C++ types in any signature;
 *   - every matrix is dense row-major FP64; a pointer may be HOST (pageable or
 *     pinned) or DEVICE memory -- detected with cudaPointerGetAttributes; outputs
 *     are written into the caller's buffer in the memory space it lives in;
 *   - every call returns 0 on success or a negative nngp_status; the message is
 *     available from nngp_last_error(); nothing aborts, throws or prints;
 *   - a handle is not re-entrant; distinct handles are independent; every call is
 *     complete (stream-synchronised) when it returns.  A handle owns ONE GPU, or -- with
 *     cfg.n_gpus > 1 -- a fit GPU plus replicas of the fitted state on the other GPUs: the
 *     fit runs on device_ids[0], its state is copied once per fit over NVLink (packed lower
 *     triangle, peer-to-peer, no host staging) and nngp_predict splits the test rows
 *     [g*T/G, (g+1)*T/G) over the G GPUs, one host worker thread per extra GPU (the
 *     reference's callers are single-process: estimator.py:42-62, train.py:178);
 *   - there is NO CPU fallback: without a usable sm_100 device nngp_create fails.
 */
#ifndef NNGP_B200_H
#define NNGP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NNGP_B200_ABI_VERSION 7
#define NNGP_MAX_GPUS 8
#define NNGP_MAX_LAYERS 16

#if defined(__GNUC__)
#define NNGP_API __attribute__((visibility("default")))
#else
#define NNGP_API
#endif

typedef enum nngp_status {
  NNGP_OK = 0,
  NNGP_EINVAL = -1,  /* bad argument / shape / non-finite input                      */
  NNGP_ENOTPD = -2,  /* K + lambda*I not positive definite (pivot in last_error)     */
  NNGP_ECUDA = -3,   /* CUDA runtime / driver error                                  */
  NNGP_ENOMEM = -4,  /* device allocation failed                                     */
  NNGP_ESTATE = -5,  /* call needs a fitted model (nngp_fit / nngp_set_state first)  */
  NNGP_ENODEV = -6   /* no usable sm_100 device                                      */
} nngp_status;

/*
 * Kernel + regulariser hyper-parameters.
 * Replaces the closure state built by
 *   stax.serial(stax.Dense(512), stax.Relu(), stax.Dense(1))        train.py:161-164,
 *                                        estimator.py:27-30, active/active_train.py:40-43
 *   nt.predict.gradient_descent_mse_ensemble(..., diag_reg=1e-3)    train.py:171-172,
 *                                        estimator.py:34-35, active/ActiveLearner.py:27-28
 * depth = number of Dense layers (reference: 2) = depth-1 ReLU arc-cosine steps.
 * kernel_type selects what predict_fn's `get=` selects in the reference (train.py:157-158,254):
 *   'nngp': K, posterior of the NNGP;   'ntk': Theta, t=infinity NTK ensemble posterior
 *   mean = Theta_* A^-1 y,  var_i = K_ii + w_i^T K_dd w_i - 2 w_i^T k_i,  w_i = A^-1 theta_i,
 *   A = Theta_dd + diag_reg*trace(Theta_dd)/N I   [nt 0.6.1 predict.gp_inference, get='ntk'].
 */
typedef struct nngp_config {
  int32_t depth;              /* >= 1                                                 */
  double sigma_w;             /* stax.Dense W_std (reference default 1.0)             */
  double sigma_b;             /* stax.Dense b_std (reference default None == 0.0)     */
  double diag_reg;            /* reference: 1e-3                                      */
  int32_t diag_reg_absolute;  /* 0: lambda = diag_reg * trace(K)/N  (nt default)      */
  int32_t device;             /* CUDA ordinal; -1 = current device                    */
  int64_t max_block_bytes;    /* cap of the test-row block buffer; 0 = default 16 GiB */
  int32_t stats_level;        /* device times nngp_stats_t fills (its counters and replicate_ms, a host clock, are kept
                                 at every level):
                                 0: sliced_ms and inverse_ms only;
                                 1: also fit_*_ms, pred_*_ms, h2d_ms and d2h_ms (one event pair per stage);
                                 2: also gemm_ms and gram_ms (one event pair per DMMA launch)                        */
  int32_t kernel_type;        /* 0 = 'nngp' (reference default), 1 = 'ntk' (train.py:254)  */
  int32_t n_gpus;             /* 0 / 1: one GPU (`device`); G > 1: prediction rows are split over G GPUs   */
  int32_t device_ids[NNGP_MAX_GPUS]; /* CUDA ordinals when n_gpus > 1 ([0] = fit GPU); all -1: 0..G-1   */
  int32_t latency_mode;       /* 1: the fit also builds the explicit inverse factor L^-1 (N^3/3 more flop) and small
                                 prediction batches (the serving case, estimator.py:42-62: a few query lines per
                                 call) run as a dependency-free triangular GEMM on it instead of the substitution
                                 chain.  Same posterior to rounding (not bitwise the substitution's); default 0.     */
  int32_t per_layer;          /* 1: Dense layer l (0-based, l < depth <= NNGP_MAX_LAYERS) uses sigma_w_layers[l] /
                                 sigma_b_layers[l] instead of the uniform sigma_w / sigma_b -- stax.serial chains whose
                                 Dense layers differ in W_std / b_std [nt allows it; the reference never does]          */
  double sigma_w_layers[NNGP_MAX_LAYERS];
  double sigma_b_layers[NNGP_MAX_LAYERS];
  int32_t variance_slices;    /* 0: off.  s = 5..9 ('nngp' only; implies the explicit inverse factor of latency_mode):
                                 the variance product K_* L^-T of LARGE prediction batches runs on the INT8 tensor cores
                                 (tcgen05.mma kind::i8, accumulators in TMEM): both operands are split row-wise into s
                                 signed 7-bit digit planes, the s(s+1)/2 - 1 exact int32 plane products with p + q < s (all but
                                 the weakest, plane s-1 of K_* times plane 0 of L^-1) are recombined in FP64.  s = 7 keeps the posterior variance within ~1e-8 relative of the
                                 FP64 path at cond(K + lambda I) = 1e7 (s = 8: 1e-10); the mean is untouched.  N <= 2^19 / s.
                                 Every row scale is carried as an integer exponent, so rows of any finite magnitude,
                                 down to the smallest subnormal, are split exactly; an entry of the product that falls
                                 below 2^-1022 is rounded once into the subnormal range. */
  int32_t reserved0;
} nngp_config;

/* Per-stage device timings (CUDA events; cfg.stats_level says which are filled) and work counters,
 * accumulated since the last nngp_stats_reset().  Replaces the wall-clock prints at
 * train.py:170-176,191-195 and estimator.py:44,52-54. */
typedef struct nngp_stats_t {
  double fit_gram_ms, fit_chol_ms, fit_solve_ms, fit_total_ms;
  double pred_gram_ms;
  double pred_mean_ms;     /* always 0: the mean is reduced inside the Gram stage (pred_gram_ms)                  */
  double pred_trsm_ms, pred_var_ms, pred_total_ms;
  double h2d_ms, d2h_ms;
  double gemm_ms;          /* stats_level 2: time inside the DMMA GEMM-update kernels  */
  double gemm_flops;       /* algorithmic flops of those launches (2*M*N*K)            */
  int64_t gemm_launches;
  double gram_ms;          /* stats_level 2: time inside the Gram+arc-cosine kernels   */
  double gram_flops;       /* 2*M*N*D of those launches                                */
  double gram_evals;       /* arc-cosine evaluations ((depth-1) per Gram entry)        */
  int64_t gram_launches;
  int64_t kernel_launches; /* every kernel this library launched                       */
  int64_t h2d_bytes, d2h_bytes;
  int64_t queries;         /* test rows predicted                                      */
  double replicate_ms;     /* n_gpus > 1: wall time of the last peer-to-peer replication of the fitted state */
  int64_t replicate_bytes; /* bytes each replica received in it                        */
  double inverse_ms;       /* latency_mode: device time of building L^-1 in the last fit */
  double sliced_ms;        /* variance_slices: device time of digit-plane splitting + the int8 plane products   */
  double sliced_macs;      /* int8 multiply-accumulates issued to the tensor cores in them                       */
  int64_t device_allocs;   /* device buffer allocations (cudaMalloc); 0 between rounds after nngp_reserve        */
} nngp_stats_t;

typedef struct nngp_handle nngp_handle;

/* Fill cfg with the reference's defaults (depth 2, W_std 1, no bias, diag_reg 1e-3
 * relative) -- train.py:161-172. */
NNGP_API void nngp_default_config(nngp_config* cfg);

/* Create a handle on one GPU.  [replaces: closure construction, train.py:161-172]
 * Same as nngp_create_with_activation(cfg, NULL, out): every hidden step is a ReLU. */
NNGP_API int nngp_create(const nngp_config* cfg, nngp_handle** out);

/*
 * The activation of the hidden steps: one activation for every step of the chain Dense (act Dense)* (per_layer
 * sigmas still apply).  For the step that maps the previous Dense layer's pre-activation covariance (q1, q2, k) to the
 * next one, with s = sqrt(max(q1 q2 - k^2, 0)) and theta = atan2(s, k):
 *   k'   = sigma_w^2 E[phi(u) phi(v)] + sigma_b^2,   q' = sigma_w^2 E[phi(u)^2] + sigma_b^2,
 *   ntk' = k' + sigma_w^2 ntk E[phi'(u) phi'(v)]     (kernel_type 'ntk')
 * NNGP_ACT_RELU   max(x, 0)                       the default; a, b, c are ignored
 * NNGP_ACT_ABRELU a min(x, 0) + b max(x, 0)       [nt 0.6.1 stax.ABRelu; LeakyRelu(alpha) = (alpha, 1), Abs = (-1, 1)]
 *                 E[phi phi] = (a-b)^2/(2 pi) s + kdot k,  kdot = (a^2+b^2)/2 - (a-b)^2 theta/(2 pi)
 * NNGP_ACT_ERF    a erf(b x) + c                  [nt 0.6.1 stax.Erf]; b != 0; with Q = b^2 q, K = b^2 k,
 *                 P = (1 + 2 Q1)(1 + 2 Q2) - 4 K^2:  E[phi phi] = a^2 (2/pi) atan2(2K, sqrt P) + c^2,
 *                 kdot = a^2 b^2 (4/pi) / sqrt P
 * a, b and c must be finite; kind must be one of the three.  Erf also needs b^2, a^2 b^2 and c^2 to be finite normal
 * (or zero) doubles, and every hidden layer's diagonal bound sigma_w^2 (a^2 + c^2) + sigma_b^2 (E[phi^2] <= a^2 + c^2)
 * to satisfy the Erf input range below.  Anything else is NNGP_EINVAL with a message.
 * Erf input range: on top of nngp_kernel's, every row's layer-0 diagonal q must have b^2 q < 2^508 (NNGP_EINVAL
 * otherwise); within it the Erf kernel needs no range guard (DESIGN.md 5.12).
 * ABRelu input range: every step forms q q', so the diagonal entering every step, sigma_w^2 (a^2+b^2)/2 q +
 * sigma_b^2 after the previous one, must stay below 2^512 like the layer-0 one; that bound is carried back to a
 * limit on the layer-0 q (NNGP_EINVAL above it, and at creation if sigma_b^2 alone reaches it).
 * act == NULL or kind == NNGP_ACT_RELU is exactly nngp_create.  A handle with n_gpus > 1 uses the activation on
 * every GPU.
 */
#define NNGP_ACT_RELU 0
#define NNGP_ACT_ABRELU 1
#define NNGP_ACT_ERF 2
typedef struct nngp_activation {
  int32_t kind;      /* NNGP_ACT_*                          */
  int32_t reserved;  /* 0                                   */
  double a, b, c;    /* ABRelu (a, b); Erf (a, b, c)        */
} nngp_activation;
NNGP_API int nngp_create_with_activation(const nngp_config* cfg, const nngp_activation* act, nngp_handle** out);
NNGP_API void nngp_destroy(nngp_handle* h);

/* Message of the last failing call on this handle (or of a failed nngp_create when
 * h == NULL).  Never NULL. */
NNGP_API const char* nngp_last_error(const nngp_handle* h);

/* The CUDA stream (cudaStream_t) every kernel of this handle is launched on, so a
 * host can bracket calls with its own events. */
NNGP_API void* nngp_get_stream(nngp_handle* h);

/*
 * kernel_fn(x1, x2-or-None, 'nngp')                         train.py:216 (disabled block),
 * live via predict_fn: train.py:157-158, estimator.py:66-67.
 * [nt: stax._inputs_to_kernel -> Dense -> Relu(ABRelu 0,1; arctan2 form) -> Dense]
 * x1: M x D, x2: N2 x D (NULL => x2 = x1, N2 ignored), k_out: M x N2.
 *
 * Accepted input range (nngp_kernel, nngp_fit, nngp_append_fit, nngp_predict): every element finite, and every
 * row's layer-0 diagonal q = sigma_w^2 |x|^2 / D + sigma_b^2 below 2^512, so that q q' is a finite double (with an
 * Erf(a, b, c) activation also b^2 q below 2^508, see nngp_activation); anything else is NNGP_EINVAL.  nngp_set_state and nngp_state_import_end hold the imported X to the same range
 * (NNGP_EINVAL, the handle is left without a fitted model).  There is no lower bound: rows down to the subnormal range (and zero rows) are
 * accepted, but an entry whose q, q q' or k^2 is subnormal carries fewer significant bits.
 */
NNGP_API int nngp_kernel(nngp_handle* h, const double* x1, int64_t M, const double* x2_or_null, int64_t N2,
                int64_t D, double* k_out);

/*
 * Fit = what the first predict_fn call does lazily in the reference:
 *   K_dd = kernel_fn(X,X); lambda = diag_reg*trace(K_dd)/N; C = chol(K_dd + lambda I);
 *   alpha = C^-T C^-1 y                      train.py:171-172,178; estimator.py:34-40;
 *   active/ActiveLearner.py:27-28  [nt: predict.gp_inference/_get_cho_solve/
 *   _add_diagonal_regularizer -> scipy cho_factor/cho_solve]
 * x_train: N x D, y_train: N (used raw, never centred).
 * alpha must come out finite: when (K + lambda I)^-1 y overflows the double range (a lambda near the bottom of the
 * normal range against O(1) labels) the fit is NNGP_EINVAL with a message instead of a model whose means are inf or
 * NaN; nngp_append_fit checks its alpha the same way.
 */
NNGP_API int nngp_fit(nngp_handle* h, const double* x_train, const double* y_train, int64_t N, int64_t D);

/*
 * predict_fn(x_test=X, get='nngp', compute_cov=True) followed by diag()
 *                                           train.py:157-158,180; estimator.py:55,66-67;
 *   active/ActiveLearner.py:44-46  [nt: gp_inference.predict_fn]
 * mean_out[T] = K(X*,X) alpha;  var_out[T] = K(x*,x*) - || C^-1 K(X,x*) ||^2, i.e. the
 * diagonal of the posterior covariance the reference materialises as T x T.  var_out
 * may be NULL (compute_cov=False).  Negative variances are returned as they come.
 */
NNGP_API int nngp_predict(nngp_handle* h, const double* x_test, int64_t T, double* mean_out, double* var_out);

/*
 * predict_fn(x_test=X, get=..., compute_cov=True) without the diag(): the full posterior covariance of a test batch
 *   'nngp': cov = K(X*,X*) - V V^T,                          V = K_* L^-T
 *   'ntk' : cov = K(X*,X*) + V M V^T - (V U^T + U V^T),       V = Theta_* L^-T, U = K_* L^-T, M as in SURVEY A.5
 * mean_out[T] as nngp_predict; cov_out[T*T] row-major, host or device memory.  cov_out is bitwise symmetric, its
 * diagonal is bitwise the var_out of nngp_predict for the same batch on the same handle (whichever variance path
 * that takes: substitution, latency mode or variance_slices; the off-diagonal products are always FP64), and the
 * mean is bitwise nngp_predict's.  The test x test Gram and every product run on the lower triangle on the DMMA
 * GEMM core, then the triangle is mirrored.  The batch is ONE prediction block: V (for 'ntk' also U and V M) of
 * all T rows must fit cfg.max_block_bytes (T * round_up(N, 16) * 8 bytes each) -- a larger T is NNGP_EINVAL and the
 * message names the largest T allowed.  With cfg.n_gpus > 1 the covariance is computed on the fit GPU.
 * Errors otherwise as nngp_predict; an imported 'ntk' state without M is NNGP_ESTATE.
 */
NNGP_API int nngp_predict_cov(nngp_handle* h, const double* x_test, int64_t T, double* mean_out, double* cov_out);

/* Fitted-state export/import: used to broadcast a fit to the other ranks of a
 * row-sharded prediction job (one process per GPU) and to save/load a model.
 * nngp_get_dims reports N, D and the lambda actually used.
 * nngp_get_state copies X (N x D), L (N x N row-major lower factor, upper triangle
 * zero) and alpha (N); any pointer may be NULL to skip it.
 * nngp_set_state installs a state produced by nngp_get_state on a handle with the
 * same config and the same activation (nngp_create_with_activation): the state does not record either. */
NNGP_API int nngp_get_dims(nngp_handle* h, int64_t* N, int64_t* D, double* lambda_out);
NNGP_API int nngp_get_state(nngp_handle* h, double* x_out, double* l_out, double* alpha_out);
NNGP_API int nngp_set_state(nngp_handle* h, const double* x, const double* l, const double* alpha, int64_t N,
                   int64_t D, double lambda);
/* 'ntk' mode only: the state additionally holds M = L^-1 K_dd L^-T (N x N row-major), which the posterior variance
 * needs (SURVEY A.5).  Export after nngp_fit; import after nngp_set_state.  Until M is set, an imported 'ntk' state
 * predicts the mean only (variance requests return NNGP_ESTATE). */
NNGP_API int nngp_get_state_ntk_m(nngp_handle* h, double* m_out);
NNGP_API int nngp_set_state_ntk_m(nngp_handle* h, const double* m);

/* Gaussian log marginal likelihood of the fitted model (model selection over depth / W_std / b_std /
 * diag_reg -- the reference's abandoned hyper-parameter path, train.py:86-103, active/active_train.py:44-49):
 *   -1/2 y^T (K + lambda I)^-1 y - sum_i log L_ii - N/2 log(2 pi).
 * Both sums are by-products of nngp_fit (z = L^-1 y rides through the factorisation). */
NNGP_API int nngp_log_marginal_likelihood(nngp_handle* h, double* lml_out);

/* ---- active-learning step on the device (SURVEY 8f-3) ------------------------------------------
 * nngp_active_select == ActiveLearner.active_test (active/ActiveLearner.py:43-55): posterior mean / variance of
 * the pool, score_i = sqrt(var_i) / max_j(mean_j), then
 *   NNGP_SELECT_TOPK   : np.argsort(score)[-k:]            (biased_sample = False, :54) -- indices in ascending
 *                        score order, ties broken by row index (larger index later), NaN scores sort last;
 *   NNGP_SELECT_SAMPLE : random.choice(T, k, replace=False, p = score / sum(score))  (biased_sample = True, :49-53)
 *                        as Gumbel-top-k with a splitmix64 stream of (seed, row) -- the reference draws from JAX's
 *                        threefry stream with PRNGKey(10), which is not reproducible without jax (unpinned);
 *                        indices come out in draw order.  Needs finite scores >= 0 (else NNGP_EINVAL).
 * k = min(budget, T) is returned in *n_selected_out; idx_out receives k int64 row numbers (host or device
 * memory); score_out (T doubles, optional) receives the normalised scores.  Selection runs on the device (exact
 * radix select); only the k winners cross PCIe.
 * nngp_append_fit == ActiveLearner.merge_data + train (:57-65, :23-31): appends M labelled rows to the training
 * set already held by the handle and refits from scratch -- bitwise the nngp_fit of the stacked arrays (the
 * reference's relative diag_reg makes every refit a new lambda, so the factor cannot be extended exactly).  With
 * cfg.diag_reg_absolute (fixed lambda, NNGP mode, even N) the factor IS extended instead: L21 = K21 L11^-T, Cholesky
 * of the M x M Schur complement, N^2 M + M^3/3 flop instead of (N+M)^3/3 -- the same model up to rounding
 * (NNGP_APPEND_INCREMENTAL=0 forces the refit).  Needs a model fitted by nngp_fit on this handle. */
#define NNGP_SELECT_TOPK 0
#define NNGP_SELECT_SAMPLE 1
NNGP_API int nngp_active_select(nngp_handle* h, const double* x_pool, int64_t T, int64_t budget, int32_t mode,
                                uint64_t seed, int64_t* idx_out, int64_t* n_selected_out, double* score_out);
NNGP_API int nngp_append_fit(nngp_handle* h, const double* x_new, const double* y_new, int64_t M);
/* Optional: size the handle's device buffers once for the largest training set / pool the loop will reach
 * (n_train_max rows of `dim` features, n_test_max rows per predict / select call; 0 = fit-side only), so that
 * no multi-GB cudaFree / cudaMalloc happens between rounds.  Call before nngp_fit: it drops a fitted model. */
NNGP_API int nngp_reserve(nngp_handle* h, int64_t n_train_max, int64_t dim, int64_t n_test_max);

NNGP_API int nngp_stats(nngp_handle* h, nngp_stats_t* out);
NNGP_API int nngp_stats_reset(nngp_handle* h);

/* Diagnostics used by bench.py / the tests (not part of the reference surface):
 *   dmma_peak: register-resident mma.sync.m8n8k4.f64 issue-rate microbenchmark -> TFLOP/s
 *   gemm_probe: C(MxN) -= A(MxK) B(NxK)^T through the production DMMA kernel on device
 *               scratch, `iters` launches -> average ms per launch
 *   potrf: in-place lower Cholesky of a caller-supplied N x N row-major matrix. */
NNGP_API int nngp_diag_dmma_peak(nngp_handle* h, double* tflops_out);
NNGP_API int nngp_diag_gemm_probe(nngp_handle* h, int64_t M, int64_t N, int64_t K, int32_t iters, double* ms_out);
NNGP_API int nngp_diag_potrf(nngp_handle* h, double* a, int64_t N);

NNGP_API int nngp_abi_version(void);
/* Hash of the sources this binary was compiled from (csrc, include, build.sh -- nngp_b200/_build.py); the Python
 * loader and __graft_entry__.build() rebuild when it does not match the tree they run in. */
NNGP_API const char* nngp_build_id(void);
/* Number of GPUs the handle predicts on (1 unless cfg.n_gpus > 1). */
NNGP_API int nngp_num_gpus(const nngp_handle* h);

/* Diagnostic / test entry of the digit-plane product behind cfg.variance_slices: V = A B^T for A [M, K] and B [N, K]
 * (dense row-major, host or device), computed with `slices` int8 planes per operand on the tcgen05 kind::i8 path;
 * `lower` != 0 treats B as lower triangular (entries with k > row ignored, N == K); `lower` == 2 also drops the plane
 * pair (slices-1, 0), exactly as the variance path does for B = L^-1 (whose rows are dominated by their diagonal entry).  v_out [M, N] receives the product,
 * rowsq_out [M] (optional) the row sums of V^2 in the order the variance uses.  Independent of any fitted model.
 * Any finite rows are accepted: each row of A and B is scaled by its own power of two (down to rows whose largest
 * magnitude is the smallest subnormal), and each entry is the folded plane sum times 2^(ea + eb - 12), rounded once.
 * [no reference counterpart: the reference's only matrix product is XLA's dot, train.py:157-158]              */
NNGP_API int nngp_sliced_product(nngp_handle* h, const double* a, int64_t M, int64_t K, const double* b, int64_t N,
                                 int32_t lower, int32_t slices, double* v_out, double* rowsq_out);

/* Packed fitted state, for shipping a fit to other processes (one process per GPU, nngp_b200/dist.py) or to a
 * file without a staging copy of the whole N x N factor.  The state is ONE logical array of doubles:
 *     [ X (N*D, row-major) | alpha (N) | lower triangle of L by rows (N(N+1)/2) | 'ntk' only: M (N*N) ].
 * nngp_state_packed_size reports its length; nngp_state_pack copies elements [offset, offset+count) into `dst`
 * (host or device memory); on the receiving side nngp_state_import_begin sizes the buffers,
 * nngp_state_unpack stores a range, nngp_state_import_end derives the rest (layer-0 diagonal, diagonal-block
 * inverses, replicas) and marks the handle fitted.  Every call is complete when it returns.  The receiving handle
 * needs the same config and activation as the one that packed the state. */
NNGP_API int nngp_state_packed_size(nngp_handle* h, int64_t* n_doubles);
NNGP_API int nngp_state_pack(nngp_handle* h, int64_t offset, int64_t count, double* dst);
NNGP_API int nngp_state_import_begin(nngp_handle* h, int64_t N, int64_t D);
NNGP_API int nngp_state_unpack(nngp_handle* h, int64_t offset, int64_t count, const double* src);
NNGP_API int nngp_state_import_end(nngp_handle* h, double lambda);

/*
 * Batch query-line encoder (host C++, multi-threaded) -- scope row f-1.
 * Replaces the per-line Python loop of Estimator.predict (estimator.py:43-50, "TODO :: parallel encoding")
 * and produces bit-identical float64 rows to NNGPEncoder.parse_line_without_card_then_encode /
 * parse_line (neuroestimator/estimator/encoder.py:207-250) and, for single-table workloads, to
 * GeneralQuerySampler.parse_line + transform_to_1d_array (QuerySampler.py:157-221).
 * schema_text, one item per line:
 *     chunk_size <1..64>
 *     table <name>
 *     col <name> num <min> <denominator>         (numerical: [ (v-min)/denominator*1000 ] x {upper, lower})
 *     col <name> cat <number of categories>      (categorical: ceil(n/chunk_size) factorised words)
 *     join <t1_id> <t2_id> <col_name>            (in the order of NNGPEncoder.all_join_triples)
 * format: 0 = "t1,t2@preds1@preds2@joins" (neuroestimator/README.md:35-48), 1 = the same + "@card",
 *         2 = single table "preds@card" (Queries/forest_data).  Lines are '\n'-separated in `blob`.
 * x_out: n_lines x nngp_encoder_dim(); card_out (formats 1, 2) may be NULL.  n_threads <= 0: all cores.
 */
typedef struct nngp_encoder nngp_encoder;
NNGP_API int nngp_encoder_create(const char* schema_text, nngp_encoder** out);
NNGP_API void nngp_encoder_destroy(nngp_encoder* enc);
NNGP_API int nngp_encoder_dim(const nngp_encoder* enc);
NNGP_API const char* nngp_encoder_last_error(const nngp_encoder* enc);
NNGP_API int nngp_encode_lines(nngp_encoder* enc, const char* blob, int64_t blob_len, int64_t n_lines,
                               int32_t format, double* x_out, double* card_out_or_null, int32_t n_threads);

#ifdef __cplusplus
}
#endif
#endif /* NNGP_B200_H */
