/* rlvi_b200.h -- C ABI of librlvi_b200.so: the RLVI E-step + weighted M-step hot path on B200 (sm_100a).
 *
 * The reference (akarakulev/rlvi) is pure Python; it has no FFI.  Its "plugin API" for this path is
 * the set of Python function signatures in standard-learning/rlvi.py, standard-learning/utils.py,
 * deep-learning/methods/train_rlvi.py and online-learning/main.py (SURVEY.md section 8b).  Each entry
 * point below names the reference expression it replaces; the Python drop-in modules in rlvi_b200/
 * (rlvi.py, utils.py, deep.py, online.py) keep the reference signatures and call ONLY these symbols
 * through ctypes (INTEGRATION.md shows the binding).
 *
 * Conventions
 *  - plain C types only; every array pointer is a DEVICE pointer owned by the caller unless the
 *    parameter name ends in `_host`; matrices are row-major, C-contiguous: X[n][d];
 *  - every call is asynchronous and ordered on `stream` (a cudaStream_t passed as void*; NULL = the
 *    legacy default stream); nothing here synchronises the device except rlvi_ctx_* and the
 *    `*_host` convenience calls, which say so;
 *  - scratch memory lives in the context (rlvi_ctx): it grows on demand (a cudaMalloc, the only place
 *    an allocation can happen) and is reused, so steady-state calls never allocate;
 *  - because the scratch is shared, the calls made on ONE context must be stream-ordered with respect
 *    to each other (one stream, or streams the caller chains with events); for concurrent streams or
 *    host threads create one context per stream -- contexts are independent and cheap (8 MiB);
 *  - return value: 0 = RLVI_OK, < 0 = error; rlvi_last_error() gives the thread-local message;
 *  - reductions are deterministic (fixed-order trees over warps, CTAs and ranks; no floating-point
 *    atomics): the same inputs on the same GPU model and world size give the same bits on every run.
 */
#ifndef RLVI_B200_H
#define RLVI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RLVI_OK 0
#define RLVI_ERR_INVALID (-1)     /* bad argument (null pointer, n < 0, ...)            */
#define RLVI_ERR_CUDA (-2)        /* a CUDA runtime call failed; see rlvi_last_error()  */
#define RLVI_ERR_UNSUPPORTED (-3) /* shape outside what the kernels cover (e.g. d > 1024) */
#define RLVI_ERR_NOMEM (-4)       /* scratch allocation failed                          */

typedef struct rlvi_ctx rlvi_ctx;

/* ---- library / context --------------------------------------------------------------------- */
int rlvi_version(void);                      /* 100 * major + minor                               */
const char* rlvi_last_error(void);           /* thread-local, never NULL                          */
int rlvi_ctx_create(int device, rlvi_ctx** out);   /* binds to `device`; synchronous              */
int rlvi_ctx_destroy(rlvi_ctx* ctx);               /* frees the scratch; synchronous              */
int rlvi_ctx_sm_count(const rlvi_ctx* ctx);        /* SMs of the bound device (148 on B200)       */
/* Number of kernels this context has launched since creation (bench.py's `gpu_launches`). */
int64_t rlvi_ctx_launch_count(const rlvi_ctx* ctx);

/* ---- E-step: epsilon fixed point ------------------------------------------------------------ */
/* Which reference loop the iteration reproduces. */
enum rlvi_fp_variant {
  /* standard-learning/rlvi.py:8-20  update_weights: pi0 = 0.95; eps = 1 - mean(pi);
   * rho = eps/(1-eps); pi' = e/(rho+e); stop when ||pi'-pi||_2 < tol; returns the last pi'.      */
  RLVI_FP_STANDARD = 0,
  /* online-learning/main.py:45-58  update_weights_rlvi: pi0 = 0.5; rho = avg/(1-avg);
   * pi' = rho e/(1+rho e); same stop; result divided by max(pi') * n.                            */
  RLVI_FP_ONLINE = 1,
  /* deep-learning/methods/train_rlvi.py:14-38  update_sample_weights: residuals -= min (in place);
   * avg0 = 0.95; pi' = rho e/(1+rho e); first-pass error against the INCOMING weights;
   * weights overwritten; finally weights /= max(weights).                                        */
  RLVI_FP_DEEP = 2
};

/* Written by the fixed-point kernels into device memory (40 bytes); copy it back when needed. */
typedef struct rlvi_fp_result {
  double eps;     /* STANDARD: the last eps = 1 - mean(pi) used; ONLINE/DEEP: 1 - last avg used    */
  double rho;     /* the last ratio used                                                           */
  double sum_pi;  /* sum of the returned posteriors BEFORE the variant's normalisation             */
  double err;     /* ||pi' - pi||_2 of the last pass                                               */
  int32_t iters;  /* passes executed (1..maxiter)                                                  */
  int32_t converged; /* 1 if err < tol stopped the loop, 0 if maxiter did                          */
} rlvi_fp_result;

/* Optional multi-GPU exchange for the fixed point (one process per GPU; the sample dimension is
 * sharded, SURVEY.md section 8e).  `inbox` is THIS rank's window of rlvi_fp_dist_inbox_doubles(world)
 * doubles, zeroed once at setup; `peer_inbox` is a DEVICE array of `world` pointers, entry r addressing rank r's
 * window through NVLink peer mapping (entry `rank` == inbox).  Every pass each rank stores its three
 * partial reductions + a sequence tag into slot `rank` of every peer's window, then sums the `world`
 * slots of its own window in rank order, so all ranks obtain the same bits and take the same stop
 * decision.  NULL => single GPU. */
typedef struct rlvi_fp_dist {
  int32_t rank;
  int32_t world;
  int64_t n_global;          /* total samples over all ranks (the mean's denominator)             */
  double* inbox;             /* device                                                            */
  double* const* peer_inbox; /* device array [world] of device pointers                           */
  uint64_t call_index;       /* 1, 2, 3, ...: the same on every rank, +1 per fixed-point call     */
} rlvi_fp_dist;
int rlvi_fp_dist_inbox_doubles(int world);   /* size of one rank's window, in doubles             */

/* Peer windows for rlvi_fp_dist (one process per GPU; all three calls synchronise the device).
 *   create: allocate + zero this rank's window, export its CUDA IPC handle (RLVI_IPC_HANDLE_BYTES bytes);
 *   open:   `all_handles` = the handles of ranks 0..world-1 concatenated (gathered by the caller over any
 *           transport); maps every peer window over NVLink and returns the DEVICE table of `world`
 *           pointers to use as rlvi_fp_dist.peer_inbox (entry `rank` = own_window);
 *   close:  unmap the peers, free the table and the window.                                            */
#define RLVI_IPC_HANDLE_BYTES 64
int rlvi_dist_window_create(rlvi_ctx* ctx, int world, void** window_out, unsigned char* handle_out);
int rlvi_dist_window_open(rlvi_ctx* ctx, int rank, int world, void* own_window,
                          const unsigned char* all_handles, void** peer_table_out);
int rlvi_dist_window_close(rlvi_ctx* ctx, int rank, int world, void* own_window, void* peer_table);

/* All-reduce (SUM) of a small FP64 statistics vector over the ranks WITHOUT NCCL: every rank stores its
 * `count` doubles into slot `rank` of every peer's window over NVLink, publishes a sequence tag, waits for the
 * `world` tags in its own window and adds the slots in rank order -- every rank ends with the same bits in
 * `buf` (in place).  One launch; replaces the NCCL all-reduce of the d*d + 2d + 2 statistics after
 * rlvi_weighted_moments_f64 (SURVEY.md section 8e).  count <= RLVI_DIST_STATS_CAPACITY; `dist->call_index`
 * must be 1, 2, 3, ... identically on every rank (its own sequence, independent of the fixed-point calls).
 * The window is the one created by rlvi_dist_window_create (it reserves the statistics area). */
#define RLVI_DIST_STATS_CAPACITY 8192
int rlvi_stats_allreduce_f64(rlvi_ctx* ctx, double* buf, int count, const rlvi_fp_dist* dist, void* stream);

/* FP64 fixed point (STANDARD or ONLINE).
 *   losses   [n]  per-sample loss l_i, or NULL when `e_work` already holds e_i = exp(-l_i)
 *   scale    device scalar s or NULL (=1): the kernel uses e_i = exp(-s * l_i); lets the caller fold
 *            the `0.5 / sigma2` of rlvi.py:51,59,74,83 in without a host round trip
 *   e_work   [n]  scratch the kernel fills with e_i on its first pass and re-reads afterwards
 *   pi_out   [n]  the returned posteriors (may alias `losses`; may NOT alias `e_work`)
 *   result   device rlvi_fp_result                                                               */
int rlvi_fixed_point_f64(rlvi_ctx* ctx, int variant, const double* losses, const double* scale,
                         double* e_work, int64_t n, double tol, int maxiter, double* pi_out,
                         rlvi_fp_result* result, const rlvi_fp_dist* dist, void* stream);

/* Same, starting from the initial posterior `pi0` in (0, 1) instead of the variant's constant.  The reference
 * restarts every online batch from 0.5 (online-learning/main.py:48, quirk Q11); carrying the previous batch's
 * mean posterior (result.sum_pi / n) into the next call is the OPT-IN extension BASELINE.json's config 4 names. */
int rlvi_fixed_point_init_f64(rlvi_ctx* ctx, int variant, const double* losses, const double* scale,
                              double* e_work, int64_t n, double tol, int maxiter, double pi0, double* pi_out,
                              rlvi_fp_result* result, const rlvi_fp_dist* dist, void* stream);

/* FP32 fixed point, DEEP variant: `residuals` [n] and `weights` [n] are both updated in place,
 * exactly as methods/train_rlvi.py:14-38 leaves them.  `e_work` [n] is FP32 scratch. */
int rlvi_fixed_point_deep_f32(rlvi_ctx* ctx, float* residuals, float* weights, float* e_work, int64_t n,
                              float tol, int maxiter, rlvi_fp_result* result, const rlvi_fp_dist* dist,
                              void* stream);

/* standard-learning/rlvi.py:34-39  shift_obj's inner sum:  out[0] = sum_i t_i/(c + t_i),
 * t_i = exp(-l_i + s).  One pass; the Brent search (scipy) stays on the host (SURVEY.md H4).
 * If `pi_out` != NULL the per-sample ratios are also written (rlvi.py:42). */
int rlvi_shift_sum_f64(rlvi_ctx* ctx, const double* losses, int64_t n, double shift, double c,
                       double* pi_out, double* out_sum, void* stream);

/* The same sum from e_i = exp(-l_i) (what rlvi_fixed_point_f64 leaves in `e_work`) and scale_t = exp(shift):
 * t_i = e_i * scale_t.  No exp per sample: the 12-21 objective evaluations of one constrained E-step become
 * HBM-bound passes.  Agrees with rlvi_shift_sum_f64 to rounding (exp(-l+s) vs exp(-l) exp(s)). */
int rlvi_shift_sum_e_f64(rlvi_ctx* ctx, const double* e, int64_t n, double scale_t, double c, double* pi_out,
                         double* out_sum, void* stream);

/* ---- per-sample losses (one pass over X) ------------------------------------------------------ */
enum rlvi_loss_kind {
  /* utils.py:19-21 cross_entropy: phi = b + x.theta;  l = -y phi + phi + log1p(exp(-phi)).
   * params = [b, theta(d)] if `intercept` else [theta(d)].                                        */
  RLVI_LOSS_LOGISTIC_CE = 0,
  /* utils.py:62-64 the loss sklearn_log_reg reports: l = -log P(class 0|x) = log(1 + exp(phi)),
   * label-independent (quirk Q3).  params as above.                                               */
  RLVI_LOSS_SOFTPLUS = 1,
  /* rlvi.py:72,81 squared residual: l = (y - x.theta)^2.   params = [theta(d)] (or [b, theta]).   */
  RLVI_LOSS_SQRES = 2,
  /* rlvi.py:49,57 squared distance to the mean: l = ||theta - x||^2.   params = [theta(d)].       */
  RLVI_LOSS_SQDIST = 3,
  /* utils.py:77-79 PCA reconstruction: l = ||x||^2 - (x.theta)^2.   params = [theta(d)].          */
  RLVI_LOSS_PCA = 4,
  /* utils.py:93-101 Gaussian NLL: l = 0.5 [(x-mu)^T cov^-1 (x-mu) + c] = 0.5 [||U (x-mu)||^2 + c].
   * params = [c, mu(d), U(d*d) row-major], U UPPER triangular with U^T U = cov^-1 (the inverse of
   * an upper Cholesky factor of cov; entries below the diagonal are ignored),
   * c = log|cov| + d log(2 pi).  d <= 128.                                                        */
  RLVI_LOSS_GAUSSIAN = 5
};

/* One pass over X (and y):
 *   losses_out [n] (or NULL)      l_i
 *   e_out      [n] (or NULL)      exp(-l_i), for the fixed point
 *   weights    [n] (or NULL)      pi_i; when given, wsum_out[0] = sum pi_i l_i, wsum_out[1] = sum pi_i
 *                                 (the sigma2 = pi.r2 / sum pi of rlvi.py:50,58,73,82)
 *   wsum_out   device double[2] (required iff weights != NULL)                                     */
int rlvi_loss_f64(rlvi_ctx* ctx, int kind, int intercept, const double* X, const double* y, int64_t n,
                  int d, const double* params, const double* weights, double* losses_out, double* e_out,
                  double* wsum_out, void* stream);

/* ---- weighted M-step statistics (one pass over X) --------------------------------------------- */
/* With w_i = weights_i (power = 1) or weights_i^2 (power = 2: the Gram of the pi-scaled rows that
 * utils.py:82-84 hands to PCA):
 *   S0   = sum w_i                       out[0]
 *   Swy  = sum w_i y_i                   out[1]            (0 if y == NULL)
 *   S1   = X^T w                         out[2 .. 2+d)     (rlvi.py:48,56; utils.py:103)
 *   Sy   = X^T (w*y)                     out[2+d .. 2+2d)  (zeros if y == NULL; rlvi.py:71,80)
 *   G    = X^T diag(w) X  (symmetric)    out[2+2d .. 2+2d+d*d) row-major, both triangles filled
 *                                        (rlvi.py:70-71,79-80; utils.py:36-38,105); skipped (left
 *                                        untouched) when want_gram == 0
 * For power = 2, S1 is still X^T weights (first power: the column mean PCA subtracts) while S0 and G
 * use the square.  `out` is a device buffer of rlvi_moments_out_doubles(d) doubles.               */
int rlvi_moments_out_doubles(int d);
int rlvi_weighted_moments_f64(rlvi_ctx* ctx, const double* X, const double* y, const double* weights,
                              int64_t n, int d, int power, int want_gram, double* out, void* stream);

/* Same statistics about a centre c[d] (device array): every x_i is replaced by (x_i - c), i.e.
 * G = sum w (x-c)(x-c)^T, S1 = sum weights (x-c), Sy = sum w y (x-c); S0, Swy unchanged.  utils.py:103-105
 * centres the samples at the weighted mean before forming the covariance; one pass for the mean
 * (want_gram = 0) followed by one centred pass reproduces that without the cancellation of G/S0 - mu mu^T. */
int rlvi_weighted_moments_centered_f64(rlvi_ctx* ctx, const double* X, const double* y, const double* weights,
                                       const double* center, int64_t n, int d, int power, int want_gram,
                                       double* out, void* stream);

/* ---- FP32-stored samples (SURVEY.md section 8d "FP32 mode"; BASELINE.json config 3: N = 2^24, d = 512) ---------
 * X is float32 [n][d] row-major; every per-sample vector (y, weights, losses, e) and every statistic stays FP64.
 * The Gram contraction runs on the 5th-generation tensor cores (tcgen05.mma kind::tf32, accumulators in TMEM):
 *   RLVI_TF32X3  three products per term (hi*hi + lo*hi + hi*lo; z = hi + lo with hi the TF32 rounding) with short FP32
 *                accumulation chains flushed into FP64; default.  Against an FP64 evaluation on the same float32 samples,
 *                entry by entry: |G - G_ref| <= 1e-5 B with B = |X|^T diag(w) |X|, |S1 - S1_ref| <= 1e-5 |X|^T weights,
 *                |Sy - Sy_ref| <= 1e-5 |X|^T |w y| (the 1e-5 FP32 tolerance of BASELINE.json's north_star; measured on
 *                a B200 at 1000 W: <= 7e-7 B for d <= 128, <= 2.8e-6 B for d > 128, 2.3e-6 B with 32 Ki-row FP32
 *                register sums of all-positive data).  Supported range: every scaled sample z = s_i x_ij, s_i =
 *                (pi_i / 2^e)^(power / 2) with 2^e the even power of two at or above max pi, is 0 or has
 *                2^-60 <= |z| < 2^56.  Below it the products leave the FP32 normal range and lose their corrections
 *                (measured: 1.4e-6 B at 2^-66, 2.6e-5 B at 2^-68, 4e-4 B at 2^-70); from 2^56 on, a 32 Ki-row FP32
 *                sum can overflow (non-finite G measured at 2^61 with 32 rows per CTA).  Rows outside the range, e.g.
 *                weights far below max pi, lose at most their own share of B.  On the CTA-pair kernel (d > 128) the two
 *                correction products run as BF16 (kind::f16), which keeps that accuracy at two thirds of the tensor
 *                time; RLVI_TF32_PURE3=1 in the environment keeps all three in TF32;
 *   RLVI_TF32X1  one TF32 product per term (operands rounded to 11 bits, zero-mean error): 3x fewer tensor-core
 *                flops, ~1e-3 / sqrt(rows) relative accuracy.
 * Same output layout as rlvi_weighted_moments_f64.  Replaces utils.py:82-84 (power = 2), rlvi.py:70-71,79-80 and
 * utils.py:36-38 (power = 1) for float32 inputs.  d <= 512 with d % 4 == 0 and a 16-byte aligned X take the tensor
 * path; other shapes (d <= 1024) are converted chunk-wise and summed by the FP64 kernels. */
#define RLVI_TF32X3 0
#define RLVI_TF32X1 1
int rlvi_weighted_moments_f32(rlvi_ctx* ctx, const float* X, const double* y, const double* weights, int64_t n,
                              int d, int power, int want_gram, int precision, double* out, void* stream);

/* rlvi_loss_f64 for float32 samples (all kinds except RLVI_LOSS_GAUSSIAN; d <= 4096): products and sums in FP64
 * from the converted samples, outputs FP64. */
int rlvi_loss_f32(rlvi_ctx* ctx, int kind, int intercept, const float* X, const double* y, int64_t n, int d,
                  const double* params, const double* weights, double* losses_out, double* e_out, double* wsum_out,
                  void* stream);

/* utils.py:40-41  the MM/gradient step's data term:  out[0] = sum c_i, out[1..d] = X^T c with
 * c_i = w_i (sigmoid(b + x_i.theta) - y_i);  params = [b, theta(d)].  `out` = device double[d+1]. */
int rlvi_logistic_grad_f64(rlvi_ctx* ctx, const double* X, const double* y, const double* weights,
                           int64_t n, int d, const double* params, double* out, void* stream);

/* utils.py:7-16  overflow-free logistic function of an N-vector: out_i = 1 / (1 + exp(-x_i)). */
int rlvi_sigmoid_f64(rlvi_ctx* ctx, const double* x, int64_t n, double* out, void* stream);

/* online-learning/main.py:84-85  cross_entropy: out_i = -t_i l_i - (1 - t_i) l_i (== -l_i up to rounding: quirk Q11). */
int rlvi_online_ce_f64(rlvi_ctx* ctx, const double* log_proba, const double* targets, int64_t n, double* out, void* stream);

/* Curvature weights of the L2-regularised logistic objective utils.py:61-73 hands to liblinear
 * (1/2 ||theta||^2 + C sum_i pi_i logloss_i): out_i = weights_i e_i (1 - e_i), where e_i = exp(-cross_entropy_i) is
 * what rlvi_loss_f64(LOGISTIC_CE, e_out) leaves behind (= sigmoid or 1 - sigmoid for a 0/1 label, either way
 * e (1 - e) = s (1 - s)).  rlvi_weighted_moments_f64 with these weights is the exact Hessian of the data term: the
 * Newton / IRLS M-step of the drop-in's sklearn_log_reg. */
int rlvi_irls_weights_f64(rlvi_ctx* ctx, const double* e, const double* weights, int64_t n, double* out, void* stream);

/* standard-learning/rrm.py:12-33 (= online-learning/main.py:61-81 update_weights_rrm), the competitor weight rule on
 * the same reduction skeleton (SURVEY.md section 8f rank 4):  out_sum[0] = sum_i max(exp(-l_i * inv_alpha), cutoff)
 * (one evaluation of the objective SciPy's Brent minimises, rrm.py:17-21); if w_out != NULL also
 * w_out_i = exp(-l_i * inv_alpha) * norm (the final weights, rrm.py:32). */
int rlvi_rrm_sum_f64(rlvi_ctx* ctx, const double* losses, int64_t n, double inv_alpha, double cutoff, double norm,
                     double* w_out, double* out_sum, void* stream);

/* standard-learning/sever.py:22-31 (linear regression) / :95-104 (PCA): the two per-sample passes of one SEVER filter
 * step on row-major FP64 X, dot_i = x_i . u (u = device double[d]):
 *   op 0: c_i = scalar * (dot_i - b_i)  (b may be NULL = 0);  out0_i = c_i, out1_i = active_i * c_i^2,
 *         out2_i = c_i != 0 ? 1 / c_i : 0   -- the per-sample gradient is g_i = c_i x_i, and
 *         rlvi_weighted_moments_f64(X, y = out2, weights = out1) then returns sum_active g_i g_i^T and sum_active g_i;
 *   op 1: out0_i = active_i != 0 ? (a_i * dot_i - scalar)^2 : -1     -- the outlier scores tau_i with a = c, u = v,
 *         scalar = mean(g) . v.   `active` (0/1 doubles, NULL = all active) is the filter's current active set. */
int rlvi_sever_pass_f64(rlvi_ctx* ctx, const double* X, int64_t n, int d, const double* u, int op, double scalar,
                        const double* a, const double* b, const double* active, double* out0, double* out1, double* out2,
                        void* stream);

/* ---- deep path (FP32) ------------------------------------------------------------------------- */
/* methods/train_rlvi.py:89-94 fused with its autograd backward (line 96):
 *   loss_i = CE(logits_i, label_i);  residuals[indexes_i] = loss_i (detached: quirk Q8);
 *   out_loss[0] = mean_i loss_i * weights[indexes_i];
 *   dlogits_i = (softmax(logits_i) - onehot(label_i)) * weights[indexes_i] / B   (NULL = forward only)
 *   out_correct[0], [1] = number of rows whose label is in the top-1 / top-5 logits (NULL = skip;
 *   replaces utils.py:65-79 `accuracy`, called at train_rlvi.py:85).
 * logits [B][C] FP32 row-major; labels, indexes int64 [B]; residuals, weights FP32 [n_train].
 * `indexes` may be NULL (identity, n_train >= B).                                                 */
int rlvi_wce_fwd_bwd_f32(rlvi_ctx* ctx, const float* logits, const int64_t* labels, const int64_t* indexes,
                         const float* weights, float* residuals, int64_t batch, int classes,
                         int64_t n_train, float* per_sample_out, float* dlogits, float* out_loss,
                         int32_t* out_correct, void* stream);

/* methods/train_rlvi.py:41-49 false_negative_criterion + lines 102-103 truncation:
 *   beta = alpha * sum(1-w); walk the weights in descending order accumulating (1-w) while the
 *   running mass stays <= beta; the threshold is the last weight reached (the smallest weight if
 *   none fits: quirk Q9).  out_threshold[0] = max(prev_threshold, that value) (line 102; pass
 *   prev_threshold = 0 for the bare criterion); if `truncate` != 0, weights[w < threshold] = 0 in
 *   place.  The running mass is accumulated in FP64 (SURVEY.md H5).                               */
int rlvi_fn_threshold_f32(rlvi_ctx* ctx, float* weights, int64_t n, float alpha, float prev_threshold,
                          int truncate, float* out_threshold, void* stream);

/* ---- batched small problems (many independent fits in one launch) ----------------------------- */
/* `nprob` problems packed back to back: problem b owns rows [offsets[b], offsets[b+1]) of every per-row array (X [rows][d]
 * row-major, y, losses, pi_out); `offsets` is a DEVICE int64[nprob + 1].  One warp runs one problem entirely on chip
 * (per-row vector, d x d statistics and Cholesky factor in shared memory), so a problem's bits depend only on its own rows,
 * never on its place in the batch or on the batch size.  Every segment is checked on the device: a segment that breaks
 * 0 <= offsets[b] < offsets[b+1] <= n_rows or is longer than the cap gets NaN outputs and status -1, and none of its rows
 * is read or written. */
enum rlvi_batched_model {
  RLVI_BATCHED_MEAN = 0,   /* standard-learning/rlvi.py:46-65  mean              */
  RLVI_BATCHED_LINREG = 1  /* standard-learning/rlvi.py:68-89  linear_regression */
};

/* Rows one problem may have at `d` features (1 <= d <= 64; 0 outside): the shared-memory budget of one warp.  At least
 * 1024 at every d.  rlvi_batched_fixed_point_f64 admits rlvi_batched_max_rows(1) rows per problem. */
int rlvi_batched_max_rows(int d);

/* standard-learning/rlvi.py:8-20 update_weights on every segment of `losses` (the RLVI_FP_STANDARD iteration of
 * rlvi_fixed_point_f64, same operation order): pi_out [n_rows], results [nprob] (a rejected segment: NaN fields,
 * iters = converged = -1, its pi rows untouched). */
int rlvi_batched_fixed_point_f64(rlvi_ctx* ctx, const double* losses, const int64_t* offsets, int nprob,
                                 int64_t n_rows, double tol, int maxiter, double* pi_out,
                                 rlvi_fp_result* results, void* stream);

/* The whole EM loop of standard-learning/rlvi.py:46-65 (MEAN) or :68-89 (LINREG) per problem, following the drop-in
 * rlvi_b200/rlvi.py: pi = 1; M-step (MEAN theta = S1/S0, r^2 = ||theta - x||^2; LINREG the normal equations
 * G theta = b with G = X^T Pi X, b = X^T Pi y by Cholesky, r^2 = (y - x.theta)^2); then up to `maxiter` times the E-step
 * (the update_weights fixed point, tol 1e-3, maxiter 100, on the losses 0.5 r^2 / sigma2) and the M-step, stopping at
 * the first theta with ||theta - prev|| / ||prev|| <= tol.  y is NULL for MEAN.  Outputs: theta_out [nprob][d],
 * iters_out [nprob] (EM iterations), status_out [nprob]: 0 stop test met, 1 maxiter reached, 2 the LINREG Cholesky
 * failed the drop-in's pivot test (min L_ii^2 / G_ii > 2^-52 (d + sqrt(n)); rank-deficient or ill-conditioned design,
 * n < d included) at some iteration: theta is NaN and the problem needs the drop-in's minimum-norm solve; -1 rejected
 * segment.  RLVI_ERR_UNSUPPORTED for d outside 1..64. */
int rlvi_batched_em_f64(rlvi_ctx* ctx, int model, const double* X, const double* y, const int64_t* offsets, int nprob,
                        int64_t n_rows, int d, double tol, int maxiter, double* theta_out, int32_t* iters_out,
                        int32_t* status_out, void* stream);

enum rlvi_batched_logreg_mstep {
  RLVI_BATCHED_LOGREG_NEWTON = 0,  /* standard-learning/utils.py:61-73 via the drop-in's Newton solve */
  RLVI_BATCHED_LOGREG_MM = 1       /* standard-learning/utils.py:32-58                              */
};

/* Rows one problem of rlvi_batched_logistic_f64 may have at `d` features (1 <= d <= 63; 0 outside): the shared-memory
 * budget of one warp.  At least 1024 at every d and at least 2000 at d <= 8. */
int rlvi_batched_logistic_max_rows(int d);

/* The whole EM loop of standard-learning/rlvi.py:92-108 per problem, following the drop-in rlvi_b200/rlvi.py
 * logistic_regression: pi = 1; M-step; then up to `maxiter` times the E-step (the update_weights fixed point, tol 1e-3,
 * maxiter 100, on the M-step's unscaled losses) and the M-step, stopping at the first theta with
 * ||theta - prev|| / ||prev|| <= tol.  The design is [1, X]: theta has d + 1 entries, intercept first.  M-steps:
 *   NEWTON  the minimiser of 1/2 |theta|^2 + 100 sum_i w_i CE_i, w = pi / max pi, by the drop-in's damped Newton
 *           iteration (Hessian I + 100 [1,X]^T diag(w e (1 - e)) [1,X] by Cholesky, Armijo backtracking, stop when a full
 *           step has |step| <= 1e-9 (1 + |theta|), at most 60 steps), warm-started from the previous EM iterate (0 first);
 *           E-step losses softplus(b + x.w), whatever the label;
 *   MM      theta <- theta - Q^-1 [1,X]^T (pi (sigmoid - y)) from theta = 0 while |delta theta| > 1e-2, with
 *           Q = 1/4 [1,X]^T Pi [1,X] factored once per M-step; E-step losses the cross-entropy with y.
 * Outputs: theta_out [nprob][d + 1], iters_out [nprob] (EM iterations), status_out [nprob]: 0 stop test met, 1 maxiter
 * reached, 2 the problem needs the single-problem drop-in (theta NaN): Newton did not converge in 60 steps (a non-finite
 * objective included), or MM's Q failed rlvi_batched_em_f64's pivot test (min L_ii^2 / Q_ii > 2^-52 (d + 1 + sqrt(n))),
 * or MM took 10000 steps; -1 rejected segment.  RLVI_ERR_UNSUPPORTED for d outside 1..63. */
int rlvi_batched_logistic_f64(rlvi_ctx* ctx, int mstep, const double* X, const double* y, const int64_t* offsets,
                              int nprob, int64_t n_rows, int d, double tol, int maxiter, double* theta_out,
                              int32_t* iters_out, int32_t* status_out, void* stream);

/* ---- host-buffer convenience (the drop-in's NumPy route; bench.py's `e2e`) ------------------- */
/* One E+M step of the logistic model on HOST buffers (pinned or pageable): chunks of X/y are copied
 * H2D on a copy stream while the loss kernel consumes the previous chunk; then the fixed point and
 * the statistics pass run on the device-resident copy, and the results are copied back.
 *   X_host [n][d], y_host [n], params_host [d+1] (intercept first)
 *   pi_host [n] (or NULL), moments_host [rlvi_moments_out_doubles(d)], result_host
 * Needs n*(d+4)*8 bytes of device memory, taken from (and kept by) the context.  Synchronous. */
int rlvi_em_step_logistic_host(rlvi_ctx* ctx, const double* X_host, const double* y_host, int64_t n, int d,
                               const double* params_host, double tol, int maxiter, double* pi_host,
                               double* moments_host, rlvi_fp_result* result_host);

/* The same step on THIS RANK'S SHARD of a sample-sharded data set (one process per GPU): the fixed point
 * exchanges its sums with the peers inside the kernel (`fp_dist`, n_global = total samples), the statistics
 * are all-reduced over the peer windows (`stats_dist`); both structs come from the same window with their own
 * call_index sequences.  moments_host receives the GLOBAL statistics, pi_host this shard's posteriors. */
int rlvi_em_step_logistic_host_sharded(rlvi_ctx* ctx, const double* X_host, const double* y_host, int64_t n, int d,
                                       const double* params_host, double tol, int maxiter, double* pi_host,
                                       double* moments_host, rlvi_fp_result* result_host,
                                       const rlvi_fp_dist* fp_dist, const rlvi_fp_dist* stats_dist);

#ifdef __cplusplus
}
#endif
#endif /* RLVI_B200_H */
