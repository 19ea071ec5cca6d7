// batched.cu -- many small, independent RLVI problems in one launch: one warp per problem, the whole loop on chip.
//
// Replaces, per problem, the drop-in calls (rlvi_b200/rlvi.py) that the reference's experiment driver makes thousands
// of times on tiny data (standard-learning/main.py: test_mean, test_linear_regression, N = 40..100, d = 2..10):
//   standard-learning/rlvi.py:8-20    update_weights     -> batched_fp_kernel
//   standard-learning/rlvi.py:46-65   mean               -> batched_em_kernel<MODEL_MEAN>
//   standard-learning/rlvi.py:68-89   linear_regression  -> batched_em_kernel<MODEL_LINREG>
//   standard-learning/rlvi.py:92-108  logistic_regression -> batched_logreg_kernel<LOGREG_NEWTON / LOGREG_MM>
// At that size a drop-in EM iteration is ~10 launches and two host synchronisations; here a problem's EM loop, its
// fixed points, the d x d Cholesky and the stop tests run inside one warp, with no host round trip.
//
// Layout: problem b owns rows [offsets[b], offsets[b+1]) of X [rows][d], y, losses and pi.  Each warp keeps in shared
// memory one per-row vector that is r^2 after an M-step, e = exp(-scale r^2) during the fixed point and pi after it, and
// (LINREG) the lower triangle of G = X^T Pi X, b = X^T Pi y and the Cholesky factor.  X and y are read from global memory
// (twice per EM iteration: statistics and residuals); e is read by every fixed-point pass.
//
// Determinism: a problem's bits depend only on its own rows.  Every sum runs in an order fixed relative to the problem's
// first row -- lane-strided partial sums plus the xor-shuffle tree, or one lane summing over the rows in order -- so neither
// the problem's index, the batch size nor the warp that runs it changes anything.  No atomics.
#include <math.h>

#include "common.cuh"

namespace {

constexpr int kMaxD = 64;
constexpr int kMinWarpDoubles = 1536;                 // at least 12 KiB of shared memory per problem
constexpr int kMinRows = 1024;                        // the cap admits n = 1024 at every supported d
constexpr int kMaxWarpsPerCta = 16;
constexpr size_t kSmemBudget = size_t(220) * 1024;    // dynamic shared memory of one CTA
constexpr double kEps52 = 2.220446049250313e-16;      // torch.finfo(float64).eps

enum { MODEL_MEAN = RLVI_BATCHED_MEAN, MODEL_LINREG = RLVI_BATCHED_LINREG };
enum { ST_CONVERGED = 0, ST_MAXITER = 1, ST_HOST_SOLVE = 2, ST_BAD_SEGMENT = -1 };

// Per-warp shared memory, in doubles: rows [cap] | G [d][d + 1] (odd row stride: the column sweeps of the Cholesky hit
// distinct banks) | b [d] | theta [d] | theta_prev [d] | diag(L) [d].
__host__ __device__ inline int g_ld(int d) { return d + 1; }
__host__ __device__ inline int warp_doubles(int d) {
  const int need = kMinRows + d * g_ld(d) + 4 * d;
  return need > kMinWarpDoubles ? need : kMinWarpDoubles;
}
__host__ __device__ inline int max_rows(int d) { return warp_doubles(d) - d * g_ld(d) - 4 * d; }
inline int warps_per_cta(size_t warp_bytes) {
  const int w = int(kSmemBudget / warp_bytes);
  return w > kMaxWarpsPerCta ? kMaxWarpsPerCta : w;
}

struct FpOut {
  double eps, rho, sum_pi, err;
  int iters, converged;
};

// The STANDARD fixed point of fp_small_kernel_f64 (fixed_point.cu) on one warp: `se` holds the n losses on entry and
// e_i = exp(-(scale l_i)) on return; the returned rho gives the last posterior pi'_i = e_i / (rho + e_i).
__device__ FpOut warp_fixed_point(double* se, int n, double scale, double tol, int maxiter) {
  const int lane = threadIdx.x & 31;
  const double pi0 = 0.95;
  double eps = 1.0 - pi0;
  double rho_new = eps / (1.0 - eps), rho_old = 0.0;
  double s1 = 0.0, s2 = 0.0;
  for (int i = lane; i < n; i += kWarp) {
    const double ev = exp(-(scale * se[i]));
    se[i] = ev;
    const double pn = ev / (rho_new + ev);
    const double d = pn - pi0;
    s1 += pn;
    s2 = fma(d, d, s2);
  }
  double S = warp_sum(s1), err = sqrt(warp_sum(s2));
  int k = 1, converged = 0;
  while (true) {
    if (err < tol) { converged = 1; break; }
    if (k >= maxiter) break;
    rho_old = rho_new;
    const double avg = S / double(n);
    eps = 1.0 - avg;
    rho_new = eps / (1.0 - eps);
    ++k;
    double a1 = 0.0, a2 = 0.0;
    for (int i = lane; i < n; i += kWarp) {
      const double ev = se[i];
      const double pn = ev / (rho_new + ev);
      const double d = pn - ev / (rho_old + ev);
      a1 += pn;
      a2 = fma(d, d, a2);
    }
    S = warp_sum(a1);
    err = sqrt(warp_sum(a2));
  }
  __syncwarp();
  return FpOut{eps, rho_new, S, err, k, converged};
}

// Segment [start, end) of problem b, checked against the arrays: 0 <= start < end <= n_rows, end - start <= cap.
__device__ __forceinline__ bool segment(const int64_t* offsets, int b, int64_t n_rows, int cap, int64_t& start, int& n) {
  start = offsets[b];
  const int64_t end = offsets[b + 1];
  if (!(start >= 0 && start < end && end <= n_rows && end - start <= cap)) return false;
  n = int(end - start);
  return true;
}

__global__ void batched_fp_kernel(const double* __restrict__ losses, const int64_t* __restrict__ offsets, int nprob,
                                  int64_t n_rows, int cap, double tol, int maxiter, double* __restrict__ pi_out,
                                  rlvi_fp_result* __restrict__ results) {
  extern __shared__ double batched_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.x * (blockDim.x >> 5) + warp;
  if (b >= nprob) return;
  double* se = batched_smem + size_t(warp) * cap;
  int64_t start;
  int n;
  if (!segment(offsets, b, n_rows, cap, start, n)) {
    if (lane == 0) results[b] = rlvi_fp_result{NAN, NAN, NAN, NAN, -1, -1};
    return;
  }
  for (int i = lane; i < n; i += kWarp) se[i] = losses[start + i];
  __syncwarp();
  const FpOut r = warp_fixed_point(se, n, 1.0, tol, maxiter);
  for (int i = lane; i < n; i += kWarp) {
    const double ev = se[i];
    pi_out[start + i] = ev / (r.rho + ev);                   // rlvi.py:15
  }
  if (lane == 0) results[b] = rlvi_fp_result{r.eps, r.rho, r.sum_pi, r.err, r.iters, r.converged};
}

// ---- M-step ------------------------------------------------------------------------------------------------------------
// On entry sr[i] = pi_i; on return sr[i] = r^2_i, th = theta, and (wl, w) = (sum pi r^2, sum pi), the weighted sums the
// drop-in's loss pass returns (rlvi_loss_f64, wsum_out).  Returns false when LINREG's Cholesky fails the pivot test of
// rlvi.py's _gpu_sym_solve (the problem then needs the host's minimum-norm solve).
template <int MODEL>
__device__ bool mstep(const double* __restrict__ X, const double* __restrict__ y, int n, int d, double* sr, double* G,
                      double* bv, double* th, double* dl, double& wl, double& w) {
  const int lane = threadIdx.x & 31;
  const int ld = g_ld(d);
  if (MODEL == MODEL_MEAN) {
    double s0 = 0.0;
    for (int i = lane; i < n; i += kWarp) s0 += sr[i];
    s0 = warp_sum(s0);
    for (int j = lane; j < d; j += kWarp) {                  // S1_j = sum_i pi_i x_ij, rows in order
      double acc = 0.0;
      for (int i = 0; i < n; ++i) acc = fma(sr[i], X[int64_t(i) * d + j], acc);
      th[j] = acc / s0;                                      // rlvi.py:48,56
    }
  } else {
    // G (lower triangle) and b: one lane per entry, rows in order
    const int T = d * (d + 1) / 2;
    for (int t = lane; t < T + d; t += kWarp) {
      int j, k;
      if (t < T) {
        j = int((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
        while (j * (j + 1) / 2 > t) --j;
        while ((j + 1) * (j + 2) / 2 <= t) ++j;
        k = t - j * (j + 1) / 2;
      } else {
        j = t - T;
        k = -1;
      }
      const double* src = k >= 0 ? X + k : y;              // column k of X, or y for b
      const int stride = k >= 0 ? d : 1;
      double acc = 0.0;
      for (int i = 0; i < n; ++i) acc = fma(sr[i] * X[int64_t(i) * d + j], src[int64_t(i) * stride], acc);
      if (k >= 0) G[j * ld + k] = acc;
      else bv[j] = acc;
    }
    __syncwarp();
    // Cholesky G = L L^T in place (lower triangle; diag(L) in dl), left-looking, one column per step.  Accepted iff every
    // pivot L_jj^2 / G_jj exceeds eps (d + sqrt(n)), the test of _gpu_sym_solve (torch.linalg.cholesky_ex info == 0 and
    // min(diag(L)^2 / diag(G)) > rtol).
    const double rtol = kEps52 * (double(d) + sqrt(double(n)));
    for (int j = 0; j < d; ++j) {
      const double gjj = G[j * ld + j];
      double s = gjj;
      for (int k = 0; k < j; ++k) s = fma(-G[j * ld + k], G[j * ld + k], s);
      const double ljj = sqrt(s);
      if (!(s > 0.0) || !(ljj * ljj / gjj > rtol)) return false;      // warp-uniform: every lane has the same bits
      for (int i = j + 1 + lane; i < d; i += kWarp) {
        double t = G[i * ld + j];
        for (int k = 0; k < j; ++k) t = fma(-G[i * ld + k], G[j * ld + k], t);
        G[i * ld + j] = t / ljj;
      }
      if (lane == 0) dl[j] = ljj;
      __syncwarp();
    }
    // L z = b, then L^T theta = z (column sweeps; z overwrites b)
    for (int k = 0; k < d; ++k) {
      const double zk = bv[k] / dl[k];
      __syncwarp();
      for (int i = k + 1 + lane; i < d; i += kWarp) bv[i] = fma(-G[i * ld + k], zk, bv[i]);
      if (lane == 0) bv[k] = zk;
      __syncwarp();
    }
    for (int k = d - 1; k >= 0; --k) {
      const double tk = bv[k] / dl[k];
      __syncwarp();
      for (int i = lane; i < k; i += kWarp) bv[i] = fma(-G[k * ld + i], tk, bv[i]);
      if (lane == 0) th[k] = tk;
      __syncwarp();
    }
  }
  __syncwarp();
  // per-row loss (rlvi_loss_f64's SQDIST / SQRES arithmetic) and the weighted sums; r^2 replaces pi in place
  double a0 = 0.0, a1 = 0.0;
  for (int i = lane; i < n; i += kWarp) {
    const double* xi = X + int64_t(i) * d;
    double a = 0.0, l;
    if (MODEL == MODEL_MEAN) {
      for (int k = 0; k < d; ++k) {
        const double t = th[k] - xi[k];
        a = fma(t, t, a);
      }
      const double r = sqrt(a);                              // rlvi.py:49,57  np.linalg.norm(theta - x)**2
      l = r * r;
    } else {
      for (int k = 0; k < d; ++k) a = fma(xi[k], th[k], a);
      const double r = y[i] - a;                             // rlvi.py:72,81
      l = r * r;
    }
    const double pi = sr[i];
    a0 = fma(pi, l, a0);
    a1 += pi;
    sr[i] = l;
  }
  wl = warp_sum(a0);
  w = warp_sum(a1);
  __syncwarp();
  return true;
}

template <int MODEL>
__global__ void batched_em_kernel(const double* __restrict__ X, const double* __restrict__ y,
                                  const int64_t* __restrict__ offsets, int nprob, int64_t n_rows, int d, double tol,
                                  int maxiter, double* __restrict__ theta_out, int32_t* __restrict__ iters_out,
                                  int32_t* __restrict__ status_out) {
  extern __shared__ double batched_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.x * (blockDim.x >> 5) + warp;
  if (b >= nprob) return;
  const int cap = max_rows(d);
  double* sr = batched_smem + size_t(warp) * warp_doubles(d);
  double* G = sr + cap;
  double* bv = G + d * g_ld(d);
  double* th = bv + d;
  double* thp = th + d;
  double* dl = thp + d;
  double* out = theta_out + int64_t(b) * d;
  int64_t start;
  int n;
  if (!segment(offsets, b, n_rows, cap, start, n)) {
    for (int j = lane; j < d; j += kWarp) out[j] = NAN;
    if (lane == 0) {
      iters_out[b] = 0;
      status_out[b] = ST_BAD_SEGMENT;
    }
    return;
  }
  const double* Xb = X + start * d;
  const double* yb = (MODEL == MODEL_LINREG) ? y + start : nullptr;
  for (int i = lane; i < n; i += kWarp) sr[i] = 1.0;         // rlvi.py:47,70  pi = 1
  __syncwarp();
  double wl, w;
  int it = 0, status = ST_MAXITER;
  if (!mstep<MODEL>(Xb, yb, n, d, sr, G, bv, th, dl, wl, w)) status = ST_HOST_SOLVE;
  while (status == ST_MAXITER && it < maxiter) {
    for (int j = lane; j < d; j += kWarp) thp[j] = th[j];
    const double scale = 0.5 * w / wl;                       // _estep_scaled: 0.5 / sigma2
    const FpOut r = warp_fixed_point(sr, n, scale, 1e-3, 100);   // update_weights' defaults (rlvi.py:54,77)
    for (int i = lane; i < n; i += kWarp) {
      const double ev = sr[i];
      sr[i] = ev / (r.rho + ev);
    }
    __syncwarp();
    ++it;
    if (!mstep<MODEL>(Xb, yb, n, d, sr, G, bv, th, dl, wl, w)) {
      status = ST_HOST_SOLVE;
      break;
    }
    double num = 0.0, den = 0.0;                             // _rel_change: ||theta - prev|| / ||prev||
    for (int j = lane; j < d; j += kWarp) {
      const double t = th[j] - thp[j];
      num = fma(t, t, num);
      den = fma(thp[j], thp[j], den);
    }
    const double rel = sqrt(warp_sum(num)) / sqrt(warp_sum(den));
    if (rel <= tol) status = ST_CONVERGED;                   // a NaN never stops the loop (_em_loop)
  }
  for (int j = lane; j < d; j += kWarp) out[j] = (status == ST_HOST_SOLVE) ? NAN : th[j];
  if (lane == 0) {
    iters_out[b] = it;
    status_out[b] = status;
  }
}

// ---- logistic regression ---------------------------------------------------------------------------------------------
// rlvi_b200/rlvi.py logistic_regression per problem, with either M-step of the drop-in:
//   LOGREG_NEWTON  utils.sklearn_log_reg: F = 1/2 |theta|^2 + C sum_i w_i CE_i, w = pi / max pi, C = 100, damped Newton
//                  with Armijo backtracking, warm-started from the previous EM iterate; E-step losses softplus(phi)
//   LOGREG_MM      utils.mm_log_reg: theta <- theta - Q^-1 [1,X]^T (pi (sigmoid - y)), Q = 1/4 [1,X]^T Pi [1,X], from 0
//                  while |delta theta| > 1e-2; E-step losses the cross-entropy with y
// D = d + 1 parameters, intercept first; the design is [1, X].  The M-step's matrices are summed one lane per entry over
// the rows in order, its vectors lane-strided plus the xor-shuffle tree, exactly as batched_em_kernel does; every branch
// decision comes from such a warp-uniform value.  Every loop is bounded, so no problem can hold its warp forever.
enum { LOGREG_NEWTON = RLVI_BATCHED_LOGREG_NEWTON, LOGREG_MM = RLVI_BATCHED_LOGREG_MM };

constexpr int kLgMinRows = 1024;                      // the cap admits n = 1024 at every d in 1..63
constexpr int kLgMinWarpDoubles = 4160;               // ... and n = 2008 at d <= 8
constexpr int kLgMaxD = 63;
constexpr double kLgC = 100.0;                        // utils.py:61 reg_coeff, which no caller varies
constexpr int kNewtonMaxSteps = 60;                   // utils.sklearn_log_reg max_newton
constexpr int kArmijoMaxHalvings = 27;                // t = 2^-27 is the first t < 1e-8
constexpr int kMmMaxSteps = 10000;                    // the drop-in's MM loop has no bound; past this one the host solves

// Per-warp shared memory, in doubles: w [cap] (pi, or Newton's pi / max pi) | v [cap] (e, curvature weights, gradient
// coefficients or losses) | M [D][D + 1] | g [D] | theta [D] | theta_prev [D] | step [D] | theta_c [D] | diag(L) [D].
__host__ __device__ inline int lg_fixed_doubles(int d) { return (d + 1) * (d + 2) + 6 * (d + 1); }
__host__ __device__ inline int lg_warp_doubles(int d) {
  const int need = 2 * kLgMinRows + lg_fixed_doubles(d);
  return need > kLgMinWarpDoubles ? need : kLgMinWarpDoubles;
}
__host__ __device__ inline int lg_max_rows(int d) { return (lg_warp_doubles(d) - lg_fixed_doubles(d)) / 2; }

// phi = theta_0 + x . theta_{1..d}, the row arithmetic of loss.cu and of the colsum gradient
__device__ __forceinline__ double lg_phi(const double* xi, const double* th, int d) {
  double a = 0.0;
  for (int k = 0; k < d; ++k) a = fma(xi[k], th[k + 1], a);
  return th[0] + a;
}

__device__ __forceinline__ double lg_sigmoid(double phi) {      // utils.py:7-16, overflow-free
  const double z = exp(-fabs(phi));
  return (phi >= 0.0 ? 1.0 : z) / (1.0 + z);
}

__device__ __forceinline__ double lg_ce(double phi, double yi) {   // loss.cu LOGISTIC_CE, utils.py:21
  return (-yi * phi + phi) + log1p(exp(-phi));
}

__device__ __forceinline__ double lg_dot(const double* a, const double* b, int D) {
  double s = 0.0;
  for (int j = threadIdx.x & 31; j < D; j += kWarp) s = fma(a[j], b[j], s);
  return warp_sum(s);
}

// M[j][k] = diag (j == k) + scale * sum_i v_i xt_ij xt_ik for k <= j < D, xt_i = [1, x_i]: one lane per entry, rows in order.
__device__ void lg_gram(const double* __restrict__ X, int n, int d, const double* v, double scale, double diag, double* M) {
  const int lane = threadIdx.x & 31;
  const int D = d + 1, ld = D + 1, T = D * (D + 1) / 2;
  for (int t = lane; t < T; t += kWarp) {
    int j = int((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
    while (j * (j + 1) / 2 > t) --j;
    while ((j + 1) * (j + 2) / 2 <= t) ++j;
    const int k = t - j * (j + 1) / 2;
    double acc = 0.0;
    for (int i = 0; i < n; ++i) {
      const double* xi = X + int64_t(i) * d;
      const double a = j ? xi[j - 1] : 1.0, b = k ? xi[k - 1] : 1.0;
      acc = fma(v[i] * a, b, acc);
    }
    M[j * ld + k] = (j == k ? diag : 0.0) + scale * acc;
  }
  __syncwarp();
}

// out_j = sum_i v_i xt_ij: one lane per entry, rows in order
__device__ void lg_xtv(const double* __restrict__ X, int n, int d, const double* v, double* out) {
  for (int j = threadIdx.x & 31; j <= d; j += kWarp) {
    double acc = 0.0;
    for (int i = 0; i < n; ++i) acc = fma(v[i], j ? X[int64_t(i) * d + j - 1] : 1.0, acc);
    out[j] = acc;
  }
  __syncwarp();
}

// Left-looking Cholesky of the lower triangle of M in place, diag(L) in dl; false unless every pivot L_jj^2 / M_jj
// exceeds rtol (batched_em_kernel's test; rtol = 0 asks for positive, finite pivots only).
__device__ bool lg_cholesky(double* M, int D, double* dl, double rtol) {
  const int lane = threadIdx.x & 31, ld = D + 1;
  for (int j = 0; j < D; ++j) {
    const double mjj = M[j * ld + j];
    double s = mjj;
    for (int k = 0; k < j; ++k) s = fma(-M[j * ld + k], M[j * ld + k], s);
    const double ljj = sqrt(s);
    if (!(s > 0.0) || !(ljj * ljj / mjj > rtol) || !isfinite(ljj)) return false;   // warp-uniform
    for (int i = j + 1 + lane; i < D; i += kWarp) {
      double t = M[i * ld + j];
      for (int k = 0; k < j; ++k) t = fma(-M[i * ld + k], M[j * ld + k], t);
      M[i * ld + j] = t / ljj;
    }
    if (lane == 0) dl[j] = ljj;
    __syncwarp();
  }
  return true;
}

// L L^T x = b in place (column sweeps)
__device__ void lg_chol_solve(const double* M, int D, const double* dl, double* b) {
  const int lane = threadIdx.x & 31, ld = D + 1;
  for (int k = 0; k < D; ++k) {
    const double zk = b[k] / dl[k];
    __syncwarp();
    for (int i = k + 1 + lane; i < D; i += kWarp) b[i] = fma(-M[i * ld + k], zk, b[i]);
    if (lane == 0) b[k] = zk;
    __syncwarp();
  }
  for (int k = D - 1; k >= 0; --k) {
    const double tk = b[k] / dl[k];
    __syncwarp();
    for (int i = lane; i < k; i += kWarp) b[i] = fma(-M[k * ld + i], tk, b[i]);
    if (lane == 0) b[k] = tk;
    __syncwarp();
  }
}

struct LgWarp {
  const double* X;
  const double* y;
  int n, d;
  double *w, *v, *M, *g, *th, *thp, *st, *tc, *dl;
};

// F(th) = 1/2 |th|^2 + C sum_i w_i CE_i (utils.sklearn_log_reg's objective); leaves e_i = exp(-CE_i) in v.
__device__ double lg_objective(const LgWarp& p, const double* th) {
  double s = 0.0;
  for (int i = threadIdx.x & 31; i < p.n; i += kWarp) {
    const double l = lg_ce(lg_phi(p.X + int64_t(i) * p.d, th, p.d), p.y[i]);
    p.v[i] = exp(-l);
    s = fma(p.w[i], l, s);
  }
  const double wl = warp_sum(s);
  const double F = 0.5 * lg_dot(th, th, p.d + 1) + kLgC * wl;
  __syncwarp();
  return F;
}

// v_i = w_i (sigmoid(phi_i(th)) - y_i), the rows of rlvi_logistic_grad_f64
__device__ void lg_grad_coeffs(const LgWarp& p, const double* th) {
  for (int i = threadIdx.x & 31; i < p.n; i += kWarp)
    p.v[i] = p.w[i] * (lg_sigmoid(lg_phi(p.X + int64_t(i) * p.d, th, p.d)) - p.y[i]);
  __syncwarp();
}

// utils.sklearn_log_reg as the drop-in solves it.  On entry w = pi and th the warm start; on success th is the minimiser
// and v its E-step losses softplus(phi); false when Newton does not converge in 60 steps or its matrix is not finite.
__device__ bool lg_newton(const LgWarp& p) {
  const int lane = threadIdx.x & 31, D = p.d + 1;
  double m = -INFINITY;
  for (int i = lane; i < p.n; i += kWarp) m = fmax(m, p.w[i]);
  m = warp_max(m);
  for (int i = lane; i < p.n; i += kWarp) p.w[i] = p.w[i] / m;              // utils.py:66
  __syncwarp();
  double F = lg_objective(p, p.th);
  bool converged = false;
  for (int it = 0; it < kNewtonMaxSteps && !converged; ++it) {
    for (int i = lane; i < p.n; i += kWarp) {                                // rlvi_irls_weights_f64
      const double s = p.v[i];
      p.v[i] = p.w[i] * s * (1.0 - s);
    }
    __syncwarp();
    lg_gram(p.X, p.n, p.d, p.v, kLgC, 1.0, p.M);                             // I + C [1,X]^T diag(h) [1,X]
    lg_grad_coeffs(p, p.th);
    lg_xtv(p.X, p.n, p.d, p.v, p.g);
    for (int j = lane; j < D; j += kWarp) {
      p.g[j] = p.th[j] + kLgC * p.g[j];                                      // grad = theta + C g
      p.st[j] = p.g[j];
    }
    __syncwarp();
    if (!lg_cholesky(p.M, D, p.dl, 0.0)) return false;
    lg_chol_solve(p.M, D, p.dl, p.st);
    const double slope = lg_dot(p.g, p.st, D);
    const bool small = sqrt(lg_dot(p.st, p.st, D)) <= 1e-9 * (1.0 + sqrt(lg_dot(p.th, p.th, D)));
    double t = 1.0, Fc = F;
    for (int h = 0; h <= kArmijoMaxHalvings; ++h) {
      for (int j = lane; j < D; j += kWarp) p.tc[j] = p.th[j] - t * p.st[j];
      __syncwarp();
      Fc = lg_objective(p, p.tc);
      if (Fc <= F - 1e-4 * t * slope) break;                                 // Armijo
      if (small && Fc <= F + 1e-12 * fabs(F)) break;                         // at the rounding floor of F
      if (t < 1e-8) break;
      t *= 0.5;
    }
    for (int j = lane; j < D; j += kWarp) p.th[j] = p.tc[j];
    __syncwarp();
    F = Fc;
    converged = small && t == 1.0;
  }
  if (!converged) return false;
  for (int i = lane; i < p.n; i += kWarp) {                                  // utils.py:70-71, label-independent
    const double phi = lg_phi(p.X + int64_t(i) * p.d, p.th, p.d);
    p.v[i] = fmax(phi, 0.0) + log1p(exp(-fabs(phi)));
  }
  __syncwarp();
  return true;
}

// utils.mm_log_reg.  On entry w = pi; on success th is the MM iterate the drop-in returns and v its cross-entropy losses;
// false when Q fails the pivot test or the step bound is reached.
__device__ bool lg_mm(const LgWarp& p) {
  const int lane = threadIdx.x & 31, D = p.d + 1;
  lg_gram(p.X, p.n, p.d, p.w, 0.25, 0.0, p.M);                                // utils.py:36-38
  if (!lg_cholesky(p.M, D, p.dl, kEps52 * (double(D) + sqrt(double(p.n))))) return false;
  for (int j = lane; j < D; j += kWarp) p.th[j] = 0.0;                       // utils.py:35
  __syncwarp();
  bool done = false;
  for (int it = 0; it < kMmMaxSteps && !done; ++it) {
    for (int j = lane; j < D; j += kWarp) p.tc[j] = p.th[j];
    __syncwarp();
    lg_grad_coeffs(p, p.tc);
    lg_xtv(p.X, p.n, p.d, p.v, p.st);
    lg_chol_solve(p.M, D, p.dl, p.st);
    double s = 0.0;
    for (int j = lane; j < D; j += kWarp) {
      p.th[j] = p.tc[j] - p.st[j];
      const double t = p.th[j] - p.tc[j];
      s = fma(t, t, s);
    }
    done = !(sqrt(warp_sum(s)) > 1e-2);                                       // utils.py:47; NaN stops too
    __syncwarp();
  }
  if (!done) return false;
  for (int i = lane; i < p.n; i += kWarp)                                     // utils.py:56
    p.v[i] = lg_ce(lg_phi(p.X + int64_t(i) * p.d, p.th, p.d), p.y[i]);
  __syncwarp();
  return true;
}

template <int MSTEP>
__device__ __forceinline__ bool lg_fit(const LgWarp& p) {
  return MSTEP == LOGREG_NEWTON ? lg_newton(p) : lg_mm(p);
}

template <int MSTEP>
__global__ void batched_logreg_kernel(const double* __restrict__ X, const double* __restrict__ y,
                                      const int64_t* __restrict__ offsets, int nprob, int64_t n_rows, int d, double tol,
                                      int maxiter, double* __restrict__ theta_out, int32_t* __restrict__ iters_out,
                                      int32_t* __restrict__ status_out) {
  extern __shared__ double batched_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.x * (blockDim.x >> 5) + warp;
  if (b >= nprob) return;
  const int D = d + 1, cap = lg_max_rows(d);
  LgWarp p;
  p.d = d;
  p.w = batched_smem + size_t(warp) * lg_warp_doubles(d);
  p.v = p.w + cap;
  p.M = p.v + cap;
  p.g = p.M + D * (D + 1);
  p.th = p.g + D;
  p.thp = p.th + D;
  p.st = p.thp + D;
  p.tc = p.st + D;
  p.dl = p.tc + D;
  double* out = theta_out + int64_t(b) * D;
  int64_t start;
  if (!segment(offsets, b, n_rows, cap, start, p.n)) {
    for (int j = lane; j < D; j += kWarp) out[j] = NAN;
    if (lane == 0) {
      iters_out[b] = 0;
      status_out[b] = ST_BAD_SEGMENT;
    }
    return;
  }
  p.X = X + start * d;
  p.y = y + start;
  for (int i = lane; i < p.n; i += kWarp) p.w[i] = 1.0;                      // rlvi.py:97  pi = 1
  for (int j = lane; j < D; j += kWarp) p.th[j] = 0.0;                       // the first Newton fit starts from 0
  __syncwarp();
  int it = 0, status = lg_fit<MSTEP>(p) ? ST_MAXITER : ST_HOST_SOLVE;
  while (status == ST_MAXITER && it < maxiter) {
    const FpOut r = warp_fixed_point(p.v, p.n, 1.0, 1e-3, 100);             // rlvi.py:100, unscaled losses
    for (int i = lane; i < p.n; i += kWarp) {
      const double ev = p.v[i];
      p.w[i] = ev / (r.rho + ev);
    }
    for (int j = lane; j < D; j += kWarp) p.thp[j] = p.th[j];               // also Newton's warm start
    __syncwarp();
    ++it;
    if (!lg_fit<MSTEP>(p)) {
      status = ST_HOST_SOLVE;
      break;
    }
    double num = 0.0, den = 0.0;                                             // _rel_change
    for (int j = lane; j < D; j += kWarp) {
      const double t = p.th[j] - p.thp[j];
      num = fma(t, t, num);
      den = fma(p.thp[j], p.thp[j], den);
    }
    if (sqrt(warp_sum(num)) / sqrt(warp_sum(den)) <= tol) status = ST_CONVERGED;   // a NaN never stops the loop
  }
  for (int j = lane; j < D; j += kWarp) out[j] = (status == ST_HOST_SOLVE) ? NAN : p.th[j];
  if (lane == 0) {
    iters_out[b] = it;
    status_out[b] = status;
  }
}

struct LaunchShape {
  int grid, threads;
  size_t smem;
};

// `wpc` problems per CTA, `per_warp_bytes` of dynamic shared memory each
template <typename K>
int launch_shape(K kernel, int nprob, int wpc, size_t per_warp_bytes, LaunchShape& ls) {
  ls.grid = (nprob + wpc - 1) / wpc;
  ls.threads = wpc * kWarp;
  ls.smem = size_t(wpc) * per_warp_bytes;
  RLVI_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(ls.smem)));
  return RLVI_OK;
}

}  // namespace

extern "C" int rlvi_batched_max_rows(int d) {
  if (d < 1 || d > kMaxD) return 0;
  return max_rows(d);
}

extern "C" int rlvi_batched_fixed_point_f64(rlvi_ctx* ctx, const double* losses, const int64_t* offsets, int nprob,
                                            int64_t n_rows, double tol, int maxiter, double* pi_out,
                                            rlvi_fp_result* results, void* stream) {
  RLVI_REQUIRE(ctx && losses && offsets && pi_out && results, "null pointer");
  RLVI_REQUIRE(nprob >= 1 && n_rows >= 1, "need at least one problem and one row");
  RLVI_REQUIRE(maxiter >= 1, "maxiter must be >= 1");
  RlviDeviceGuard guard(ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int cap = max_rows(1);
  LaunchShape ls;
  const int rc = launch_shape(batched_fp_kernel, nprob, warps_per_cta(size_t(warp_doubles(1)) * sizeof(double)),
                              size_t(cap) * sizeof(double), ls);
  if (rc != RLVI_OK) return rc;
  batched_fp_kernel<<<ls.grid, ls.threads, ls.smem, st>>>(losses, offsets, nprob, n_rows, cap, tol, maxiter, pi_out, results);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}

extern "C" int rlvi_batched_em_f64(rlvi_ctx* ctx, int model, const double* X, const double* y, const int64_t* offsets,
                                   int nprob, int64_t n_rows, int d, double tol, int maxiter, double* theta_out,
                                   int32_t* iters_out, int32_t* status_out, void* stream) {
  RLVI_REQUIRE(ctx && X && offsets && theta_out && iters_out && status_out, "null pointer");
  RLVI_REQUIRE(model == RLVI_BATCHED_MEAN || model == RLVI_BATCHED_LINREG, "model: RLVI_BATCHED_MEAN, RLVI_BATCHED_LINREG");
  RLVI_REQUIRE(model == RLVI_BATCHED_MEAN || y, "RLVI_BATCHED_LINREG needs y");
  RLVI_REQUIRE(nprob >= 1 && n_rows >= 1, "need at least one problem and one row");
  RLVI_REQUIRE(maxiter >= 0, "maxiter must be >= 0");
  if (d < 1 || d > kMaxD) {
    rlvi_set_error("rlvi_batched_em_f64: d = %d outside 1..%d", d, kMaxD);
    return RLVI_ERR_UNSUPPORTED;
  }
  RlviDeviceGuard guard(ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t per_warp = size_t(warp_doubles(d)) * sizeof(double);
  LaunchShape ls;
  int rc;
  if (model == RLVI_BATCHED_MEAN) {
    rc = launch_shape(batched_em_kernel<MODEL_MEAN>, nprob, warps_per_cta(per_warp), per_warp, ls);
    if (rc != RLVI_OK) return rc;
    batched_em_kernel<MODEL_MEAN><<<ls.grid, ls.threads, ls.smem, st>>>(X, nullptr, offsets, nprob, n_rows, d, tol, maxiter,
                                                               theta_out, iters_out, status_out);
  } else {
    rc = launch_shape(batched_em_kernel<MODEL_LINREG>, nprob, warps_per_cta(per_warp), per_warp, ls);
    if (rc != RLVI_OK) return rc;
    batched_em_kernel<MODEL_LINREG><<<ls.grid, ls.threads, ls.smem, st>>>(X, y, offsets, nprob, n_rows, d, tol, maxiter,
                                                                 theta_out, iters_out, status_out);
  }
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}

extern "C" int rlvi_batched_logistic_max_rows(int d) {
  if (d < 1 || d > kLgMaxD) return 0;
  return lg_max_rows(d);
}

extern "C" int rlvi_batched_logistic_f64(rlvi_ctx* ctx, int mstep, const double* X, const double* y,
                                         const int64_t* offsets, int nprob, int64_t n_rows, int d, double tol,
                                         int maxiter, double* theta_out, int32_t* iters_out, int32_t* status_out,
                                         void* stream) {
  RLVI_REQUIRE(ctx && X && y && offsets && theta_out && iters_out && status_out, "null pointer");
  RLVI_REQUIRE(mstep == RLVI_BATCHED_LOGREG_NEWTON || mstep == RLVI_BATCHED_LOGREG_MM,
               "mstep: RLVI_BATCHED_LOGREG_NEWTON, RLVI_BATCHED_LOGREG_MM");
  RLVI_REQUIRE(nprob >= 1 && n_rows >= 1, "need at least one problem and one row");
  RLVI_REQUIRE(maxiter >= 0, "maxiter must be >= 0");
  if (d < 1 || d > kLgMaxD) {
    rlvi_set_error("rlvi_batched_logistic_f64: d = %d outside 1..%d", d, kLgMaxD);
    return RLVI_ERR_UNSUPPORTED;
  }
  RlviDeviceGuard guard(ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t per_warp = size_t(lg_warp_doubles(d)) * sizeof(double);
  LaunchShape ls;
  int rc;
  if (mstep == RLVI_BATCHED_LOGREG_NEWTON) {
    rc = launch_shape(batched_logreg_kernel<LOGREG_NEWTON>, nprob, warps_per_cta(per_warp), per_warp, ls);
    if (rc != RLVI_OK) return rc;
    batched_logreg_kernel<LOGREG_NEWTON><<<ls.grid, ls.threads, ls.smem, st>>>(X, y, offsets, nprob, n_rows, d, tol,
                                                                               maxiter, theta_out, iters_out, status_out);
  } else {
    rc = launch_shape(batched_logreg_kernel<LOGREG_MM>, nprob, warps_per_cta(per_warp), per_warp, ls);
    if (rc != RLVI_OK) return rc;
    batched_logreg_kernel<LOGREG_MM><<<ls.grid, ls.threads, ls.smem, st>>>(X, y, offsets, nprob, n_rows, d, tol, maxiter,
                                                                           theta_out, iters_out, status_out);
  }
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}
