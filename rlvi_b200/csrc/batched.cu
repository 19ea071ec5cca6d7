// batched.cu -- many small, independent RLVI problems in one launch: one warp per problem, the whole loop on chip.
//
// Replaces, per problem, the drop-in calls (rlvi_b200/rlvi.py) that the reference's experiment driver makes thousands
// of times on tiny data (standard-learning/main.py: test_mean, test_linear_regression, N = 40..100, d = 2..10):
//   standard-learning/rlvi.py:8-20    update_weights     -> batched_fp_kernel
//   standard-learning/rlvi.py:46-65   mean               -> batched_em_kernel<MODEL_MEAN>
//   standard-learning/rlvi.py:68-89   linear_regression  -> batched_em_kernel<MODEL_LINREG>
//   standard-learning/rlvi.py:92-108  logistic_regression -> batched_em_kernel<LOGREG_NEWTON / LOGREG_MM>
// At that size a drop-in EM iteration is ~10 launches and two host synchronisations; here a problem's EM loop, its
// fixed points, the D x D Cholesky and the stop tests run inside one warp, with no host round trip.  The EM loop is
// written once; a model supplies its M-step and its shared-memory layout.
//
// Layout: problem b owns rows [offsets[b], offsets[b+1]) of X [rows][d], y, losses and pi.  Each warp keeps in shared
// memory the per-row vectors pi and losses (one vector for mean and linear regression: r^2 after an M-step,
// e = exp(-scale r^2) during the fixed point and pi after it; two for logistic regression, whose M-steps need pi while
// they overwrite the losses), the lower triangle of the M-step's matrix with its Cholesky factor, and a few D-vectors.
// X and y are read from global memory by every pass over the rows; e is read by every fixed-point pass.
//
// Determinism: a problem's bits depend only on its own rows.  Every sum runs in an order fixed relative to the problem's
// first row -- lane-strided partial sums plus the xor-shuffle tree, or one lane summing over the rows in order -- so neither
// the problem's index, the batch size nor the warp that runs it changes anything.  No atomics.
#include <math.h>

#include "common.cuh"

namespace {

constexpr int kMaxD = 64;                             // mean and linear regression
constexpr int kLgMaxD = 63;                           // logistic regression: D = d + 1 <= 64
constexpr int kMinRows = 1024;                        // the cap admits n = 1024 at every supported d
constexpr int kMaxWarpsPerCta = 16;
constexpr size_t kSmemBudget = size_t(220) * 1024;    // dynamic shared memory of one CTA
constexpr double kEps52 = 2.220446049250313e-16;      // torch.finfo(float64).eps

// The kernels' models.  The ABI's RLVI_BATCHED_* values number the models of each entry point from 0, so they cannot
// tell all four apart.
enum { MODEL_MEAN, MODEL_LINREG, LOGREG_NEWTON, LOGREG_MM };
enum { ST_CONVERGED = 0, ST_MAXITER = 1, ST_HOST_SOLVE = 2, ST_BAD_SEGMENT = -1 };

// Per-warp shared memory, in doubles: `bufs` per-row vectors of cap doubles | M [D][D + 1] (odd row stride: the column
// sweeps of the Cholesky hit distinct banks) | `vecs` D-vectors.  At small d the share is raised to `min_doubles`, and
// the rows take what the rest leaves.
struct Layout {
  int bufs, vecs, D, min_doubles;
};
__host__ __device__ inline Layout layout(int model, int d) {
  if (model == LOGREG_NEWTON || model == LOGREG_MM)
    return Layout{2, 6, d + 1, 4160};                 // pi, losses | M | g, theta, theta_prev, diag(L), step, trial;
                                                      // 32.5 KiB: n = 2008 at d <= 8
  return Layout{1, 4, d, 1536};                       // pi / r^2 | G | b, theta, theta_prev, diag(L); at least 12 KiB
}
__host__ __device__ inline int fixed_doubles(const Layout& L) { return L.D * (L.D + 1) + L.vecs * L.D; }
__host__ __device__ inline int warp_doubles(const Layout& L) {
  const int need = L.bufs * kMinRows + fixed_doubles(L);
  return need > L.min_doubles ? need : L.min_doubles;
}
__host__ __device__ inline int max_rows(const Layout& L) { return (warp_doubles(L) - fixed_doubles(L)) / L.bufs; }
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

// ---- the models' M-steps --------------------------------------------------------------------------------------------
// One problem's view of its warp: w holds pi; v the per-row losses, e during the fixed point, and the logistic M-steps'
// working rows (curvature weights, gradient coefficients); M the lower triangle of the M-step's D x D matrix and then its
// Cholesky factor, dl = diag(L); g the right-hand side; th theta and thp the previous theta; st and tc the logistic
// M-steps' step and trial point.
struct Warp {
  const double* X;
  const double* y;
  int n, d;
  double *w, *v, *M, *g, *th, *thp, *dl, *st, *tc;
};

// Column j of the design at row xi: [1, x_i] with the intercept, x_i without.
template <bool ICPT>
__device__ __forceinline__ double design(const double* xi, int j) {
  return ICPT ? (j ? xi[j - 1] : 1.0) : xi[j];
}

// M[j][k] = diag [j == k] + scale sum_i v_i xt_ij xt_ik for k <= j < D: one lane per entry, rows in order.  With y (the
// normal equations of linear regression), b_j = sum_i (v_i xt_ij) y_i takes D more entries of the same sweep and M keeps
// the raw sums (0.0 + 1.0 sum would turn a -0.0 sum into +0.0).
template <bool ICPT>
__device__ void gram(const double* __restrict__ X, int n, int d, const double* v, double scale, double diag, double* M,
                     const double* __restrict__ y = nullptr, double* b = nullptr) {
  const int lane = threadIdx.x & 31;
  const int D = d + ICPT, ld = D + 1, T = D * (D + 1) / 2;
  for (int t = lane; t < T + (y ? D : 0); t += kWarp) {
    int j, k = -1;
    if (t < T) {
      j = int((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
      while (j * (j + 1) / 2 > t) --j;
      while ((j + 1) * (j + 2) / 2 <= t) ++j;
      k = t - j * (j + 1) / 2;
    } else {
      j = t - T;
    }
    double acc = 0.0;
    if (k >= 0) {                        // two row loops: a select of y inside one would halve the loop's unrolling
      for (int i = 0; i < n; ++i) {
        const double* xi = X + int64_t(i) * d;
        acc = fma(v[i] * design<ICPT>(xi, j), design<ICPT>(xi, k), acc);
      }
      M[j * ld + k] = y ? acc : (j == k ? diag : 0.0) + scale * acc;
    } else {
      for (int i = 0; i < n; ++i) acc = fma(v[i] * design<ICPT>(X + int64_t(i) * d, j), y[i], acc);
      b[j] = acc;
    }
  }
  __syncwarp();
}

// out_j = sum_i v_i xt_ij: one lane per entry, rows in order
template <bool ICPT>
__device__ void xtv(const double* __restrict__ X, int n, int d, const double* v, double* out) {
  for (int j = threadIdx.x & 31; j < d + ICPT; j += kWarp) {
    double acc = 0.0;
    for (int i = 0; i < n; ++i) acc = fma(v[i], design<ICPT>(X + int64_t(i) * d, j), acc);
    out[j] = acc;
  }
  __syncwarp();
}

// Left-looking Cholesky of the lower triangle of M in place, one column per step, diag(L) in dl; false unless every pivot
// L_jj^2 / M_jj exceeds rtol (rlvi.py's _gpu_sym_solve: torch.linalg.cholesky_ex info == 0 and min(diag(L)^2 / diag(M))
// > rtol; rtol = 0 asks for positive, finite pivots only).
__device__ bool cholesky(double* M, int D, double* dl, double rtol) {
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
__device__ void chol_solve(const double* M, int D, const double* dl, double* b) {
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

// Mean and linear regression, with v aliasing w: on return v holds r^2 and scale = 0.5 sum pi / sum pi r^2 (_estep_scaled's
// 0.5 / sigma2, from the weighted sums the drop-in's loss pass returns: rlvi_loss_f64, wsum_out).  False when LINREG's
// normal equations fail the pivot test of _gpu_sym_solve (the problem then needs the host's minimum-norm solve).
template <int MODEL>
__device__ bool lsq_mstep(const Warp& p, double& scale) {
  const int lane = threadIdx.x & 31, d = p.d;
  if (MODEL == MODEL_MEAN) {
    double s0 = 0.0;
    for (int i = lane; i < p.n; i += kWarp) s0 += p.w[i];
    s0 = warp_sum(s0);
    xtv<false>(p.X, p.n, d, p.w, p.th);                      // S1 = X^T pi
    for (int j = lane; j < d; j += kWarp) p.th[j] /= s0;     // rlvi.py:48,56
  } else {
    gram<false>(p.X, p.n, d, p.w, 1.0, 0.0, p.M, p.y, p.g);  // G = X^T Pi X, b = X^T Pi y
    if (!cholesky(p.M, d, p.dl, kEps52 * (double(d) + sqrt(double(p.n))))) return false;
    chol_solve(p.M, d, p.dl, p.g);
    for (int j = lane; j < d; j += kWarp) p.th[j] = p.g[j];
  }
  __syncwarp();
  // per-row loss (rlvi_loss_f64's SQDIST / SQRES arithmetic) and the weighted sums; r^2 replaces pi in place
  double a0 = 0.0, a1 = 0.0;
  for (int i = lane; i < p.n; i += kWarp) {
    const double* xi = p.X + int64_t(i) * d;
    double a = 0.0, l;
    if (MODEL == MODEL_MEAN) {
      for (int k = 0; k < d; ++k) {
        const double t = p.th[k] - xi[k];
        a = fma(t, t, a);
      }
      const double r = sqrt(a);                              // rlvi.py:49,57  np.linalg.norm(theta - x)**2
      l = r * r;
    } else {
      for (int k = 0; k < d; ++k) a = fma(xi[k], p.th[k], a);
      const double r = p.y[i] - a;                           // rlvi.py:72,81
      l = r * r;
    }
    const double pi = p.w[i];
    a0 = fma(pi, l, a0);
    a1 += pi;
    p.v[i] = l;
  }
  const double wl = warp_sum(a0), w = warp_sum(a1);
  scale = 0.5 * w / wl;
  __syncwarp();
  return true;
}

// ---- logistic regression ---------------------------------------------------------------------------------------------
// rlvi_b200/rlvi.py logistic_regression per problem, with either M-step of the drop-in:
//   LOGREG_NEWTON  utils.sklearn_log_reg: F = 1/2 |theta|^2 + C sum_i w_i CE_i, w = pi / max pi, C = 100, damped Newton
//                  with Armijo backtracking, warm-started from the previous EM iterate; E-step losses softplus(phi)
//   LOGREG_MM      utils.mm_log_reg: theta <- theta - Q^-1 [1,X]^T (pi (sigmoid - y)), Q = 1/4 [1,X]^T Pi [1,X], from 0
//                  while |delta theta| > 1e-2; E-step losses the cross-entropy with y
// D = d + 1 parameters, intercept first; the design is [1, X].  Every branch decision comes from a warp-uniform value, and
// every loop is bounded, so no problem can hold its warp forever.
constexpr double kLgC = 100.0;                        // utils.py:61 reg_coeff, which no caller varies
constexpr int kNewtonMaxSteps = 60;                   // utils.sklearn_log_reg max_newton
constexpr int kArmijoMaxHalvings = 27;                // t = 2^-27 is the first t < 1e-8
constexpr int kMmMaxSteps = 10000;                    // the drop-in's MM loop has no bound; past this one the host solves

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

// F(th) = 1/2 |th|^2 + C sum_i w_i CE_i (utils.sklearn_log_reg's objective); leaves e_i = exp(-CE_i) in v.
__device__ double lg_objective(const Warp& p, const double* th) {
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
__device__ void lg_grad_coeffs(const Warp& p, const double* th) {
  for (int i = threadIdx.x & 31; i < p.n; i += kWarp)
    p.v[i] = p.w[i] * (lg_sigmoid(lg_phi(p.X + int64_t(i) * p.d, th, p.d)) - p.y[i]);
  __syncwarp();
}

// utils.sklearn_log_reg as the drop-in solves it.  On entry w = pi and th the warm start; on success th is the minimiser
// and v its E-step losses softplus(phi); false when Newton does not converge in 60 steps or its matrix is not finite.
__device__ bool lg_newton(const Warp& p) {
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
    gram<true>(p.X, p.n, p.d, p.v, kLgC, 1.0, p.M);                          // I + C [1,X]^T diag(h) [1,X]
    lg_grad_coeffs(p, p.th);
    xtv<true>(p.X, p.n, p.d, p.v, p.g);
    for (int j = lane; j < D; j += kWarp) {
      p.g[j] = p.th[j] + kLgC * p.g[j];                                      // grad = theta + C g
      p.st[j] = p.g[j];
    }
    __syncwarp();
    if (!cholesky(p.M, D, p.dl, 0.0)) return false;
    chol_solve(p.M, D, p.dl, p.st);
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
__device__ bool lg_mm(const Warp& p) {
  const int lane = threadIdx.x & 31, D = p.d + 1;
  gram<true>(p.X, p.n, p.d, p.w, 0.25, 0.0, p.M);                            // utils.py:36-38
  if (!cholesky(p.M, D, p.dl, kEps52 * (double(D) + sqrt(double(p.n))))) return false;
  for (int j = lane; j < D; j += kWarp) p.th[j] = 0.0;                       // utils.py:35
  __syncwarp();
  bool done = false;
  for (int it = 0; it < kMmMaxSteps && !done; ++it) {
    for (int j = lane; j < D; j += kWarp) p.tc[j] = p.th[j];
    __syncwarp();
    lg_grad_coeffs(p, p.tc);
    xtv<true>(p.X, p.n, p.d, p.v, p.st);
    chol_solve(p.M, D, p.dl, p.st);
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

// ---- the EM driver ---------------------------------------------------------------------------------------------------
// M-step contract: on entry w holds pi and th the previous theta (Newton's warm start); on success th holds theta, v the
// per-row losses and `scale` the next E-step's loss scale.  False sends the problem to the host (status 2).
template <int MODEL>
__device__ __forceinline__ bool mstep(const Warp& p, double& scale) {
  if constexpr (MODEL == MODEL_MEAN || MODEL == MODEL_LINREG) {
    return lsq_mstep<MODEL>(p, scale);
  } else {
    scale = 1.0;                                             // rlvi.py:100, unscaled losses
    return MODEL == LOGREG_NEWTON ? lg_newton(p) : lg_mm(p);
  }
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
  const Layout L = layout(MODEL, d);
  const int D = L.D, cap = max_rows(L);
  Warp p;
  p.d = d;
  p.w = batched_smem + size_t(warp) * warp_doubles(L);
  p.v = L.bufs == 2 ? p.w + cap : p.w;
  p.M = p.w + L.bufs * cap;
  p.g = p.M + D * (D + 1);
  p.th = p.g + D;
  p.thp = p.th + D;
  p.dl = p.thp + D;
  p.st = p.dl + D;
  p.tc = p.st + D;
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
  p.y = MODEL == MODEL_MEAN ? nullptr : y + start;
  for (int i = lane; i < p.n; i += kWarp) p.w[i] = 1.0;                      // rlvi.py:47,70,97  pi = 1
  for (int j = lane; j < D; j += kWarp) p.th[j] = 0.0;                       // the first Newton fit starts from 0
  __syncwarp();
  double scale;
  int it = 0, status = mstep<MODEL>(p, scale) ? ST_MAXITER : ST_HOST_SOLVE;
  while (status == ST_MAXITER && it < maxiter) {
    const FpOut r = warp_fixed_point(p.v, p.n, scale, 1e-3, 100);           // update_weights' defaults (rlvi.py:54,77,100)
    for (int i = lane; i < p.n; i += kWarp) {
      const double ev = p.v[i];
      p.w[i] = ev / (r.rho + ev);
    }
    for (int j = lane; j < D; j += kWarp) p.thp[j] = p.th[j];
    __syncwarp();
    ++it;
    if (!mstep<MODEL>(p, scale)) {
      status = ST_HOST_SOLVE;
      break;
    }
    double num = 0.0, den = 0.0;                                             // _rel_change: ||theta - prev|| / ||prev||
    for (int j = lane; j < D; j += kWarp) {
      const double t = p.th[j] - p.thp[j];
      num = fma(t, t, num);
      den = fma(p.thp[j], p.thp[j], den);
    }
    if (sqrt(warp_sum(num)) / sqrt(warp_sum(den)) <= tol) status = ST_CONVERGED;   // a NaN never stops the loop (_em_loop)
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

// One launch of batched_em_kernel<MODEL>: the entry points have checked the arguments.
template <int MODEL>
int run_em(rlvi_ctx* ctx, const double* X, const double* y, const int64_t* offsets, int nprob, int64_t n_rows, int d,
           double tol, int maxiter, double* theta_out, int32_t* iters_out, int32_t* status_out, void* stream) {
  RlviDeviceGuard guard(ctx->device);
  const size_t per_warp = size_t(warp_doubles(layout(MODEL, d))) * sizeof(double);
  LaunchShape ls;
  const int rc = launch_shape(batched_em_kernel<MODEL>, nprob, warps_per_cta(per_warp), per_warp, ls);
  if (rc != RLVI_OK) return rc;
  batched_em_kernel<MODEL><<<ls.grid, ls.threads, ls.smem, static_cast<cudaStream_t>(stream)>>>(
      X, y, offsets, nprob, n_rows, d, tol, maxiter, theta_out, iters_out, status_out);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}

}  // namespace

extern "C" int rlvi_batched_max_rows(int d) {
  if (d < 1 || d > kMaxD) return 0;
  return max_rows(layout(MODEL_MEAN, d));
}

extern "C" int rlvi_batched_fixed_point_f64(rlvi_ctx* ctx, const double* losses, const int64_t* offsets, int nprob,
                                            int64_t n_rows, double tol, int maxiter, double* pi_out,
                                            rlvi_fp_result* results, void* stream) {
  RLVI_REQUIRE(ctx && losses && offsets && pi_out && results, "null pointer");
  RLVI_REQUIRE(nprob >= 1 && n_rows >= 1, "need at least one problem and one row");
  RLVI_REQUIRE(maxiter >= 1, "maxiter must be >= 1");
  RlviDeviceGuard guard(ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const Layout L = layout(MODEL_MEAN, 1);
  const int cap = max_rows(L);
  LaunchShape ls;
  const int rc = launch_shape(batched_fp_kernel, nprob, warps_per_cta(size_t(warp_doubles(L)) * sizeof(double)),
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
  const auto run = model == RLVI_BATCHED_MEAN ? run_em<MODEL_MEAN> : run_em<MODEL_LINREG>;
  return run(ctx, X, y, offsets, nprob, n_rows, d, tol, maxiter, theta_out, iters_out, status_out, stream);
}

extern "C" int rlvi_batched_logistic_max_rows(int d) {
  if (d < 1 || d > kLgMaxD) return 0;
  return max_rows(layout(LOGREG_NEWTON, d));
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
  const auto run = mstep == RLVI_BATCHED_LOGREG_NEWTON ? run_em<LOGREG_NEWTON> : run_em<LOGREG_MM>;
  return run(ctx, X, y, offsets, nprob, n_rows, d, tol, maxiter, theta_out, iters_out, status_out, stream);
}
