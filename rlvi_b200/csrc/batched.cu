// batched.cu -- many small, independent RLVI problems in one launch: one warp per problem, the whole loop on chip.
//
// Replaces, per problem, the drop-in calls (rlvi_b200/rlvi.py) that the reference's experiment driver makes thousands
// of times on tiny data (standard-learning/main.py: test_mean, test_linear_regression, N = 40..100, d = 2..10):
//   standard-learning/rlvi.py:8-20    update_weights     -> batched_fp_kernel
//   standard-learning/rlvi.py:46-65   mean               -> batched_em_kernel<MODEL_MEAN>
//   standard-learning/rlvi.py:68-89   linear_regression  -> batched_em_kernel<MODEL_LINREG>
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
inline int warps_per_cta(int d) {
  const int w = int(kSmemBudget / (size_t(warp_doubles(d)) * sizeof(double)));
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

struct LaunchShape {
  int grid, threads;
  size_t smem;
};

// warps_per_cta(d) problems per CTA, `per_warp_bytes` of dynamic shared memory each
template <typename K>
int launch_shape(K kernel, int nprob, int d, size_t per_warp_bytes, LaunchShape& ls) {
  const int wpc = warps_per_cta(d);
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
  const int rc = launch_shape(batched_fp_kernel, nprob, 1, size_t(cap) * sizeof(double), ls);
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
    rc = launch_shape(batched_em_kernel<MODEL_MEAN>, nprob, d, per_warp, ls);
    if (rc != RLVI_OK) return rc;
    batched_em_kernel<MODEL_MEAN><<<ls.grid, ls.threads, ls.smem, st>>>(X, nullptr, offsets, nprob, n_rows, d, tol, maxiter,
                                                               theta_out, iters_out, status_out);
  } else {
    rc = launch_shape(batched_em_kernel<MODEL_LINREG>, nprob, d, per_warp, ls);
    if (rc != RLVI_OK) return rc;
    batched_em_kernel<MODEL_LINREG><<<ls.grid, ls.threads, ls.smem, st>>>(X, y, offsets, nprob, n_rows, d, tol, maxiter,
                                                                 theta_out, iters_out, status_out);
  }
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}
