// aux.cu -- small N-sized passes around the hot path (HBM-bound, one launch each):
//   rlvi_sigmoid_f64       standard-learning/utils.py:7-16   overflow-free logistic function of an N-vector
//   rlvi_online_ce_f64     online-learning/main.py:84-85     -t l - (1 - t) l, the label-independent "cross-entropy"
//   rlvi_irls_weights_f64  the Newton / IRLS curvature weights h_i = pi_i s_i (1 - s_i) of the L2-regularised logistic
//                          objective that utils.py:61-73 hands to liblinear (s_i or 1 - s_i = exp(-cross-entropy_i))
//   rlvi_rrm_sum_f64       standard-learning/rrm.py:12-33 and online-learning/main.py:61-81 (update_weights_rrm): the
//                          sum over max(exp(-l_i / alpha), cutoff) that SciPy's Brent evaluates, and the final weights
//   rlvi_sever_pass_f64    standard-learning/sever.py:22-31,95-104: the two per-sample passes of a SEVER filter step
//                          (gradient coefficients c_i, outlier scores tau_i), one projection x_i . u each
#include <math.h>

#include "common.cuh"

namespace {

__global__ void __launch_bounds__(256) sigmoid_kernel(const double* __restrict__ x, int64_t n, double* __restrict__ out) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const double v = x[i];
    const double z = exp(-fabs(v));                       // utils.py:12-15
    out[i] = (v >= 0.0 ? 1.0 : z) / (1.0 + z);
  }
}

__global__ void __launch_bounds__(256) online_ce_kernel(const double* __restrict__ lp, const double* __restrict__ t, int64_t n,
                                                        double* __restrict__ out) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const double ti = t[i], li = lp[i];
    out[i] = __dsub_rn(__dmul_rn(-ti, li), __dmul_rn(1.0 - ti, li));   // main.py:85, term by term (no FMA contraction)
  }
}

__global__ void __launch_bounds__(256) irls_weights_kernel(const double* __restrict__ e, const double* __restrict__ pi,
                                                           int64_t n, double* __restrict__ out) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const double s = e[i];
    out[i] = pi[i] * s * (1.0 - s);
  }
}

__global__ void __launch_bounds__(256) rrm_sum_kernel(const double* __restrict__ losses, int64_t n, double inv_alpha,
                                                      double cutoff, double norm, double* w_out, double* partials,
                                                      unsigned int* ticket, double* out_sum) {
  __shared__ double s_red[8];
  double acc = 0.0;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const double phi = exp(-losses[i] * inv_alpha);       // rrm.py:18,27
    acc += (phi < cutoff) ? cutoff : phi;                 // rrm.py:19,28 (the clipping only enters the sum)
    if (w_out) w_out[i] = phi * norm;                     // rrm.py:32
  }
  double v[1] = {acc};
  block_sum<1>(v, s_red);
  if (grid_total<1>(v, partials, ticket)) out_sum[0] = v[0];
}


// One warp per row (grid-stride over rows), lanes stride over the features with 16-byte loads when the row allows it:
// dot = x_i . u, then
//   op 0  c = alpha (dot - b_i);  out0_i = c;  out1_i = active_i c^2;  out2_i = c != 0 ? 1 / c : 0
//         (sever.py:22 / :95: the per-sample gradient is g_i = c_i x_i; out1, out2 are the weights and the "y" that make ONE
//          statistics pass return sum_active g_i g_i^T and sum_active g_i)
//   op 1  out0_i = active_i ? (a_i dot - m)^2 : -1     (sever.py:29-31: tau_i = ((g_i - mean g) . v)^2, m = mean g . v)
__global__ void __launch_bounds__(256) sever_pass_kernel(const double* __restrict__ X, int64_t n, int d,
                                                         const double* __restrict__ u, int op, double scalar,
                                                         const double* __restrict__ a, const double* __restrict__ b,
                                                         const double* __restrict__ active, double* __restrict__ out0,
                                                         double* __restrict__ out1, double* __restrict__ out2) {
  extern __shared__ double su[];
  for (int j = threadIdx.x; j < d; j += blockDim.x) su[j] = u[j];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = (int64_t(gridDim.x) * blockDim.x) >> 5;
  const bool vec = (d % 2 == 0) && ((reinterpret_cast<uintptr_t>(X) & 15u) == 0u);
  for (int64_t i = warp0; i < n; i += nwarps) {
    const double* row = X + i * d;
    double acc = 0.0;
    if (vec) {
      const double2* r2 = reinterpret_cast<const double2*>(row);
      for (int j = lane; j < d / 2; j += 32) {
        const double2 x = r2[j];
        acc = fma(x.x, su[2 * j], acc);
        acc = fma(x.y, su[2 * j + 1], acc);
      }
    } else {
      for (int j = lane; j < d; j += 32) acc = fma(row[j], su[j], acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      const double act = active ? active[i] : 1.0;
      if (op == 0) {
        const double c = scalar * (acc - (b ? b[i] : 0.0));
        out0[i] = c;
        out1[i] = act * c * c;
        out2[i] = (c != 0.0) ? 1.0 / c : 0.0;
      } else {
        const double t = a[i] * acc - scalar;
        out0[i] = (act != 0.0) ? t * t : -1.0;
      }
    }
  }
}

}  // namespace

extern "C" int rlvi_sigmoid_f64(rlvi_ctx* ctx, const double* x, int64_t n, double* out, void* stream) {
  RLVI_REQUIRE(ctx && x && out, "null pointer");
  RLVI_REQUIRE(n > 0, "n must be positive");
  RlviDeviceGuard guard(ctx->device);
  sigmoid_kernel<<<grid_for(ctx, n, 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, n, out);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}

extern "C" int rlvi_online_ce_f64(rlvi_ctx* ctx, const double* log_proba, const double* targets, int64_t n, double* out,
                                  void* stream) {
  RLVI_REQUIRE(ctx && log_proba && targets && out, "null pointer");
  RLVI_REQUIRE(n > 0, "n must be positive");
  RlviDeviceGuard guard(ctx->device);
  online_ce_kernel<<<grid_for(ctx, n, 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(log_proba, targets, n, out);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}

extern "C" int rlvi_irls_weights_f64(rlvi_ctx* ctx, const double* e, const double* weights, int64_t n, double* out,
                                     void* stream) {
  RLVI_REQUIRE(ctx && e && weights && out, "null pointer");
  RLVI_REQUIRE(n > 0, "n must be positive");
  RlviDeviceGuard guard(ctx->device);
  irls_weights_kernel<<<grid_for(ctx, n, 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(e, weights, n, out);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}

extern "C" int rlvi_rrm_sum_f64(rlvi_ctx* ctx, const double* losses, int64_t n, double inv_alpha, double cutoff,
                                double norm, double* w_out, double* out_sum, void* stream) {
  RLVI_REQUIRE(ctx && losses && out_sum, "null pointer");
  RLVI_REQUIRE(n > 0, "n must be positive");
  RlviDeviceGuard guard(ctx->device);
  const int grid = grid_for(ctx, n, 4);
  RlviScratch s;
  const int rc = rlvi_scratch_header(ctx, size_t(grid) * sizeof(double), &s);
  if (rc != RLVI_OK) return rc;
  rrm_sum_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(losses, n, inv_alpha, cutoff, norm, w_out,
                                                                      s.partials, s.ticket, out_sum);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}

extern "C" int rlvi_sever_pass_f64(rlvi_ctx* ctx, const double* X, int64_t n, int d, const double* u, int op, double scalar,
                                   const double* a, const double* b, const double* active, double* out0, double* out1,
                                   double* out2, void* stream) {
  RLVI_REQUIRE(ctx && X && u && out0, "null pointer");
  RLVI_REQUIRE(n > 0 && d > 0 && d <= 4096, "n must be positive and 0 < d <= 4096");
  RLVI_REQUIRE(op == 0 || op == 1, "op must be 0 (gradient coefficients) or 1 (scores)");
  RLVI_REQUIRE(op == 1 || (out1 && out2), "op 0 writes three arrays");
  RLVI_REQUIRE(op == 0 || a, "op 1 needs the coefficients a");
  RlviDeviceGuard guard(ctx->device);
  int64_t want = (n + 7) / 8;                                   // 8 warps per block, one row per warp and trip
  const int64_t cap = int64_t(ctx->sm_count) * 8;
  const int grid = int(want < 1 ? 1 : (want > cap ? cap : want));
  sever_pass_kernel<<<grid, 256, size_t(d) * sizeof(double), static_cast<cudaStream_t>(stream)>>>(X, n, d, u, op, scalar, a, b,
                                                                                             active, out0, out1, out2);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}
