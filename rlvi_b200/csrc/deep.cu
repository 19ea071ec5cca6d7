// deep.cu -- the deep-learning RLVI pieces in FP32.
//
//   rlvi_wce_fwd_bwd_f32   deep-learning/methods/train_rlvi.py:89-94 + the autograd backward of line 96
//                          (and utils.py:65-79 `accuracy`, called at train_rlvi.py:85) in ONE launch
//                          instead of ~12 ATen kernels (SURVEY.md section 2a).
//   rlvi_fn_threshold_f32  train_rlvi.py:41-49 (false_negative_criterion) + :102-103 (truncation)
//                          as one single-CTA bisection select instead of sort + cumsum + compare + index.
#include <math.h>

#include "common.cuh"

namespace {

constexpr int kWceThreads = 256;

struct WceParams {
  const float* logits;
  const int64_t* labels;
  const int64_t* indexes;
  const float* weights;
  float* residuals;
  float* per_sample;
  float* dlogits;
  float* out_loss;
  int32_t* out_correct;
  int64_t batch;
  int classes;
  int64_t n_train;
  double* partials;
  unsigned int* ticket;
};

// One warp per row; NV logits per lane held in registers (classes <= 32 * NV).
template <int NV>
__global__ void __launch_bounds__(kWceThreads) wce_kernel(const WceParams p) {
  __shared__ double s_red[kWceThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int C = p.classes;
  const float inv_b = 1.0f / float(p.batch);
  double wl_sum = 0.0;   // sum_i loss_i * w_i over this warp's rows (lane 0)
  int top1 = 0, top5 = 0;
  for (int64_t row = int64_t(blockIdx.x) * nwarp + warp; row < p.batch; row += int64_t(gridDim.x) * nwarp) {
    const float* x = p.logits + row * C;
    float v[NV];
    float m = -INFINITY;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int c = lane + 32 * k;
      v[k] = (c < C) ? __ldg(x + c) : -INFINITY;
      m = fmaxf(m, v[k]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int c = lane + 32 * k;
      if (c < C) s += expf(v[k] - m);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float logs = logf(s);
    const int64_t label = p.labels[row];
    const int64_t idx = p.indexes ? p.indexes[row] : row;
    // A label outside [0, C) or an index outside [0, n_train) raises IndexError / a device assert in the reference.
    // An asynchronous kernel cannot raise: it never reads or writes out of bounds and POISONS the row instead -- NaN
    // loss, NaN gradient row, NaN batch loss -- so the error is loud at the first host read of the loss.
    const bool valid = label >= 0 && label < C && idx >= 0 && idx < p.n_train;
    const float xl = valid ? __ldg(x + label) : __int_as_float(0x7fc00000);
    const float loss = -((xl - m) - logs);                 // -log_softmax[label]
    const float w = valid ? p.weights[idx] : __int_as_float(0x7fc00000);
    if (lane == 0) {
      if (valid) p.residuals[idx] = loss;                          // line 90, detached (quirk Q8)
      if (p.per_sample) p.per_sample[row] = loss;
      wl_sum += double(loss * w);                                  // line 93: loss * batch_weights in FP32
    }
    if (p.dlogits) {
      const float gsc = w * inv_b;                                 // d mean / d loss_i, times pi_i
      float* dx = p.dlogits + row * C;
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        const int c = lane + 32 * k;
        if (c < C) {
          float d = expf((v[k] - m) - logs) * gsc;
          if (c == label) d -= gsc;
          dx[c] = d;
        }
      }
    }
    if (p.out_correct) {
      // rank of the label among the logits (ties: lower class index first)
      int rank = 0;
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        const int c = lane + 32 * k;
        if (c < C && (v[k] > xl || (v[k] == xl && c < label))) ++rank;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) rank += __shfl_xor_sync(0xffffffffu, rank, o);
      if (lane == 0) {
        top1 += (rank < 1);
        top5 += (rank < 5);
      }
    }
  }
  if (p.out_correct && lane == 0 && (top1 | top5)) {
    atomicAdd(p.out_correct, top1);        // integer atomics: order-independent
    atomicAdd(p.out_correct + 1, top5);
  }
  // block partial of the weighted loss: warps in order
  if (lane == 0) s_red[warp] = wl_sum;
  __syncthreads();
  double v[1] = {0.0};
  if (threadIdx.x == 0) {
    for (int w = 0; w < nwarp; ++w) v[0] += s_red[w];
  }
  if (grid_total<1>(v, p.partials, p.ticket)) p.out_loss[0] = float(v[0] / double(p.batch));   // .mean() (line 94)
}

// ---------------------------------------------------------------------------------------------
// false-negative threshold (train_rlvi.py:41-49): selection by bisection over the FP32 bit patterns.
//
// With the weights sorted descending, c_j = sum_{i<=j} (1 - w_(i)) and J = #{j : c_j <= beta}; the threshold
// is w_(J) (J = 0 wraps to the smallest weight, quirk Q9).  M(tau) = sum_{w >= tau} (1 - w) is non-increasing
// in tau, so tau* = min{tau : M(tau) <= beta} is found with <= 33 passes over the weights (cached in shared
// memory), each one contention-free block reduction of a 64-bit fixed-point mass (2^-40 units: exact, order
// independent).  Then P = #{w >= tau*}, and of the next lower weight value kappa (mass u each)
// t = floor((beta - M(tau*)) / u) more elements fit:  J = P + t.
// (A first version histogrammed 8-bit digits with shared-memory atomics: the weights of clean samples pile
// into one or two bins and the atomics serialised, ~1 ms for 45 000 weights.)
// ---------------------------------------------------------------------------------------------
constexpr int kThrThreads = 1024;
constexpr double kFix = 1099511627776.0;   // 2^40

__device__ __forceinline__ unsigned long long mass_of(float w) {
  const float u = 1.0f - w;                      // the FP32 value torch forms (line 46)
  return u > 0.f ? (unsigned long long)__double2ll_rn(double(u) * kFix) : 0ull;
}

struct ThrRed {
  unsigned long long m[2][kThrThreads / 32];
  unsigned int c[2][kThrThreads / 32];
};

// block-wide sums of a 64-bit mass and a 32-bit count; every thread gets both totals; one __syncthreads
__device__ __forceinline__ void thr_allreduce(ThrRed& red, unsigned long long& m, unsigned int& c, unsigned int& round) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned int b = round & 1u;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    m += __shfl_xor_sync(0xffffffffu, m, o);
    c += __shfl_xor_sync(0xffffffffu, c, o);
  }
  if (lane == 0) {
    red.m[b][warp] = m;
    red.c[b][warp] = c;
  }
  __syncthreads();
  m = red.m[b][lane];
  c = red.c[b][lane];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    m += __shfl_xor_sync(0xffffffffu, m, o);
    c += __shfl_xor_sync(0xffffffffu, c, o);
  }
  round += 1u;
}
__device__ __forceinline__ unsigned int thr_allmin(ThrRed& red, unsigned int v, unsigned int& round, bool want_max) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned int b = round & 1u;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned int t = __shfl_xor_sync(0xffffffffu, v, o);
    v = want_max ? max(v, t) : min(v, t);
  }
  if (lane == 0) red.c[b][warp] = v;
  __syncthreads();
  v = red.c[b][lane];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned int t = __shfl_xor_sync(0xffffffffu, v, o);
    v = want_max ? max(v, t) : min(v, t);
  }
  round += 1u;
  return v;
}

template <bool CACHED>
__global__ void __launch_bounds__(kThrThreads, 1) fn_threshold_kernel(float* weights, int64_t n, float alpha,
                                                                      float prev_threshold, int truncate,
                                                                      float* out_threshold) {
  extern __shared__ __align__(16) unsigned char thr_smem[];
  __shared__ ThrRed red;
  unsigned int* skeys = reinterpret_cast<unsigned int*>(thr_smem);
  const unsigned int* keys = CACHED ? skeys : reinterpret_cast<const unsigned int*>(weights);
  const int tid = threadIdx.x;
  unsigned int round = 0;
  // ---- pass 0: cache the keys, total mass, smallest key
  unsigned long long tm = 0ull;
  unsigned int kmin = 0xffffffffu, cnt0 = 0u;
  for (int64_t i = tid; i < n; i += kThrThreads) {
    const float w = weights[i];
    if (CACHED) skeys[i] = __float_as_uint(w);
    tm += mass_of(w);
    kmin = min(kmin, __float_as_uint(w));
  }
  thr_allreduce(red, tm, cnt0, round);                    // also orders the key cache (its __syncthreads)
  const unsigned int key_min = thr_allmin(red, kmin, round, false);
  const float total = float(double(tm) / kFix);           // torch.sum(1 - weights): FP32 scalar
  const float beta = total * alpha;                       // line 44
  const unsigned long long beta_fix = (unsigned long long)(double(beta) * kFix);

  unsigned int result_key;
  if (tm <= beta_fix) {
    result_key = key_min;                                 // everything fits: index n-1 -> the smallest weight
  } else {
    // ---- largest tau_f with M(tau_f) > beta, bit by bit; tau* = tau_f + 1   (M(0) = total > beta here)
    unsigned int cur = 0u;
    for (int bit = 31; bit >= 0; --bit) {
      const unsigned int cand = cur | (1u << bit);
      unsigned long long m = 0ull;
      unsigned int c = 0u;
      for (int64_t i = tid; i < n; i += kThrThreads) {
        const unsigned int k = keys[i];
        if (k >= cand) m += mass_of(__uint_as_float(k));
      }
      thr_allreduce(red, m, c, round);
      if (m > beta_fix) cur = cand;
    }
    // cur = tau_f is an actual key (the largest key whose "keys >= it" mass exceeds beta) = kappa
    const unsigned int kappa = cur;
    unsigned long long m_hi = 0ull;
    unsigned int p_hi = 0u, c_kappa = 0u, key_hi = 0xffffffffu;
    for (int64_t i = tid; i < n; i += kThrThreads) {
      const unsigned int k = keys[i];
      if (k > kappa) {
        m_hi += mass_of(__uint_as_float(k));
        ++p_hi;
        key_hi = min(key_hi, k);
      }
    }
    thr_allreduce(red, m_hi, p_hi, round);
    key_hi = thr_allmin(red, key_hi, round, false);
    const unsigned long long u = mass_of(__uint_as_float(kappa));     // > 0: else M(kappa) = M(kappa+1) <= beta
    const unsigned long long t = (beta_fix - m_hi) / (u ? u : 1ull);  // elements of value kappa that still fit
    (void)c_kappa;
    if (t >= 1ull) result_key = kappa;
    else if (p_hi >= 1u) result_key = key_hi;
    else result_key = key_min;                            // nothing fits: index -1 wraps (quirk Q9)
  }
  const float thr = fmaxf(prev_threshold, __uint_as_float(result_key));   // line 102
  if (tid == 0) out_threshold[0] = thr;
  if (truncate) {
    for (int64_t i = tid; i < n; i += kThrThreads) {
      if (weights[i] < thr) weights[i] = 0.f;                // line 103
    }
  }
}

// ---------------------------------------------------------------------------------------------
// KKT shift objective (standard-learning/rlvi.py:34-42)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) shift_sum_kernel(const double* __restrict__ losses, int64_t n, double shift,
                                                        double c, double* pi_out, double* partials,
                                                        unsigned int* ticket, double* out_sum) {
  __shared__ double s_red[8];
  double acc = 0.0;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const double t = exp(-losses[i] + shift);
    const double r = t / (c + t);
    acc += r;
    if (pi_out) pi_out[i] = r;
  }
  double v[1] = {acc};
  block_sum<1>(v, s_red);
  if (grid_total<1>(v, partials, ticket)) out_sum[0] = v[0];
}

// Same objective from the precomputed e_i = exp(-l_i) the fixed point leaves behind:  t_i = e_i * exp(shift).
// One reciprocal instead of an exp + a division per sample: the Brent search of rlvi.py:41 evaluates this
// 12-21 times per E-step, each a full pass (HBM-bound here, FP64-bound with the exp).
__device__ __forceinline__ double shift_rcp(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  const double d = fma(-x, r, 1.0);      // r (1 + d + d^2): see rcp_fast in fixed_point.cu
  const double s = fma(d, d, d);
  return fma(r, s, r);
}
__global__ void __launch_bounds__(256) shift_sum_e_kernel(const double* __restrict__ e, int64_t n, double scale_t,
                                                          double c, double* pi_out, double* partials,
                                                          unsigned int* ticket, double* out_sum) {
  __shared__ double s_red[8];
  constexpr int U = 4;
  const bool vec = ((reinterpret_cast<uintptr_t>(e) | reinterpret_cast<uintptr_t>(pi_out)) & 15u) == 0;
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  double acc0 = 0.0, acc1 = 0.0;
  auto one = [&](double ev) {
    const double t = ev * scale_t;
    const double den = c + t;
    // IEEE division where the weights are returned (rlvi.py:42), fast reciprocal for the objective only;
    // den outside the normal range (t = inf, c + t = 0) takes the IEEE path too
    const unsigned int ex = (unsigned int)(__double2hiint(den) >> 20) & 0x7ffu;
    return (pi_out != nullptr || (ex - 123u) >= 1800u) ? t / den : t * shift_rcp(den);
  };
  if (vec) {
    const double2* ev = reinterpret_cast<const double2*>(e);
    double2* pv = reinterpret_cast<double2*>(pi_out);
    const int64_t nvec = n >> 1;
    int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    for (; i < nvec; i += U * stride) {
      double2 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) v[u] = (i + u * stride < nvec) ? ev[i + u * stride] : make_double2(0.0, 0.0);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (i + u * stride < nvec) {
          const double r0 = one(v[u].x), r1 = one(v[u].y);
          acc0 += r0;
          acc1 += r1;
          if (pi_out) pv[i + u * stride] = make_double2(r0, r1);
        }
      }
    }
    if ((n & 1) && blockIdx.x == 0 && threadIdx.x == 0) {
      const double r0 = one(e[n - 1]);
      acc0 += r0;
      if (pi_out) pi_out[n - 1] = r0;
    }
  } else {
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
      const double r0 = one(e[i]);
      acc0 += r0;
      if (pi_out) pi_out[i] = r0;
    }
  }
  double v[1] = {acc0 + acc1};
  block_sum<1>(v, s_red);
  if (grid_total<1>(v, partials, ticket)) out_sum[0] = v[0];
}

}  // namespace

extern "C" int rlvi_wce_fwd_bwd_f32(rlvi_ctx* ctx, const float* logits, const int64_t* labels,
                                    const int64_t* indexes, const float* weights, float* residuals, int64_t batch,
                                    int classes, int64_t n_train, float* per_sample_out, float* dlogits,
                                    float* out_loss, int32_t* out_correct, void* stream) {
  RLVI_REQUIRE(ctx && logits && labels && weights && residuals && out_loss, "null pointer");
  RLVI_REQUIRE(batch > 0 && classes > 0 && n_train > 0, "batch, classes, n_train must be positive");
  if (classes > 1024) {
    rlvi_set_error("rlvi_wce_fwd_bwd_f32 supports classes <= 1024 (got %d)", classes);
    return RLVI_ERR_UNSUPPORTED;
  }
  RlviDeviceGuard guard(ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int nwarp = kWceThreads / 32;
  int64_t want = (batch + nwarp - 1) / nwarp;
  const int64_t cap = int64_t(ctx->sm_count) * 8;
  const int grid = int(want > cap ? cap : want);
  RlviScratch s;
  const int rc = rlvi_scratch_header(ctx, size_t(grid) * sizeof(double), &s);
  if (rc != RLVI_OK) return rc;
  WceParams p;
  p.logits = logits;
  p.labels = labels;
  p.indexes = indexes;
  p.weights = weights;
  p.residuals = residuals;
  p.per_sample = per_sample_out;
  p.dlogits = dlogits;
  p.out_loss = out_loss;
  p.out_correct = out_correct;
  p.batch = batch;
  p.classes = classes;
  p.n_train = n_train;
  p.ticket = s.ticket;
  p.partials = s.partials;
  if (out_correct) RLVI_CUDA(cudaMemsetAsync(out_correct, 0, 2 * sizeof(int32_t), st));
  if (classes <= 128)
    wce_kernel<4><<<grid, kWceThreads, 0, st>>>(p);
  else if (classes <= 256)
    wce_kernel<8><<<grid, kWceThreads, 0, st>>>(p);
  else
    wce_kernel<32><<<grid, kWceThreads, 0, st>>>(p);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}

extern "C" int rlvi_fn_threshold_f32(rlvi_ctx* ctx, float* weights, int64_t n, float alpha, float prev_threshold,
                                     int truncate, float* out_threshold, void* stream) {
  RLVI_REQUIRE(ctx && weights && out_threshold, "null pointer");
  RLVI_REQUIRE(n > 0, "n must be positive");
  RLVI_REQUIRE(n < (int64_t(1) << 22), "single-CTA selection supports n < 2^22");
  RlviDeviceGuard guard(ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t cache = (size_t(n) * 4 + 15) & ~size_t(15);
  if (cache <= size_t(200) * 1024) {
    RLVI_CUDA(cudaFuncSetAttribute(fn_threshold_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   200 * 1024));
    fn_threshold_kernel<true><<<1, kThrThreads, cache, st>>>(weights, n, alpha, prev_threshold, truncate,
                                                             out_threshold);
  } else {
    fn_threshold_kernel<false><<<1, kThrThreads, 0, st>>>(weights, n, alpha, prev_threshold, truncate,
                                                          out_threshold);
  }
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}

extern "C" int rlvi_shift_sum_f64(rlvi_ctx* ctx, const double* losses, int64_t n, double shift, double c,
                                  double* pi_out, double* out_sum, void* stream) {
  RLVI_REQUIRE(ctx && losses && out_sum, "null pointer");
  RLVI_REQUIRE(n > 0, "n must be positive");
  RlviDeviceGuard guard(ctx->device);
  const int grid = grid_for(ctx, n, 4);
  RlviScratch s;
  const int rc = rlvi_scratch_header(ctx, size_t(grid) * sizeof(double), &s);
  if (rc != RLVI_OK) return rc;
  shift_sum_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(losses, n, shift, c, pi_out, s.partials, s.ticket,
                                                                        out_sum);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}

extern "C" int rlvi_shift_sum_e_f64(rlvi_ctx* ctx, const double* e, int64_t n, double scale_t, double c, double* pi_out,
                                    double* out_sum, void* stream) {
  RLVI_REQUIRE(ctx && e && out_sum, "null pointer");
  RLVI_REQUIRE(n > 0, "n must be positive");
  RLVI_REQUIRE(scale_t >= 0.0 && scale_t < 1e300, "scale_t = exp(shift) must be finite and non-negative");
  RlviDeviceGuard guard(ctx->device);
  const int grid = grid_for(ctx, n, 8);
  RlviScratch s;
  const int rc = rlvi_scratch_header(ctx, size_t(grid) * sizeof(double), &s);
  if (rc != RLVI_OK) return rc;
  shift_sum_e_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(e, n, scale_t, c, pi_out, s.partials, s.ticket,
                                                                          out_sum);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}
