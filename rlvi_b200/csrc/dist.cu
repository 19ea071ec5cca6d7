// dist.cu -- NVLink peer windows for the in-kernel exchange of the sharded fixed point.
//
// One process per GPU.  Each rank allocates a small window (rlvi_fp_dist_inbox_doubles(world) doubles),
// exports it as a CUDA IPC handle, the host side gathers the handles of all ranks (any transport: the
// Python layer uses torch.distributed), and every rank maps its peers' windows.  The fixed-point kernel
// then stores its per-pass partial sums straight into the peers' windows over NVLink
// (fixed_point.cu: grid_allreduce3) -- no NCCL call, no host round trip per pass.
#include "common.cuh"

extern "C" int rlvi_dist_window_create(rlvi_ctx* ctx, int world, void** window_out, unsigned char* handle_out) {
  RLVI_REQUIRE(ctx && window_out && handle_out, "null pointer");
  RLVI_REQUIRE(world >= 1 && world <= 32, "world must be in 1..32");
  RlviDeviceGuard guard(ctx->device);
  static_assert(sizeof(cudaIpcMemHandle_t) == RLVI_IPC_HANDLE_BYTES, "IPC handle size");
  const size_t bytes = size_t(rlvi_fp_dist_inbox_doubles(world)) * sizeof(double);
  void* w = nullptr;
  RLVI_CUDA(cudaMalloc(&w, bytes));
  RLVI_CUDA(cudaMemset(w, 0, bytes));
  RLVI_CUDA(cudaDeviceSynchronize());
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, w);
  if (e != cudaSuccess) {
    cudaFree(w);
    rlvi_set_error("cudaIpcGetMemHandle -> %s", cudaGetErrorString(e));
    return RLVI_ERR_CUDA;
  }
  memcpy(handle_out, &h, sizeof(h));
  *window_out = w;
  return RLVI_OK;
}

extern "C" int rlvi_dist_window_open(rlvi_ctx* ctx, int rank, int world, void* own_window,
                                     const unsigned char* all_handles, void** peer_table_out) {
  RLVI_REQUIRE(ctx && own_window && all_handles && peer_table_out, "null pointer");
  RLVI_REQUIRE(world >= 1 && world <= 32 && rank >= 0 && rank < world, "bad rank/world");
  RlviDeviceGuard guard(ctx->device);
  void* host_table[32];
  for (int r = 0; r < world; ++r) {
    if (r == rank) {
      host_table[r] = own_window;
      continue;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, all_handles + size_t(r) * sizeof(h), sizeof(h));
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      for (int q = 0; q < r; ++q)
        if (q != rank) cudaIpcCloseMemHandle(host_table[q]);
      rlvi_set_error("cudaIpcOpenMemHandle(rank %d) -> %s", r, cudaGetErrorString(e));
      return RLVI_ERR_CUDA;
    }
    host_table[r] = p;
  }
  void* table = nullptr;
  RLVI_CUDA(cudaMalloc(&table, sizeof(void*) * 32));
  RLVI_CUDA(cudaMemcpy(table, host_table, sizeof(void*) * world, cudaMemcpyHostToDevice));
  *peer_table_out = table;
  return RLVI_OK;
}

extern "C" int rlvi_dist_window_close(rlvi_ctx* ctx, int rank, int world, void* own_window, void* peer_table) {
  RLVI_REQUIRE(ctx != nullptr, "null context");
  RlviDeviceGuard guard(ctx->device);
  cudaDeviceSynchronize();
  if (peer_table) {
    void* host_table[32];
    if (world >= 1 && world <= 32 &&
        cudaMemcpy(host_table, peer_table, sizeof(void*) * world, cudaMemcpyDeviceToHost) == cudaSuccess) {
      for (int r = 0; r < world; ++r)
        if (r != rank && host_table[r]) cudaIpcCloseMemHandle(host_table[r]);
    }
    cudaFree(peer_table);
  }
  if (own_window) cudaFree(own_window);
  return RLVI_OK;
}

// ---------------------------------------------------------------------------------------------
// statistics all-reduce over the peer windows (no NCCL)
// ---------------------------------------------------------------------------------------------
namespace {

__device__ __forceinline__ unsigned long long ld_acq_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_rel_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ double ld_vol(const double* p) {
  double v;
  asm volatile("ld.volatile.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}

struct StatsParams {
  double* buf;
  int count;
  int rank, world;
  double* inbox;
  double* const* peer_inbox;
  unsigned long long call_index;
  unsigned int* control;   // [0] ticket, [1] failure flag
};

__global__ void __launch_bounds__(256) stats_allreduce_kernel(const StatsParams p) {
  __shared__ int s_last, s_fail;
  const int parity = int(p.call_index & 1ull);
  const size_t tag_off = size_t(24) * p.world + size_t(parity) * p.world;
  const size_t data_off = size_t(26) * p.world + size_t(parity) * p.world * RLVI_DIST_STATS_CAPACITY;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  // ---- phase A: my values into slot `rank` of every rank's window (remote stores over NVLink)
  if (e < p.count) {
    const double v = p.buf[e];
    for (int r = 0; r < p.world; ++r) p.peer_inbox[r][data_off + size_t(p.rank) * RLVI_DIST_STATS_CAPACITY + e] = v;
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int t = atomicAdd(p.control, 1u);
    s_last = (t == gridDim.x - 1) ? 1 : 0;
  }
  __syncthreads();
  if (s_last && threadIdx.x < p.world) {   // all blocks of this rank have stored: publish the tag to everyone
    __threadfence_system();
    st_rel_sys(reinterpret_cast<unsigned long long*>(p.peer_inbox[threadIdx.x] + tag_off + p.rank), p.call_index);
  }
  // ---- phase B: wait for every rank's tag in my own window, then add the slots in rank order
  if (threadIdx.x < p.world) {
    const unsigned long long* flag = reinterpret_cast<const unsigned long long*>(p.inbox + tag_off + threadIdx.x);
    unsigned long long t0;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t0));
    int fail = 0;
    while (ld_acq_sys(flag) != p.call_index) {
      unsigned long long t1;
      asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t1));
      if (t1 - t0 > 20ull * 1000ull * 1000ull * 1000ull) { fail = 1; break; }
    }
    if (fail) atomicExch(p.control + 1, 1u);
  }
  __syncthreads();
  if (threadIdx.x == 0) s_fail = int(*reinterpret_cast<volatile unsigned int*>(p.control + 1));
  __syncthreads();
  if (e < p.count) {
    double s = 0.0;
    for (int r = 0; r < p.world; ++r) s += ld_vol(p.inbox + data_off + size_t(r) * RLVI_DIST_STATS_CAPACITY + e);
    p.buf[e] = s_fail ? nan("") : s;       // a dead peer poisons the result instead of hanging
  }
}

}  // namespace

extern "C" int rlvi_stats_allreduce_f64(rlvi_ctx* ctx, double* buf, int count, const rlvi_fp_dist* dist, void* stream) {
  RLVI_REQUIRE(ctx && buf && dist, "null pointer");
  RLVI_REQUIRE(count > 0 && count <= RLVI_DIST_STATS_CAPACITY, "count must be in 1..RLVI_DIST_STATS_CAPACITY");
  RLVI_REQUIRE(dist->world >= 1 && dist->world <= 32 && dist->rank >= 0 && dist->rank < dist->world, "bad rank/world");
  RLVI_REQUIRE(dist->inbox && dist->peer_inbox && dist->call_index > 0, "incomplete rlvi_fp_dist");
  RlviDeviceGuard guard(ctx->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  RlviScratch s;
  const int rc = rlvi_scratch_header(ctx, 0, &s);
  if (rc != RLVI_OK) return rc;
  StatsParams p;
  p.buf = buf;
  p.count = count;
  p.rank = dist->rank;
  p.world = dist->world;
  p.inbox = dist->inbox;
  p.peer_inbox = dist->peer_inbox;
  p.call_index = dist->call_index;
  p.control = s.control;
  RLVI_CUDA(cudaMemsetAsync(p.control, 0, kScratchControlBytes, st));
  const int grid = (count + 255) / 256;     // <= 32 CTAs: always co-resident
  stats_allreduce_kernel<<<grid, 256, 0, st>>>(p);
  RLVI_LAUNCH_CHECK(ctx);
  return RLVI_OK;
}
