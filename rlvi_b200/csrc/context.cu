// context.cu -- library context, scratch management, error reporting.
#include <stdarg.h>

#include "common.cuh"

static thread_local char g_err[512] = "";

void rlvi_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" const char* rlvi_last_error(void) { return g_err; }
extern "C" int rlvi_version(void) { return 100; }

extern "C" int rlvi_ctx_create(int device, rlvi_ctx** out) {
  RLVI_REQUIRE(out != nullptr, "null output pointer");
  *out = nullptr;
  int count = 0;
  RLVI_CUDA(cudaGetDeviceCount(&count));
  RLVI_REQUIRE(device >= 0 && device < count, "no such CUDA device");
  RlviDeviceGuard guard(device);
  cudaDeviceProp prop;
  RLVI_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) {
    rlvi_set_error("librlvi_b200 needs an sm_100a device (B200); device %d is sm_%d%d", device, prop.major,
                   prop.minor);
    return RLVI_ERR_UNSUPPORTED;
  }
  rlvi_ctx* ctx = new rlvi_ctx();
  memset(ctx, 0, sizeof(*ctx));
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  // 8 MiB covers every per-launch scratch need at d <= 64; larger shapes grow it on demand.
  ctx->scratch_bytes = size_t(8) << 20;
  if (cudaMalloc(&ctx->scratch, ctx->scratch_bytes) != cudaSuccess) {
    rlvi_set_error("cudaMalloc of %zu scratch bytes failed", ctx->scratch_bytes);
    delete ctx;
    return RLVI_ERR_NOMEM;
  }
  cudaMemset(ctx->scratch, 0, ctx->scratch_bytes);
  ctx->pinned_bytes = size_t(1) << 20;
  if (cudaMallocHost(&ctx->pinned, ctx->pinned_bytes) != cudaSuccess) {
    cudaFree(ctx->scratch);
    delete ctx;
    rlvi_set_error("cudaMallocHost failed");
    return RLVI_ERR_NOMEM;
  }
  cudaError_t e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
  for (int i = 0; i < 4 && e == cudaSuccess; ++i) e = cudaEventCreateWithFlags(&ctx->ev[i], cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    rlvi_set_error("context set-up -> %s", cudaGetErrorString(e));
    rlvi_ctx_destroy(ctx);
    return RLVI_ERR_CUDA;
  }
  *out = ctx;
  return RLVI_OK;
}

extern "C" int rlvi_ctx_destroy(rlvi_ctx* ctx) {
  if (!ctx) return RLVI_OK;
  RlviDeviceGuard guard(ctx->device);
  cudaDeviceSynchronize();
  if (ctx->scratch) cudaFree(ctx->scratch);
  if (ctx->big) cudaFree(ctx->big);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  for (int i = 0; i < 4; ++i)
    if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
  delete ctx;
  return RLVI_OK;
}

extern "C" int rlvi_ctx_sm_count(const rlvi_ctx* ctx) { return ctx ? ctx->sm_count : 0; }
extern "C" int64_t rlvi_ctx_launch_count(const rlvi_ctx* ctx) { return ctx ? ctx->launches : 0; }

// New scratch is zeroed.  Its layout (a header of control words, then per-launch partials) and which words must be
// left at zero are stated once, next to rlvi_scratch_header in common.cuh.
int rlvi_scratch(rlvi_ctx* ctx, size_t bytes, void** out) {
  if (bytes > ctx->scratch_bytes) {
    // Growing is rare (only for d > 64 shapes); it synchronises the device so that no in-flight
    // kernel still uses the old block.
    RLVI_CUDA(cudaDeviceSynchronize());
    void* p = nullptr;
    size_t want = bytes + (bytes >> 2);
    if (cudaMalloc(&p, want) != cudaSuccess) {
      rlvi_set_error("cudaMalloc of %zu scratch bytes failed", want);
      return RLVI_ERR_NOMEM;
    }
    if (cudaMemset(p, 0, want) != cudaSuccess) {
      cudaFree(p);
      rlvi_set_error("cudaMemset of the new scratch failed");
      return RLVI_ERR_CUDA;
    }
    cudaFree(ctx->scratch);
    ctx->scratch = p;
    ctx->scratch_bytes = want;
  }
  *out = ctx->scratch;
  return RLVI_OK;
}
