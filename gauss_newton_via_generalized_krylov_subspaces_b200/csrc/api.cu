// api.cu -- context lifecycle and error reporting of the gnk_b200 C ABI.
#include <stdlib.h>

#include "common.cuh"

void gnk_comm_teardown(gnk_ctx* ctx);

namespace {
thread_local std::string g_err;
}

void gnk_set_error(const std::string& s) { g_err = s; }

int gnk_fail(const char* what, cudaError_t e, const char* file, int line) {
  char buf[512];
  snprintf(buf, sizeof(buf), "%s failed: %s (%s:%d)", what, cudaGetErrorString(e), file, line);
  g_err = buf;
  return -1;
}

int gnk_pdl_mode() {
  static const int mode = getenv("GNK_PDL") ? atoi(getenv("GNK_PDL")) : 1;
  return mode;
}

extern "C" {

int gnk_abi_version(void) { return GNK_B200_ABI_VERSION; }

const char* gnk_last_error(void) { return g_err.c_str(); }

int gnk_create(gnk_ctx** out, int device) {
  GNK_REQUIRE(out, "gnk_create: null argument");
  *out = nullptr;
  int count = 0;
  GNK_CUDA(cudaGetDeviceCount(&count));
  GNK_REQUIRE(device >= 0 && device < count, "gnk_create: no such CUDA device");
  GNK_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  GNK_CUDA(cudaGetDeviceProperties(&prop, device));
  gnk_ctx* ctx = new gnk_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  GNK_CUDA(cudaMalloc(&ctx->d_partials, sizeof(double) * GNK_PARTIALS));
  GNK_CUDA(cudaMemset(ctx->d_partials, 0, sizeof(double) * GNK_PARTIALS));
  GNK_CUDA(cudaMalloc(&ctx->d_tickets, sizeof(unsigned int) * GNK_TICKETS));
  GNK_CUDA(cudaMemset(ctx->d_tickets, 0, sizeof(unsigned int) * GNK_TICKETS));
  GNK_CUDA(cudaMallocHost(&ctx->h_pinned, sizeof(double) * 64));
  *out = ctx;
  return 0;
}

int gnk_destroy(gnk_ctx* ctx) {
  if (!ctx) return 0;
  cudaSetDevice(ctx->device);
  gnk_comm_teardown(ctx);
  if (ctx->d_partials) cudaFree(ctx->d_partials);
  if (ctx->d_tickets) cudaFree(ctx->d_tickets);
  for (int b = 0; b < 2; ++b)
    if (ctx->d_rbuf[b]) cudaFree(ctx->d_rbuf[b]);
  if (ctx->d_gather) cudaFree(ctx->d_gather);
  if (ctx->d_apart) cudaFree(ctx->d_apart);
  if (ctx->d_cholqr) cudaFree(ctx->d_cholqr);
  if (ctx->d_gramw) cudaFree(ctx->d_gramw);
  if (ctx->d_pattern) cudaFree(ctx->d_pattern);
  if (ctx->d_dqr) cudaFree(ctx->d_dqr);
  if (ctx->d_wls) cudaFree(ctx->d_wls);
  if (ctx->d_wdots) cudaFree(ctx->d_wdots);
  if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
  if (ctx->fetch_stream) cudaStreamDestroy(ctx->fetch_stream);
  if (ctx->fetch_event) cudaEventDestroy(ctx->fetch_event);
  for (cudaEvent_t e : ctx->cg_event)
    if (e) cudaEventDestroy(e);
  delete ctx;
  return 0;
}

int gnk_sm_count(gnk_ctx* ctx) { return ctx ? ctx->sm_count : 0; }

int64_t gnk_launch_count(gnk_ctx* ctx) { return ctx ? ctx->launches : 0; }

// The scalar read-back of an outer iteration (gnk_b200.h): the copy waits for the work enqueued on `stream` so far and
// runs on the context's own copy stream, so kernels enqueued on `stream` AFTER this call keep the device busy while the
// host sits in gnk_scalars_wait.  Two driver calls and one wait instead of an event, a stream switch, a tensor copy and
// a stream synchronisation through the framework (~25 us of host time per outer iteration in the latency regime).
int gnk_scalars_fetch(gnk_ctx* ctx, const double* d_src, int count, double* h_dst, void* stream) {
  GNK_REQUIRE(ctx && d_src && h_dst && count >= 1, "gnk_scalars_fetch: bad argument");
  if (int rc = gnk_ensure_fetch_stream(ctx)) return rc;
  GNK_CUDA(cudaEventRecord(ctx->fetch_event, (cudaStream_t)stream));
  GNK_CUDA(cudaStreamWaitEvent(ctx->fetch_stream, ctx->fetch_event, 0));
  GNK_CUDA(cudaMemcpyAsync(h_dst, d_src, sizeof(double) * (size_t)count, cudaMemcpyDeviceToHost, ctx->fetch_stream));
  return 0;
}

int gnk_scalars_wait(gnk_ctx* ctx) {
  GNK_REQUIRE(ctx && ctx->fetch_stream, "gnk_scalars_wait: no fetch in flight");
  GNK_CUDA(cudaStreamSynchronize(ctx->fetch_stream));
  return 0;
}

}  // extern "C"

int gnk_ensure_fetch_stream(gnk_ctx* ctx) {
  if (!ctx->fetch_stream) {
    GNK_CUDA(cudaSetDevice(ctx->device));
    GNK_CUDA(cudaStreamCreateWithFlags(&ctx->fetch_stream, cudaStreamNonBlocking));
    GNK_CUDA(cudaEventCreateWithFlags(&ctx->fetch_event, cudaEventDisableTiming));
  }
  return 0;
}
