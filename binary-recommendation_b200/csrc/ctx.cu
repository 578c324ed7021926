// Context, error string and workspace of libbrk_b200.
#include <stdarg.h>
#include <string.h>
#include <stdlib.h>
#include "common.cuh"

static thread_local char g_err[512] = "";

void brk_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" int brk_abi_version(void) { return BRK_ABI_VERSION; }
extern "C" const char* brk_last_error(void) { return g_err; }

extern "C" int brk_create(brk_ctx** out, int device) {
  BRK_REQUIRE(out != nullptr, BRK_E_ARG, "brk_create: out is null");
  *out = nullptr;
  int ndev = 0;
  BRK_CUDA(cudaGetDeviceCount(&ndev));
  BRK_REQUIRE(device >= 0 && device < ndev, BRK_E_ARG, "brk_create: device %d of %d", device, ndev);
  BRK_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  BRK_CUDA(cudaGetDeviceProperties(&prop, device));
  BRK_REQUIRE(prop.major == 10, BRK_E_STATE,
              "brk_create: device is sm_%d%d; this library is built for sm_100a only", prop.major, prop.minor);
  brk_ctx* c = (brk_ctx*)calloc(1, sizeof(brk_ctx));
  BRK_REQUIRE(c != nullptr, BRK_E_STATE, "brk_create: out of host memory");
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  BRK_CUDA(cudaMalloc(&c->loss_acc, BRK_LOSS_SLOTS * sizeof(double)));
  BRK_CUDA(cudaMemset(c->loss_acc, 0, BRK_LOSS_SLOTS * sizeof(double)));
  BRK_CUDA(cudaMalloc(&c->tickets, BRK_TICKETS * sizeof(unsigned int)));
  BRK_CUDA(cudaMemset(c->tickets, 0, BRK_TICKETS * sizeof(unsigned int)));
  const size_t bar_bytes = BRK_BAR_FAMILIES * BRK_BAR_LINE_WORDS * sizeof(unsigned int);
  BRK_CUDA(cudaMalloc(&c->bar[0], bar_bytes));
  BRK_CUDA(cudaMemset(c->bar[0], 0, bar_bytes));
  for (int k = 1; k < BRK_BAR_FAMILIES; ++k) c->bar[k] = c->bar[0] + k * BRK_BAR_LINE_WORDS;
  c->scratch = nullptr;
  c->scratch_bytes = 0;
  for (int j = 0; j < BRK_FORK_STREAMS; ++j) {
    BRK_CUDA(cudaStreamCreateWithFlags(&c->fork_stream[j], cudaStreamNonBlocking));
    BRK_CUDA(cudaEventCreateWithFlags(&c->ev_fork[j], cudaEventDisableTiming));
    BRK_CUDA(cudaEventCreateWithFlags(&c->ev_join[j], cudaEventDisableTiming));
  }
  BRK_CUDA(cudaDeviceSynchronize());
  *out = c;
  return 0;
}

int brk_ctx_ensure_copy(brk_ctx* ctx) {
  if (ctx->copy_ready) return 0;
  BRK_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  for (int q = 0; q < BRK_STAGE_EVENTS; ++q) {
    BRK_CUDA(cudaEventCreateWithFlags(&ctx->ev_ready[q], cudaEventDisableTiming));
    BRK_CUDA(cudaEventCreateWithFlags(&ctx->ev_done[q], cudaEventDisableTiming));
  }
  for (int a = 0; a < BRK_COPY_AUX; ++a) {
    BRK_CUDA(cudaStreamCreateWithFlags(&ctx->copy_aux[a], cudaStreamNonBlocking));
    BRK_CUDA(cudaEventCreateWithFlags(&ctx->ev_aux[a], cudaEventDisableTiming));
  }
  BRK_CUDA(cudaEventCreateWithFlags(&ctx->ev_go, cudaEventDisableTiming));
  ctx->copy_ready = 1;
  return 0;
}

extern "C" int brk_destroy(brk_ctx* c) {
  if (!c) return 0;
  cudaSetDevice(c->device);
  if (c->loss_acc) cudaFree(c->loss_acc);
  if (c->tickets) cudaFree(c->tickets);
  if (c->scratch) cudaFree(c->scratch);
  if (c->neumf_img) cudaFree(c->neumf_img);
  if (c->neumf_part) cudaFree(c->neumf_part);
  if (c->neumf_gen) cudaFree(c->neumf_gen);
  if (c->tt_part) cudaFree(c->tt_part);
  if (c->tt_logq) cudaFree(c->tt_logq);
  if (c->bar[0]) cudaFree(c->bar[0]);
  for (int j = 0; j < BRK_FORK_STREAMS; ++j)
    if (c->fork_stream[j]) { cudaStreamDestroy(c->fork_stream[j]); cudaEventDestroy(c->ev_fork[j]); cudaEventDestroy(c->ev_join[j]); }
  if (c->copy_ready) {
    cudaStreamDestroy(c->copy_stream);
    for (int i = 0; i < BRK_STAGE_EVENTS; ++i) { cudaEventDestroy(c->ev_ready[i]); cudaEventDestroy(c->ev_done[i]); }
    for (int i = 0; i < BRK_COPY_AUX; ++i) { cudaStreamDestroy(c->copy_aux[i]); cudaEventDestroy(c->ev_aux[i]); }
    cudaEventDestroy(c->ev_go);
  }
  free(c);
  return 0;
}

extern "C" int brk_sm_count(const brk_ctx* c) { return c ? c->sm_count : BRK_E_ARG; }
