// Shared device/host helpers for libbrk_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/brk_b200.h"

// brk_ctx::bar: one block of grid-barrier words per cooperative kernel family
enum { BRK_BAR_BPR, BRK_BAR_TT, BRK_BAR_NEUMF, BRK_BAR_FAMILIES };
#define BRK_BAR_LINE_WORDS 32

struct brk_ctx {
  int device;
  int sm_count;
  double*       loss_acc;     // [BRK_LOSS_SLOTS] double accumulators, zero between calls
  unsigned int* tickets;      // [BRK_TICKETS] last-block tickets, zero between calls
  void*         scratch;      // sort / misc scratch
  size_t        scratch_bytes;
  // host-fed training: copy stream + events for H2D prefetch / loss D2H (created on first use)
  cudaStream_t  copy_stream;
  cudaEvent_t   ev_ready[4], ev_done[4];
  cudaStream_t  copy_aux[3];  // extra DMA lanes: several H2D copies in flight
  cudaEvent_t   ev_aux[3], ev_go;
  int           copy_ready;
  // NeuMF tensor-core path: swizzled weight images, rebuilt every step (csrc/neumf_tc.cu)
  float*        neumf_img;
  size_t        neumf_img_floats;
  // one-launch NeuMF step (csrc/neumf_fused.cu): per-tile slots of partial sums, summed after a grid barrier
  float*        neumf_part;
  size_t        neumf_part_floats;
  // one-launch two-tower step (csrc/twotower_fused.cu): per-tile softmax partials
  float*        tt_part;
  size_t        tt_part_floats;
  // grid-barrier words of the cooperative step kernels (layout at brk_grid_barrier): bar[BRK_BAR_*], each on its own
  // 128-byte line of one allocation (bar[0]).  Launches of one family on one context are stream-ordered: a launch reads
  // the base (and tag) that its predecessor wrote back.
  unsigned int* bar[BRK_BAR_FAMILIES];
  // any-width NeuMF path (csrc/neumf_generic.cu): feature-major intermediates
  float*        neumf_gen;
  size_t        neumf_gen_floats;
  // fork/join inside one call: independent kernel chains of a step (the two towers of twotower.cu and, inside each,
  // the Dense-gradient products beside the embedding-gradient chain) run side by side on these streams
  cudaStream_t  fork_stream[3];
  cudaEvent_t   ev_fork[3], ev_join[3];
};
#define BRK_FORK_STREAMS 3

// Runs what follows on ctx->fork_stream[j] after everything queued on `from` so far ...
#define BRK_FORK(ctx, from, j)                                                   \
  do {                                                                           \
    BRK_CUDA(cudaEventRecord((ctx)->ev_fork[j], (from)));                        \
    BRK_CUDA(cudaStreamWaitEvent((ctx)->fork_stream[j], (ctx)->ev_fork[j], 0));  \
  } while (0)
// ... and makes `into` wait for that chain (both work under stream capture: the chain becomes a graph branch).
#define BRK_JOIN(ctx, into, j)                                                   \
  do {                                                                           \
    BRK_CUDA(cudaEventRecord((ctx)->ev_join[j], (ctx)->fork_stream[j]));         \
    BRK_CUDA(cudaStreamWaitEvent((into), (ctx)->ev_join[j], 0));                 \
  } while (0)

#define BRK_STAGE_EVENTS 4
#define BRK_COPY_AUX 3
#define BRK_LOSS_SLOTS 16
#define BRK_TICKETS 16

void brk_set_error(const char* fmt, ...);
// copy stream + staging events of the host-fed training entry points (created on first use)
int brk_ctx_ensure_copy(brk_ctx* ctx);

#define BRK_REQUIRE(cond, code, ...)            \
  do {                                          \
    if (!(cond)) {                              \
      brk_set_error(__VA_ARGS__);               \
      return (code);                            \
    }                                           \
  } while (0)

#define BRK_CUDA(expr)                                                            \
  do {                                                                            \
    cudaError_t _e = (expr);                                                      \
    if (_e != cudaSuccess) {                                                      \
      brk_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),       \
                    __FILE__, __LINE__);                                          \
      return (int)_e;                                                             \
    }                                                                             \
  } while (0)

#define BRK_LAUNCH_CHECK()                                                        \
  do {                                                                            \
    cudaError_t _e = cudaGetLastError();                                          \
    if (_e != cudaSuccess) {                                                      \
      brk_set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e),   \
                    __FILE__, __LINE__);                                          \
      return (int)_e;                                                             \
    }                                                                             \
  } while (0)

#ifdef __CUDACC__
#define BRK_HD __host__ __device__
#else
#define BRK_HD
#endif
BRK_HD static inline bool brk_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Lanes-per-row for a vectorised row of d4 float4 chunks: smallest power of two >= d4, capped at 32.
static inline int brk_lanes_per_row(int d4) {
  int l = 1;
  while (l < d4 && l < 32) l <<= 1;
  return l;
}

#ifdef __CUDACC__

// 128-bit streaming loads/stores. Table rows are read through the read-only path; rows that are
// written once and not re-read by the same kernel bypass L1 allocation.
__device__ __forceinline__ float4 ldg_nc_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_na_f4(float4* p, const float4& v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
// Vector reduction to global memory: one 16-byte RED instead of four scalar ones (sm_90+).
__device__ __forceinline__ void red_add_f4(float* p, const float4& v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

__device__ __forceinline__ float warp_sum(float x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}
template <int LANES>
__device__ __forceinline__ float group_sum(float x) {   // sum over aligned groups of LANES lanes
#pragma unroll
  for (int o = LANES / 2; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}

// Block-wide sum of a per-thread double; result valid in thread 0. smem: >= 32 doubles.
__device__ __forceinline__ double block_sum_double(double x, double* smem) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) smem[w] = x;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  x = (threadIdx.x < nw) ? smem[threadIdx.x] : 0.0;
  if (w == 0) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  }
  return x;
}

// Grid barrier of a cooperative launch: one release-RED per CTA on an arrival counter that only grows, then an acquire
// spin by thread 0 (cg::grid.sync() costs two fences and an atomic with return: ~1 us more per barrier in nfz::fused_step,
// 0.3-0.5 us in bpr_steps_coop).  Words of one kernel family (brk_ctx::bar):
//   [0] count  arrivals since the context was created (wraps; compared as a signed difference)
//   [1] error  set by a wait that timed out (and by nfz's tagged-slot waits)
//   [2] base   count at which the next launch starts: read by every CTA at entry, written back by one thread after the
//              launch's last barrier, so launches chain (and replay from a CUDA graph) with no host bookkeeping
//   [3] tag    nfz only: tag of the last launch's self-validating slot words (a launch uses the next one, never 0)
// `target` starts at the base and is the count at which every CTA of the current round has arrived.  The wait is bounded:
// a lost CTA sets the error word and TRAPS (the launch fails at the next synchronisation) instead of hanging the GPU.
constexpr long long kBrkBarrierSpin = 8000000000LL;   // clock64 cycles
__device__ __forceinline__ void brk_grid_arrive(unsigned int* bar, unsigned int& target) {
  __syncthreads();
  target += gridDim.x;
  if (threadIdx.x == 0) asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(bar) : "memory");
}
__device__ __forceinline__ void brk_grid_wait(unsigned int* bar, unsigned int target) {
  if (threadIdx.x == 0) {
    const long long t0 = clock64();
    unsigned int v;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(bar) : "memory");
      if (clock64() - t0 > kBrkBarrierSpin) { atomicExch(bar + 1, 1u); __trap(); }
    } while (int(v - target) < 0);
  }
}
__device__ __forceinline__ void brk_grid_barrier(unsigned int* bar, unsigned int& target) {
  brk_grid_arrive(bar, target);
  brk_grid_wait(bar, target);
  __syncthreads();
}

// Philox4x32-10 (Random123).  Known answers in tests/test_philox.py.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}

// "brk sampler v2" BPR stream (oracle/philox.py): one Philox draw picks rank r among the I - n items the
// user has NOT interacted with; the negative is the r-th such item: r + t with t the smallest index in
// [0, n] such that t == n or a[t] - t > r (a = the user's sorted positive list).  One binary search, no
// rejection loop, so the slowest sample of a batch costs the same as every other one.
constexpr uint32_t kBrkTagBpr = 0xB9u;
__device__ __forceinline__ int32_t brk_sample_bpr_negative(uint64_t idx, int64_t u, uint32_t seed, uint32_t epoch,
                                                           uint32_t num_items, const int64_t* __restrict__ indptr,
                                                           const int32_t* __restrict__ items) {
  const int64_t base = __ldg(indptr + u);
  const uint32_t n = uint32_t(__ldg(indptr + u + 1) - base);
  const uint4 w = philox4x32_10(make_uint4(uint32_t(idx), uint32_t(idx >> 32), 0u, kBrkTagBpr), seed, epoch);
  if (n >= num_items) return int32_t(__umulhi(w.x, num_items));
  const uint32_t r = __umulhi(w.x, num_items - n);
  const int32_t* __restrict__ a = items + base;
  uint32_t lo = 0, hi = n;                       // smallest t in [0, n] with t == n or a[t] - t > r
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (__ldg(a + mid) - int32_t(mid) > int32_t(r)) hi = mid; else lo = mid + 1;
  }
  return int32_t(r + lo);
}

__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

#endif  // __CUDACC__
