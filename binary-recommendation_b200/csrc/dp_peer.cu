// Fused data-parallel optimizer over NVLink peer memory: reduce-scatter of the gradient arena, Adam
// on the owned slice, all-gather of the updated weights -- ONE kernel, no NCCL on the data path.
// Replaces the per-step gradient all-reduce of tf.distribute's MultiWorkerMirroredStrategy
// (/root/reference/src/models/RModel.py:119-121) followed by Adam (NeuMFModel.py:89, BPRModel.py:70).
//
// Every rank holds the full weight arena w and gradient arena g in symmetric (peer-mapped) memory.
// Rank r owns float4 slice [r*n4/G, (r+1)*n4/G):
//   barrier-in   all ranks' fused fwd/bwd kernels have finished (their g is complete)
//   reduce       g_sum = sum_p g_p[slice]           (G-1 of G reads cross NVLink, 16-byte loads)
//   Adam         m, v exist ONLY for the owned slice (optimizer state is sharded G ways)
//   broadcast    w_p[slice] = w_new for every rank p (16-byte stores over NVLink) -> replicas stay
//                bit-identical because one rank computes each element
//   barrier-out  every rank has finished reading my g and writing my w
//   zero         my g arena (local) for the next step
// NVLink bytes per rank per step: (G-1)/G * 4n read + (G-1)/G * 4n written (n floats in the arena).
// Cross-rank flags are monotonic epochs (no reset), written with st.release.sys and polled with
// ld.acquire.sys; every spin has a clock64() deadline that raises an error flag instead of hanging.
#include <stdlib.h>
#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr long long kSpinBudget = 60000000000LL;    // default ~30 s at 2 GHz (BRK_PEER_SPIN_MS overrides): a rank may be
                                                    // seconds late into its first step (host-side data staging, checkpoint I/O)
long long spin_budget_cycles() {
  const char* e = getenv("BRK_PEER_SPIN_MS");
  if (e == nullptr) return kSpinBudget;
  const long long ms = atoll(e);
  return ms > 0 ? ms * 2000000LL : kSpinBudget;
}

struct DpParams {
  float* const* peer_w;
  float* const* peer_g;
  uint32_t* const* peer_flags;    // each: [2][world] uint32 (in, out)
  float* m; float* v;
  uint32_t* local_sync;           // [0] in_done [1] out_done [2] block counter [3] epoch [4] error
  int64_t n4;                     // arena length in float4
  int32_t rank, world;
  brk_adam_hyper h;
  int64_t* state;
  long long spin_budget;
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ bool spin_until(const uint32_t* p, uint32_t epoch, bool sys, uint32_t* err,
                                           long long budget = kSpinBudget) {
  const long long t0 = clock64();
  while (true) {
    const uint32_t v = sys ? ld_acquire_sys(p) : ld_acquire_gpu(p);
    if (int32_t(v - epoch) >= 0) return true;
    if (clock64() - t0 > budget) { atomicExch(err, 1u); return false; }
    __nanosleep(64);
  }
}

__global__ void __launch_bounds__(kThreads) dp_adam_peer_kernel(const DpParams P) {
  const int t = threadIdx.x, G = P.world, me = P.rank;
  uint32_t* sync = P.local_sync;
  const uint32_t epoch = sync[3] + 1u;               // sync[3] is only written by the last block, after all reads
  uint32_t* my_flags = P.peer_flags[me];

  // ---- barrier in: every rank's gradients are complete -------------------------------------------
  if (blockIdx.x == 0) {
    if (t < G) {
      st_release_sys(P.peer_flags[t] + me, epoch);               // "rank `me` is ready", posted on peer t
      spin_until(my_flags + t, epoch, true, sync + 4, P.spin_budget);   // wait for peer t's post on my pad
    }
    __syncthreads();
    if (t == 0) st_release_gpu(sync + 0, epoch);
  } else {
    if (t == 0) spin_until(sync + 0, epoch, false, sync + 4, 2 * P.spin_budget);
    __syncthreads();
  }
  // A peer that never arrived: this step is ABORTED on this rank -- no reduce over incomplete gradients, no Adam, no
  // broadcast, the gradient arena stays as it is.  The error word is sticky; PeerArena.check() raises on it.
  const bool dead = *reinterpret_cast<volatile uint32_t*>(sync + 4) != 0u;

  // Adam step size from the device-side optimizer state (running beta powers, see optim.cu)
  __shared__ float s_alpha;
  if (t == 0) {
    const double* pw = reinterpret_cast<const double*>(P.state);
    const double p1 = pw[1] * double(P.h.beta1), p2 = pw[2] * double(P.h.beta2);
    s_alpha = float(double(P.h.lr) * sqrt(1.0 - p2) / (1.0 - p1));
  }
  __syncthreads();
  const float alpha = s_alpha, b1 = P.h.beta1, b2 = P.h.beta2, eps = P.h.eps;
  const float omb1 = 1.f - b1, omb2 = 1.f - b2;

  // ---- reduce my slice from all peers, Adam, broadcast ---------------------------------------------
  const int64_t lo = P.n4 * me / G, hi = P.n4 * (me + 1) / G;
  float4* w_me = reinterpret_cast<float4*>(P.peer_w[me]);
  float4* m4 = reinterpret_cast<float4*>(P.m);
  float4* v4 = reinterpret_cast<float4*>(P.v);
  for (int64_t i = lo + int64_t(blockIdx.x) * kThreads + t; i < hi && !dead; i += int64_t(gridDim.x) * kThreads) {
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int p = 0; p < G; ++p) {                                // fixed order: deterministic sum
      const float4 x = *(reinterpret_cast<const float4*>(P.peer_g[p]) + i);
      g.x += x.x; g.y += x.y; g.z += x.z; g.w += x.w;
    }
    float4 w = w_me[i], mm = m4[i - lo], vv = v4[i - lo];
    mm.x = b1 * mm.x + omb1 * g.x; vv.x = b2 * vv.x + omb2 * g.x * g.x; w.x -= alpha * mm.x / (sqrtf(vv.x) + eps);
    mm.y = b1 * mm.y + omb1 * g.y; vv.y = b2 * vv.y + omb2 * g.y * g.y; w.y -= alpha * mm.y / (sqrtf(vv.y) + eps);
    mm.z = b1 * mm.z + omb1 * g.z; vv.z = b2 * vv.z + omb2 * g.z * g.z; w.z -= alpha * mm.z / (sqrtf(vv.z) + eps);
    mm.w = b1 * mm.w + omb1 * g.w; vv.w = b2 * vv.w + omb2 * g.w * g.w; w.w -= alpha * mm.w / (sqrtf(vv.w) + eps);
    m4[i - lo] = mm; v4[i - lo] = vv;
    for (int p = 0; p < G; ++p) *(reinterpret_cast<float4*>(P.peer_w[p]) + i) = w;
  }
  __threadfence_system();
  __syncthreads();

  // ---- barrier out: last block of this rank posts to / waits for the peers ---------------------------
  __shared__ bool s_last;
  if (t == 0) s_last = atomicAdd(sync + 2, 1u) == gridDim.x - 1;
  __syncthreads();
  if (s_last) {
    __threadfence_system();
    if (t < G && !dead) {
      st_release_sys(P.peer_flags[t] + G + me, epoch);
      spin_until(my_flags + G + t, epoch, true, sync + 4, P.spin_budget);
    }
    __syncthreads();
    if (t == 0) {
      double* pw = reinterpret_cast<double*>(P.state);           // advance the optimizer state (once per rank)
      if (!dead) { P.state[0] += 1; pw[1] *= double(P.h.beta1); pw[2] *= double(P.h.beta2); }
      sync[2] = 0u;
      sync[3] = epoch;
      __threadfence();
      st_release_gpu(sync + 1, epoch);
    }
  }
  if (t == 0) spin_until(sync + 1, epoch, false, sync + 4, 2 * P.spin_budget);
  __syncthreads();
  if (*reinterpret_cast<volatile uint32_t*>(sync + 4) != 0u) return;   // aborted: keep the gradients

  // ---- zero my gradient arena for the next step ----------------------------------------------------
  float4* g_me = reinterpret_cast<float4*>(P.peer_g[me]);
  for (int64_t i = int64_t(blockIdx.x) * kThreads + t; i < P.n4; i += int64_t(gridDim.x) * kThreads)
    g_me[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

// All-reduce (sum) of a flat fp32 arena over NVLink peer memory, in place on every rank: barrier in, every rank sums ITS
// float4 slice over all peers' arenas (fixed order: identical bits everywhere) and stores the sum into that slice of
// every peer's arena, barrier out.  The collective of a mirrored data-parallel step whose optimizer is not the fused
// Adam above (Keras Adagrad of the two-tower model, lazy Adam): stands in for the gradient all-reduce of
// MultiWorkerMirroredStrategy (src/models/RModel.py:119-121) without an NCCL call on the step's path.
__global__ void __launch_bounds__(kThreads) allreduce_peer_kernel(float* const* peer_buf, uint32_t* const* peer_flags,
                                                                  uint32_t* sync, int64_t n4, int me, int G, long long budget) {
  const int t = threadIdx.x;
  const uint32_t epoch = sync[3] + 1u;
  uint32_t* my_flags = peer_flags[me];
  if (blockIdx.x == 0) {
    if (t < G) {
      __threadfence_system();
      st_release_sys(peer_flags[t] + me, epoch);
      spin_until(my_flags + t, epoch, true, sync + 4, budget);
    }
    __syncthreads();
    if (t == 0) st_release_gpu(sync + 0, epoch);
  } else {
    if (t == 0) spin_until(sync + 0, epoch, false, sync + 4, 2 * budget);
    __syncthreads();
  }
  const bool dead = *reinterpret_cast<volatile uint32_t*>(sync + 4) != 0u;
  const int64_t lo = n4 * me / G, hi = n4 * (me + 1) / G;
  for (int64_t i = lo + int64_t(blockIdx.x) * kThreads + t; i < hi && !dead; i += int64_t(gridDim.x) * kThreads) {
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int p = 0; p < G; ++p) {
      const float4 x = *(reinterpret_cast<const float4*>(peer_buf[p]) + i);
      g.x += x.x; g.y += x.y; g.z += x.z; g.w += x.w;
    }
    for (int p = 0; p < G; ++p) *(reinterpret_cast<float4*>(peer_buf[p]) + i) = g;
  }
  __threadfence_system();
  __syncthreads();
  __shared__ bool s_last;
  if (t == 0) s_last = atomicAdd(sync + 2, 1u) == gridDim.x - 1;
  __syncthreads();
  if (s_last) {
    __threadfence_system();
    if (t < G && !dead) {
      st_release_sys(peer_flags[t] + G + me, epoch);
      spin_until(my_flags + G + t, epoch, true, sync + 4, budget);
    }
    __syncthreads();
    if (t == 0) { sync[2] = 0u; sync[3] = epoch; __threadfence(); st_release_gpu(sync + 1, epoch); }
  }
  if (t == 0) spin_until(sync + 1, epoch, false, sync + 4, 2 * budget);
  __syncthreads();
}

// Stand-alone cross-GPU barrier (one CTA): rank r posts epoch e on every peer's flag block and waits
// until every peer has posted e on its own.  Used between the sharded fused step (whose REDs land in the
// peers' accumulators) and the owners' optimizer pass.
__global__ void peer_barrier_kernel(uint32_t* const* peer_flags, uint32_t* local_sync, int rank, int world, long long budget) {
  const int t = threadIdx.x;
  const uint32_t epoch = local_sync[0] + 1u;
  __threadfence_system();
  if (t < world) {
    st_release_sys(peer_flags[t] + rank, epoch);
    spin_until(peer_flags[rank] + t, epoch, true, local_sync + 1, budget);
  }
  __syncthreads();
  if (t == 0) local_sync[0] = epoch;
}

}  // namespace

extern "C" int brk_dp_adam_peer(brk_ctx* ctx, const brk_dp_peer* d, brk_adam_hyper h, int64_t* state, void* stream) {
  BRK_REQUIRE(ctx && d && state, BRK_E_ARG, "brk_dp_adam_peer: null argument");
  BRK_REQUIRE(d->peer_w && d->peer_g && d->peer_flags && d->m && d->v && d->local_sync, BRK_E_ARG,
              "brk_dp_adam_peer: descriptor incomplete");
  BRK_REQUIRE(d->world >= 1 && d->world <= 64 && d->rank >= 0 && d->rank < d->world && d->n > 0 && (d->n & 3) == 0,
              BRK_E_ARG, "brk_dp_adam_peer: world=%d rank=%d n=%lld (n must be a multiple of 4)", d->world, d->rank,
              (long long)d->n);
  DpParams P;
  P.peer_w = d->peer_w; P.peer_g = d->peer_g; P.peer_flags = d->peer_flags; P.m = d->m; P.v = d->v;
  P.local_sync = d->local_sync; P.n4 = d->n / 4; P.rank = d->rank; P.world = d->world; P.h = h; P.state = state;
  P.spin_budget = spin_budget_cycles();
  // all CTAs spin on flags set by other CTAs: they must be co-resident -> cooperative launch, one CTA per SM at most
  const int64_t slice4 = (P.n4 + d->world - 1) / d->world;
  int64_t need = (P.n4 + kThreads - 1) / kThreads;        // the zeroing pass covers the whole arena
  (void)slice4;
  int grid = int(need < ctx->sm_count ? need : ctx->sm_count);
  if (grid < 1) grid = 1;
  void* args[] = {(void*)&P};
  BRK_CUDA(cudaLaunchCooperativeKernel((void*)dp_adam_peer_kernel, dim3(grid), dim3(kThreads), args, 0,
                                       (cudaStream_t)stream));
  return 0;
}

extern "C" int brk_allreduce_dense_peer(brk_ctx* ctx, float* const* peer_buf, uint32_t* const* peer_flags, uint32_t* local_sync,
                                        int64_t n, int32_t rank, int32_t world, void* stream) {
  BRK_REQUIRE(ctx && peer_buf && peer_flags && local_sync, BRK_E_ARG, "brk_allreduce_dense_peer: null argument");
  BRK_REQUIRE(world >= 1 && world <= 64 && rank >= 0 && rank < world && n > 0 && (n & 3) == 0, BRK_E_ARG,
              "brk_allreduce_dense_peer: world=%d rank=%d n=%lld (n must be a multiple of 4)", world, rank, (long long)n);
  const int64_t n4 = n / 4;
  const int64_t need = (n4 / world + kThreads) / kThreads;
  int grid = int(need < ctx->sm_count ? need : ctx->sm_count);
  if (grid < 1) grid = 1;
  long long budget = spin_budget_cycles();
  void* args[] = {(void*)&peer_buf, (void*)&peer_flags, (void*)&local_sync, (void*)&n4, (void*)&rank, (void*)&world, (void*)&budget};
  // every CTA spins on a flag another CTA sets: they must be co-resident -> cooperative launch
  BRK_CUDA(cudaLaunchCooperativeKernel((void*)allreduce_peer_kernel, dim3(grid), dim3(kThreads), args, 0, (cudaStream_t)stream));
  return 0;
}

extern "C" int brk_peer_barrier(brk_ctx* ctx, uint32_t* const* peer_flags, uint32_t* local_sync, int32_t rank,
                                int32_t world, void* stream) {
  BRK_REQUIRE(ctx && peer_flags && local_sync, BRK_E_ARG, "brk_peer_barrier: null argument");
  BRK_REQUIRE(world >= 1 && world <= 64 && rank >= 0 && rank < world, BRK_E_ARG, "brk_peer_barrier: rank=%d world=%d",
              rank, world);
  peer_barrier_kernel<<<1, 64, 0, (cudaStream_t)stream>>>(peer_flags, local_sync, rank, world, spin_budget_cycles());
  BRK_LAUNCH_CHECK();
  return 0;
}
