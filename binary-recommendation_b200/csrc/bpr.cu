// Fused BPR triplet forward + backward (K1+K4+K5 in one pass; no activations ever reach HBM).
// Reference graph: /root/reference/src/models/BPRModel.py:49-74, loss :124-144 (1 - sigmoid).
// Per triplet: 3 rows gathered (3*4d B) and 3 row gradients reduced into the dense accumulators
// (3*4d B of RED traffic) => 1536 B of algorithmic traffic at d = 64.
// Mapping: a group of LPR lanes owns a triplet, each lane holds NCH float4 chunks of u, p and n in
// registers; the dot product is a group shuffle-reduction; gradients leave as 16-byte vector REDs.
#include "neumf_common.cuh"      // TabRef / locate / mark_row: row-sharded table addressing
#include <stdlib.h>
#include <vector>

namespace {

constexpr int kThreads = 256;

// Touched-row bitmask: the word is read early (plain load, issued with the row loads; a stale
// value only costs a redundant RED) and the bit is set with a fire-and-forget RED.OR.
__device__ __forceinline__ uint32_t peek_touched(const uint32_t* touched, int64_t row) {
  return touched ? __ldg(touched + (row >> 5)) : 0xffffffffu;
}
__device__ __forceinline__ void mark_touched(uint32_t* touched, int64_t row, uint32_t seen) {
  const uint32_t bit = 1u << (row & 31);
  if (!(seen & bit)) atomicOr(touched + (row >> 5), bit);
}

// Adds this block's partial loss; the last block to arrive publishes the mean and resets the slot.
__device__ __forceinline__ void finish_loss(double part, double inv_batch, double* acc, unsigned int* ticket,
                                            float* loss_out) {
  __shared__ double red[32];
  const double tot = block_sum_double(part, red);
  if (threadIdx.x == 0) {
    atomicAdd(acc, tot);
    __threadfence();
    const unsigned int t = atomicAdd(ticket, 1u);
    if (t == gridDim.x - 1) {
      __threadfence();
      const double sum = atomicAdd(acc, 0.0);
      if (loss_out) loss_out[0] = float(sum * inv_batch);
      *acc = 0.0;
      *ticket = 0u;
      __threadfence();
    }
  }
}

template <int LPR, int NCH, bool TRAIN>
__global__ void __launch_bounds__(kThreads)
bpr_vec(const float* __restrict__ Wu, const float* __restrict__ Wi, float* __restrict__ Gu,
        float* __restrict__ Gi, uint32_t* __restrict__ Tu, uint32_t* __restrict__ Ti, int d4,
        const int32_t* __restrict__ uid, const int32_t* __restrict__ pid, const int32_t* __restrict__ nid,
        int64_t batch, float inv_batch, double inv_local, double* loss_acc, unsigned int* ticket, float* __restrict__ out) {
  constexpr int GPW = 32 / LPR;  // groups (triplets) per warp
  const int lane_in = threadIdx.x & (LPR - 1);
  const int64_t group = (int64_t(blockIdx.x) * kThreads + threadIdx.x) / LPR;
  const int64_t n_groups = int64_t(gridDim.x) * kThreads / LPR;
  const int64_t warp_first = group - ((threadIdx.x & 31) / LPR);  // first triplet of this warp
  const float4* __restrict__ Wu4 = reinterpret_cast<const float4*>(Wu);
  const float4* __restrict__ Wi4 = reinterpret_cast<const float4*>(Wi);
  float loss_local = 0.f;

  for (int64_t wb = warp_first; wb < batch; wb += n_groups) {
    const int64_t b = wb + (threadIdx.x & 31) / LPR;
    const bool valid = b < batch;
    int64_t ru = 0, rp = 0, rn = 0;
    if (valid) { ru = __ldg(uid + b); rp = __ldg(pid + b); rn = __ldg(nid + b); }
    uint32_t su = 0xffffffffu, sp = 0xffffffffu, sn = 0xffffffffu;
    if (TRAIN && valid && lane_in == 0) { su = peek_touched(Tu, ru); sp = peek_touched(Ti, rp); sn = peek_touched(Ti, rn); }
    float4 u[NCH], p[NCH], n[NCH];
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const int c = lane_in + k * LPR;
      if (valid && c < d4) {
        u[k] = __ldg(Wu4 + ru * d4 + c);
        p[k] = __ldg(Wi4 + rp * d4 + c);
        n[k] = __ldg(Wi4 + rn * d4 + c);
      } else {
        u[k] = p[k] = n[k] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    float dot = 0.f;
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      // difference first, then the product: mirrors x = <u,p> - <u,n> up to fp32 reassociation
      dot = fmaf(u[k].x, p[k].x - n[k].x, dot);
      dot = fmaf(u[k].y, p[k].y - n[k].y, dot);
      dot = fmaf(u[k].z, p[k].z - n[k].z, dot);
      dot = fmaf(u[k].w, p[k].w - n[k].w, dot);
    }
    const float x = group_sum<LPR>(dot);
    if constexpr (!TRAIN) {
      if (valid && lane_in == 0) out[b] = x;
    } else {
      const float s = sigmoidf_acc(x);
      if (valid && lane_in == 0) loss_local += 1.0f - s;
      const float g = -s * (1.0f - s) * inv_batch;
      if (valid) {
#pragma unroll
        for (int k = 0; k < NCH; ++k) {
          const int c = lane_in + k * LPR;
          if (c < d4) {
            const float4 du = make_float4(g * (p[k].x - n[k].x), g * (p[k].y - n[k].y),
                                          g * (p[k].z - n[k].z), g * (p[k].w - n[k].w));
            const float4 dp = make_float4(g * u[k].x, g * u[k].y, g * u[k].z, g * u[k].w);
            const float4 dn = make_float4(-dp.x, -dp.y, -dp.z, -dp.w);
            red_add_f4(Gu + (ru * d4 + c) * 4, du);
            red_add_f4(Gi + (rp * d4 + c) * 4, dp);
            red_add_f4(Gi + (rn * d4 + c) * 4, dn);
          }
        }
        if (lane_in == 0) { mark_touched(Tu, ru, su); mark_touched(Ti, rp, sp); mark_touched(Ti, rn, sn); }
      }
    }
  }
  (void)GPW;
  if constexpr (TRAIN) finish_loss(double(loss_local), inv_local, loss_acc, ticket, out);
}

// Row-sharded tables (row r on rank r % world, local row r / world; peer shards are NVLink mappings): the same
// fused triplet kernel with every row address resolved through the shard table -- peer rows are gathered with
// ordinary loads, the three row gradients leave as 16-byte REDs into the owners' accumulators.
template <int LPR, int NCH>
__global__ void __launch_bounds__(kThreads)
bpr_vec_sharded(const v2::TabRef TU, const v2::TabRef TI, int d4, const int32_t* __restrict__ uid,
                const int32_t* __restrict__ pid, const int32_t* __restrict__ nid, int64_t batch, float inv_batch,
                double inv_local, double* loss_acc, unsigned int* ticket, float* __restrict__ out) {
  const int lane_in = threadIdx.x & (LPR - 1);
  const int64_t group = (int64_t(blockIdx.x) * kThreads + threadIdx.x) / LPR;
  const int64_t n_groups = int64_t(gridDim.x) * kThreads / LPR;
  const int64_t warp_first = group - ((threadIdx.x & 31) / LPR);
  float loss_local = 0.f;
  auto locate = [&](const v2::TabRef& T, int64_t row) {
    int o = 0; int64_t l = row;
    if (T.world > 1) { o = int(row % T.world); l = row / T.world; }
    v2::RowRef r; r.w = T.w[o] + l * d4 * 4; r.g = T.g[o] + l * d4 * 4; r.t = T.t[o]; r.lrow = l;
    return r;
  };
  for (int64_t wb = warp_first; wb < batch; wb += n_groups) {
    const int64_t b = wb + (threadIdx.x & 31) / LPR;
    const bool valid = b < batch;
    v2::RowRef ru, rp, rn;
    ru = rp = rn = locate(TU, 0);
    if (valid) { ru = locate(TU, __ldg(uid + b)); rp = locate(TI, __ldg(pid + b)); rn = locate(TI, __ldg(nid + b)); }
    float4 u[NCH], p[NCH], n[NCH];
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const int c = lane_in + k * LPR;
      if (valid && c < d4) {
        u[k] = __ldg(reinterpret_cast<const float4*>(ru.w) + c);
        p[k] = __ldg(reinterpret_cast<const float4*>(rp.w) + c);
        n[k] = __ldg(reinterpret_cast<const float4*>(rn.w) + c);
      } else {
        u[k] = p[k] = n[k] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    float dot = 0.f;
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      dot = fmaf(u[k].x, p[k].x - n[k].x, dot); dot = fmaf(u[k].y, p[k].y - n[k].y, dot);
      dot = fmaf(u[k].z, p[k].z - n[k].z, dot); dot = fmaf(u[k].w, p[k].w - n[k].w, dot);
    }
    const float x = group_sum<LPR>(dot);
    const float s = sigmoidf_acc(x);
    if (valid && lane_in == 0) loss_local += 1.0f - s;
    const float g = -s * (1.0f - s) * inv_batch;
    if (valid) {
#pragma unroll
      for (int k = 0; k < NCH; ++k) {
        const int c = lane_in + k * LPR;
        if (c < d4) {
          const float4 dp = make_float4(g * u[k].x, g * u[k].y, g * u[k].z, g * u[k].w);
          red_add_f4(ru.g + c * 4, make_float4(g * (p[k].x - n[k].x), g * (p[k].y - n[k].y), g * (p[k].z - n[k].z),
                                               g * (p[k].w - n[k].w)));
          red_add_f4(rp.g + c * 4, dp);
          red_add_f4(rn.g + c * 4, make_float4(-dp.x, -dp.y, -dp.z, -dp.w));
        }
      }
      if (lane_in == 0) { v2::mark_row(ru); v2::mark_row(rp); v2::mark_row(rn); }
    }
  }
  finish_loss(double(loss_local), inv_local, loss_acc, ticket, out);
}

// Generic width (d % 4 != 0 or unaligned): one warp per triplet, rows re-read for the backward.
template <bool TRAIN>
__global__ void __launch_bounds__(kThreads)
bpr_scalar(const float* __restrict__ Wu, const float* __restrict__ Wi, float* __restrict__ Gu,
           float* __restrict__ Gi, uint32_t* __restrict__ Tu, uint32_t* __restrict__ Ti, int d,
           const int32_t* __restrict__ uid, const int32_t* __restrict__ pid, const int32_t* __restrict__ nid,
           int64_t batch, float inv_batch, double inv_local, double* loss_acc, unsigned int* ticket, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t(blockIdx.x) * kThreads + threadIdx.x) >> 5;
  const int64_t n_warps = int64_t(gridDim.x) * kThreads >> 5;
  float loss_local = 0.f;
  for (int64_t b = warp; b < batch; b += n_warps) {
    const int64_t ru = __ldg(uid + b), rp = __ldg(pid + b), rn = __ldg(nid + b);
    uint32_t su = 0xffffffffu, sp = 0xffffffffu, sn = 0xffffffffu;
    if (TRAIN && lane == 0) { su = peek_touched(Tu, ru); sp = peek_touched(Ti, rp); sn = peek_touched(Ti, rn); }
    float dot = 0.f;
    for (int c = lane; c < d; c += 32)
      dot = fmaf(__ldg(Wu + ru * d + c), __ldg(Wi + rp * d + c) - __ldg(Wi + rn * d + c), dot);
    const float x = warp_sum(dot);
    if constexpr (!TRAIN) {
      if (lane == 0) out[b] = x;
    } else {
      const float s = sigmoidf_acc(x);
      if (lane == 0) loss_local += 1.0f - s;
      const float g = -s * (1.0f - s) * inv_batch;
      for (int c = lane; c < d; c += 32) {
        const float uu = __ldg(Wu + ru * d + c), pp = __ldg(Wi + rp * d + c), nn = __ldg(Wi + rn * d + c);
        atomicAdd(Gu + ru * d + c, g * (pp - nn));
        atomicAdd(Gi + rp * d + c, g * uu);
        atomicAdd(Gi + rn * d + c, -g * uu);
      }
      if (lane == 0) { mark_touched(Tu, ru, su); mark_touched(Ti, rp, sp); mark_touched(Ti, rn, sn); }
    }
  }
  if constexpr (TRAIN) finish_loss(double(loss_local), inv_local, loss_acc, ticket, out);
}

// ---- whole training steps in ONE cooperative kernel ------------------------------------------------
// K steps x (fused fwd/bwd -> grid barrier -> exact Keras Adam over both tables -> grid barrier): no kernel
// launch and no host involvement between steps; both phases are single-wave and latency-bound, so the
// launch gaps and cold starts between separate kernels were ~40 % of the step.
// Sampling mode (P.n == nullptr): the kernel draws its own Philox negatives.  Two warps of every CTA
// spend the Adam phase of step s staging step s+1 -- ids copied from P.u / P.p (which may be MAPPED HOST
// memory: this is where the PCIe reads happen) into a device ring, negatives sampled next to them --
// while the other six warps run Adam, so neither the binary search in the positive lists nor the PCIe
// latency is on the step's critical path (only step 0 is staged up front).
struct BprStep {                   // one training step of a cooperative launch
  int64_t off;                     // first triplet of the step inside P.u / P.p / P.n
  int64_t sample_index;            // Philox sample index of that triplet (sampling mode)
  int32_t count;                   // triplets in the step (ragged tail batches are shorter)
  int32_t _pad;
};
constexpr int kInlineSteps = 16;
struct BprCoopParams {
  brk_table user, item;
  const int32_t* u; const int32_t* p; const int32_t* n;
  const BprStep* steps;           // device [n_steps] (long calls) ...
  BprStep inline_steps[kInlineSteps];   // ... or by value (n_steps <= 16: no H2D copy at all)
  int32_t use_inline;
  int32_t n_steps;
  brk_adam_hyper h;
  int64_t* state;                 // [t, beta1^t, beta2^t]
  float* losses;                  // [n_steps] or null; device memory or mapped page-locked host memory
  double* loss_acc;               // 2 doubles (ping-pong), zero on entry
  // sampling mode
  int32_t* stage;                 // device [2][3][stage_pitch]: u, p, n of the step being staged / consumed
  int64_t stage_pitch;
  const int64_t* csr_indptr; const int32_t* csr_items;
  uint32_t seed, epoch, num_items;
  // mirrored data parallelism (world > 1): both tables' w and g are views into per-rank arenas in NVLink
  // peer-mapped memory; phase 2 becomes barrier -> reduce my slice over all ranks' g -> Adam -> write the new
  // weights into every rank's arena -> barrier (csrc/dp_peer.cu, here inside the multi-step kernel)
  float* const* peer_w; float* const* peer_g; uint32_t* const* peer_flags;
  float* dp_m; float* dp_v; uint32_t* dp_sync;
  int64_t arena_n4;
  int32_t rank, world;
  float inv_global;               // 1 / (world * batch): gradient scale of the global mean loss
  // optional [n_steps][8] globaltimer stamps of block 0 (BRK_COOP_TRACE).  world == 1: 0 step start, 2 phase 1 done,
  // 1 gradient barrier passed, 3 Adam done, 6 trailing barrier passed (= 3 when skipped); step 0 also holds 7 kernel entry
  // and, in word 4, 1 if the Adam ran from shared memory (0: global memory).  world > 1: see profiles/dp_trace.py.
  unsigned long long* dbg;
  long long spin_budget;          // clock64 budget of one cross-GPU wait (default ~30 s; BRK_PEER_SPIN_MS)
  unsigned int* bar;              // grid-barrier words {count, error, base} (common.cuh)
  // Adam operands in shared memory (world == 1): CTA b owns float4 [b * slice4[k], (b + 1) * slice4[k]) of table k's
  // w / m / v / g; 0 = Adam straight from global memory (slices too large, or BRK_BPR_NO_SMEM_ADAM=1)
  int32_t slice4[2];
  int32_t last_sync;              // 1: grid barrier after the launch's last step too (only BRK_BPR_NO_SMEM_ADAM=1 keeps it)
};

__device__ __forceinline__ void coop_st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ bool coop_spin_sys(const uint32_t* p, uint32_t epoch, uint32_t* err, long long budget) {
  const long long t0 = clock64();
  while (true) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    if (int32_t(v - epoch) >= 0) return true;
    if (clock64() - t0 > budget) { atomicExch(err, 1u); return false; }            // a peer never arrived
    __nanosleep(32);
  }
}

__device__ __forceinline__ void coop_stamp(const BprCoopParams& P, int s, int k) {
  if (P.dbg && blockIdx.x == 0 && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    P.dbg[s * 8 + k] = t;
  }
}

__device__ __forceinline__ void adam4(float4& w, float4& m, float4& v, const float4 g, float alpha, float b1, float b2,
                                      float eps) {
  const float omb1 = 1.f - b1, omb2 = 1.f - b2;
  m.x = b1 * m.x + omb1 * g.x; v.x = b2 * v.x + omb2 * g.x * g.x; w.x -= alpha * m.x / (sqrtf(v.x) + eps);
  m.y = b1 * m.y + omb1 * g.y; v.y = b2 * v.y + omb2 * g.y * g.y; w.y -= alpha * m.y / (sqrtf(v.y) + eps);
  m.z = b1 * m.z + omb1 * g.z; v.z = b2 * v.z + omb2 * g.z * g.z; w.z -= alpha * m.z / (sqrtf(v.z) + eps);
  m.w = b1 * m.w + omb1 * g.w; v.w = b2 * v.w + omb2 * g.w * g.w; w.w -= alpha * m.w / (sqrtf(v.w) + eps);
}

// Stage one step: ids into the device ring, one Philox negative per triplet (thread-per-triplet).
__device__ __forceinline__ void bpr_stage_step(const BprCoopParams& P, const BprStep sd, int slot, int64_t tid, int64_t nthr) {
  int32_t* su = P.stage + int64_t(slot) * 3 * P.stage_pitch;
  int32_t* sp = su + P.stage_pitch; int32_t* sn = sp + P.stage_pitch;
  for (int64_t b = tid; b < sd.count; b += nthr) {
    const int32_t uu = P.u[sd.off + b];
    su[b] = uu; sp[b] = P.p[sd.off + b];
    sn[b] = brk_sample_bpr_negative(uint64_t(sd.sample_index + b), uu, P.seed, P.epoch, P.num_items, P.csr_indptr, P.csr_items);
  }
}

constexpr int kStageThreads = 64;   // threads per CTA that stage the next step during the Adam phase

__device__ __forceinline__ bool coop_mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
               : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}

template <int LPR, int NCH>
__global__ void __launch_bounds__(kThreads, 4) bpr_steps_coop(const BprCoopParams P) {
  unsigned int bar_target = *reinterpret_cast<volatile unsigned int*>(P.bar + 2);
  // Data parallel: in front of a cross-GPU flag exchange only block 0 has to know that every local block has arrived (it is
  // the one that tells the peers); the other blocks go straight on to poll the flags -- their own rank's flag among them,
  // which block 0 posts after this collection -- so the second half of a full barrier (everybody spinning on the counter)
  // is not paid twice per step.
  auto gcollect = [&]() {
    brk_grid_arrive(P.bar, bar_target);
    if (blockIdx.x == 0) {
      brk_grid_wait(P.bar, bar_target);
      __syncthreads();
    }
  };
  __shared__ double red[32];
  const bool sample = P.n == nullptr;
  const int d4 = P.user.d >> 2;
  const int lane_in = threadIdx.x & (LPR - 1);
  const int sub = (threadIdx.x & 31) / LPR;
  // 32-bit thread and group indices (a cooperative grid is a few hundred CTAs): the kernel runs at its 64-register bound
  const int group = int(blockIdx.x * kThreads + threadIdx.x) / LPR;
  const int n_groups = int(gridDim.x) * kThreads / LPR;
  const int warp_first = group - sub;
  const int tid = int(blockIdx.x * kThreads + threadIdx.x), nthr = int(gridDim.x) * kThreads;
  // no __restrict__/read-only path here: phase 2 of this same kernel rewrites the tables, so rows are
  // read with ld.global.cg (L2 only) -- another SM's L1 could otherwise hold a stale line across steps
  const float4* Wu4 = reinterpret_cast<const float4*>(P.user.w);
  const float4* Wi4 = reinterpret_cast<const float4*>(P.item.w);
  const double* pw = reinterpret_cast<const double*>(P.state);
  // Running beta powers, advanced once per step: step s reads pair s & 1 and thread 0 writes pair (s + 1) & 1, which no
  // thread reads again before the next __syncthreads.  Shared rather than registers: the kernel runs at its register bound.
  __shared__ double beta_pow[2][2];
  if (threadIdx.x == 0) { beta_pow[0][0] = pw[1]; beta_pow[0][1] = pw[2]; }
  const brk_table tabs[2] = {P.user, P.item};

  // The whole optimizer state is asked into L2 up front with BULK prefetches (one instruction per CTA and array slice,
  // streamed by the copy engine of the SM): when other work has evicted the 10 MB since the last launch -- bench.py's
  // flushed-L2 measurement is exactly that -- phase 2 of the first step otherwise starts on cold m / v / g lines.
  // (Per-line prefetch.global.L2, 80 k requests, cost more than it hid: section 4.3 of DESIGN.md.)
  // With the shared-memory Adam (P.slice4) the CTA's slices of w, m and v are instead bulk-copied into its shared memory
  // (the same one instruction per array slice, completing on `adam_bar`): they stream in while phase 1 runs, phase 1 only
  // reads w from global memory and never m or v, and the first Adam phase waits for them.  g keeps its L2 prefetch.
  // Shared layout: [w | m | v], each nA float4 = this CTA's user slice followed by its item slice.
  extern __shared__ float4 adam_smem[];
  __shared__ __align__(8) uint64_t adam_bar;
  const bool smem_adam = P.slice4[0] > 0;
  coop_stamp(P, 0, 7);
  if (P.dbg && P.world == 1 && blockIdx.x == 0 && threadIdx.x == 0) P.dbg[4] = smem_adam ? 1u : 0u;   // which Adam ran
  if (threadIdx.x == 0) {
    const uint32_t bar = uint32_t(__cvta_generic_to_shared(&adam_bar));
    if (smem_adam) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
      asm volatile("fence.mbarrier_init.release.cluster;\n\tfence.proxy.async.shared::cta;" ::: "memory");
    }
    uint32_t nb[2], tx = 0;
    int64_t offs[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int64_t bytes = tabs[k].rows * tabs[k].d * 4;
      int64_t per = smem_adam ? int64_t(P.slice4[k]) * 16 : (bytes + gridDim.x - 1) / gridDim.x;
      per = (per + 15) & ~int64_t(15);
      offs[k] = int64_t(blockIdx.x) * per;
      nb[k] = offs[k] < bytes ? uint32_t((offs[k] + per <= bytes ? per : bytes - offs[k]) & ~int64_t(15)) : 0u;
      tx += nb[k];
    }
    if (smem_adam) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(3 * tx) : "memory");
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (nb[k] == 0) continue;
      const float* arrs[4] = {tabs[k].g, tabs[k].w, P.world > 1 ? nullptr : tabs[k].m, P.world > 1 ? nullptr : tabs[k].v};
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const char* src = reinterpret_cast<const char*>(arrs[a]) + offs[k];
        if (smem_adam && a > 0) {
          const uint32_t dst = uint32_t(__cvta_generic_to_shared(adam_smem)) + (a - 1) * tx + (k ? nb[0] : 0u);
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                       ::"r"(dst), "l"(src), "r"(nb[k]), "r"(bar) : "memory");
        } else if (arrs[a] != nullptr && brk_aligned16(arrs[a])) {
          asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(nb[k]) : "memory");
        }
      }
    }
  }
  if (sample) {                                         // step 0 is staged by everybody, up front
    bpr_stage_step(P, P.use_inline ? P.inline_steps[0] : P.steps[0], 0, tid, nthr);
    brk_grid_barrier(P.bar, bar_target);
  }
  for (int s = 0; s < P.n_steps; ++s) {
    const BprStep sd = P.use_inline ? P.inline_steps[s] : P.steps[s];
    const int64_t batch = sd.count;
    const float inv_batch = P.world > 1 ? P.inv_global : 1.0f / float(batch);
    coop_stamp(P, s, 0);
    const int32_t *uid, *pid, *nid;
    if (sample) { uid = P.stage + int64_t(s & 1) * 3 * P.stage_pitch; pid = uid + P.stage_pitch; nid = pid + P.stage_pitch; }
    else { uid = P.u + sd.off; pid = P.p + sd.off; nid = P.n + sd.off; }
    // ---- phase 1: fused gather + loss + gradient REDs (same math as bpr_vec) ----
    float loss_local = 0.f;
    for (int wb = warp_first; wb < batch; wb += n_groups) {
      const int b = wb + sub;
      const bool valid = b < batch;
      int64_t ru = 0, rp = 0, rn = 0;
      if (valid) { ru = __ldcg(uid + b); rp = __ldcg(pid + b); rn = __ldcg(nid + b); }
      float4 u[NCH], p[NCH], n[NCH];
#pragma unroll
      for (int k = 0; k < NCH; ++k) {
        const int c = lane_in + k * LPR;
        if (valid && c < d4) {           // L2-only loads: the tables are rewritten by phase 2 of the same kernel
          u[k] = __ldcg(Wu4 + ru * d4 + c); p[k] = __ldcg(Wi4 + rp * d4 + c); n[k] = __ldcg(Wi4 + rn * d4 + c);
        } else {
          u[k] = p[k] = n[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      float dot = 0.f;
#pragma unroll
      for (int k = 0; k < NCH; ++k) {
        dot = fmaf(u[k].x, p[k].x - n[k].x, dot); dot = fmaf(u[k].y, p[k].y - n[k].y, dot);
        dot = fmaf(u[k].z, p[k].z - n[k].z, dot); dot = fmaf(u[k].w, p[k].w - n[k].w, dot);
      }
      const float x = group_sum<LPR>(dot);
      const float sg = sigmoidf_acc(x);
      if (valid && lane_in == 0) loss_local += 1.0f - sg;
      const float g = -sg * (1.0f - sg) * inv_batch;
      if (valid) {
#pragma unroll
        for (int k = 0; k < NCH; ++k) {
          const int c = lane_in + k * LPR;
          if (c < d4) {
            const float4 dp = make_float4(g * u[k].x, g * u[k].y, g * u[k].z, g * u[k].w);
            red_add_f4(P.user.g + (ru * d4 + c) * 4, make_float4(g * (p[k].x - n[k].x), g * (p[k].y - n[k].y),
                                                                 g * (p[k].z - n[k].z), g * (p[k].w - n[k].w)));
            red_add_f4(P.item.g + (rp * d4 + c) * 4, dp);
            red_add_f4(P.item.g + (rn * d4 + c) * 4, make_float4(-dp.x, -dp.y, -dp.z, -dp.w));
          }
        }
      }
    }
    const double part = block_sum_double(double(loss_local), red);
    if (threadIdx.x == 0) atomicAdd(P.loss_acc + (s & 1), part);
    if (P.world > 1) {
      gcollect();
    } else {
      coop_stamp(P, s, 2);                              // phase 1 done in block 0
      brk_grid_barrier(P.bar, bar_target);
    }
    coop_stamp(P, s, 1);
    // ---- phase 2: exact Keras Adam over every element of both tables; zero the accumulators.  In sampling
    //      mode the first two warps of each CTA stage step s+1 instead (ids + negatives) ----
    const double p1 = beta_pow[s & 1][0] * double(P.h.beta1), p2 = beta_pow[s & 1][1] * double(P.h.beta2);
    if (threadIdx.x == 0) { beta_pow[(s + 1) & 1][0] = p1; beta_pow[(s + 1) & 1][1] = p2; }
    const float alpha = float(double(P.h.lr) * sqrt(1.0 - p2) / (1.0 - p1));
    const bool staging = sample && s + 1 < P.n_steps;
    const bool stager = staging && threadIdx.x < kStageThreads;
    const int atid = staging ? int(blockIdx.x) * (kThreads - kStageThreads) + (int(threadIdx.x) - kStageThreads) : tid;
    const int anthr = staging ? int(gridDim.x) * (kThreads - kStageThreads) : nthr;
    if (stager) {
      bpr_stage_step(P, P.use_inline ? P.inline_steps[s + 1] : P.steps[s + 1], (s + 1) & 1,
                     int64_t(blockIdx.x) * kStageThreads + threadIdx.x, int64_t(gridDim.x) * kStageThreads);
    }
    if (P.world == 1 && smem_adam) {
      // This CTA's slices only: w, m, v from shared memory (the entry copies, then what the previous step left there),
      // g from L2 where the REDs landed; the new w goes to global memory for the next step's gathers and to shared
      // memory, m and v stay on chip until the end of the launch.
      if (s == 0) {
        const uint32_t bar = uint32_t(__cvta_generic_to_shared(&adam_bar));
        while (!coop_mbar_try_wait(bar, 0)) {}
      }
      if (!stager) {
        int64_t o4[2];
        int n4[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const int64_t tot = tabs[k].rows * tabs[k].d / 4;
          o4[k] = int64_t(blockIdx.x) * P.slice4[k];
          n4[k] = o4[k] < tot ? int(tot - o4[k] < P.slice4[k] ? tot - o4[k] : P.slice4[k]) : 0;
        }
        const int nA = n4[0] + n4[1];
        float4* sw = adam_smem; float4* sm = sw + nA; float4* sv = sm + nA;
        const int t0 = staging ? int(threadIdx.x) - kStageThreads : int(threadIdx.x);
        const int T = staging ? kThreads - kStageThreads : kThreads;
        // One element at a time.  Issuing a thread's two g loads before either update (a CTA owns 265 float4 for 256
        // threads at the bench shape) fits the 64 registers only with per-step recomputation elsewhere, and measured
        // slower: Adam phase 2.1 -> 2.8 us, 600-step hot launch 1.45 -> 1.38 G interactions/s (DESIGN.md 7.1).
        for (int j = t0; j < nA; j += T) {
          const bool u = j < n4[0];
          float4* w4 = reinterpret_cast<float4*>(u ? P.user.w : P.item.w) + (u ? o4[0] + j : o4[1] + (j - n4[0]));
          float4* g4 = reinterpret_cast<float4*>(u ? P.user.g : P.item.g) + (u ? o4[0] + j : o4[1] + (j - n4[0]));
          float4 w = sw[j], m = sm[j], v = sv[j];
          adam4(w, m, v, __ldcg(g4), alpha, P.h.beta1, P.h.beta2, P.h.eps);
          sw[j] = w; sm[j] = m; sv[j] = v;
          *w4 = w; *g4 = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    } else if (P.world == 1) {
      if (!stager) {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const int64_t n4 = tabs[k].rows * tabs[k].d / 4;
          float4* w4 = reinterpret_cast<float4*>(tabs[k].w); float4* g4 = reinterpret_cast<float4*>(tabs[k].g);
          float4* m4 = reinterpret_cast<float4*>(tabs[k].m); float4* v4 = reinterpret_cast<float4*>(tabs[k].v);
          for (int64_t i = atid; i < n4; i += anthr) {
            float4 w = w4[i], m = m4[i], v = v4[i];
            adam4(w, m, v, g4[i], alpha, P.h.beta1, P.h.beta2, P.h.eps);
            w4[i] = w; m4[i] = m; v4[i] = v; g4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
      }
    } else {
      // ---- data-parallel phase 2 over NVLink peer memory ----
      const int G = P.world, me = P.rank;
      const uint32_t ep = P.dp_sync[3] + uint32_t(s) + 1u;      // dp_sync[3]: epochs completed before this launch
      uint32_t* my_flags = P.peer_flags[me];
      // barrier A: every rank's gradients are complete.  Block 0 posts this rank's arrival on every peer; EVERY block
      // then polls this rank's own flag block (local L2), which saves a second grid-wide barrier
      if (blockIdx.x == 0 && threadIdx.x < G) {
        __threadfence_system();
        coop_st_release_sys(P.peer_flags[threadIdx.x] + me, ep);
      }
      // A peer that never arrives ABORTS the exchange on this rank: no reduce over incomplete gradients, no Adam, no
      // pull; the sticky error word dp_sync[4] ends the launch at the next step boundary and PeerArena.check() raises.
      bool okA = true;
      if (threadIdx.x < G) okA = coop_spin_sys(my_flags + threadIdx.x, ep, P.dp_sync + 4, P.spin_budget);
      const bool deadA = __syncthreads_or(okA ? 0 : 1) != 0 || *reinterpret_cast<volatile uint32_t*>(P.dp_sync + 4) != 0u;
      coop_stamp(P, s, 2);
      if (!stager && !deadA) {
        const int64_t lo = P.arena_n4 * me / G, hi = P.arena_n4 * (me + 1) / G;
        float4* w_me = reinterpret_cast<float4*>(P.peer_w[me]);
        float4* m4 = reinterpret_cast<float4*>(P.dp_m); float4* v4 = reinterpret_cast<float4*>(P.dp_v);
        for (int64_t i = lo + atid; i < hi; i += anthr) {
          float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
          for (int p = 0; p < G; ++p) {                          // fixed order: every rank computes the same sum
            const float4 x = __ldcg(reinterpret_cast<const float4*>(P.peer_g[p]) + i);
            g.x += x.x; g.y += x.y; g.z += x.z; g.w += x.w;
          }
          float4 w = __ldcg(w_me + i), m = m4[i - lo], v = v4[i - lo];
          adam4(w, m, v, g, alpha, P.h.beta1, P.h.beta2, P.h.eps);
          m4[i - lo] = m; v4[i - lo] = v;
          w_me[i] = w;                                           // my slice, my arena only: the peers pull it below
        }
      }
      coop_stamp(P, s, 3);
      __threadfence();
      gcollect();
      coop_stamp(P, s, 4);
      const bool deadG = *reinterpret_cast<volatile uint32_t*>(P.dp_sync + 4) != 0u;   // sticky error word of an earlier time-out
      if (!deadG && blockIdx.x == 0 && threadIdx.x < G) {       // barrier B: every rank's slice is final, reads of my g are done
        __threadfence_system();
        coop_st_release_sys(P.peer_flags[threadIdx.x] + G + me, ep);
      }
      bool okB = true;
      if (!deadG && threadIdx.x < G) okB = coop_spin_sys(my_flags + G + threadIdx.x, ep, P.dp_sync + 4, P.spin_budget);
      const bool deadB = __syncthreads_or(okB ? 0 : 1) != 0 || deadG;
      coop_stamp(P, s, 5);
      // all-gather by PULL: remote loads complete when their data arrives, so nothing has to wait for NVLink write
      // acknowledgements (pushing the slices and fencing them system-wide cost ~8 us per step); zero my g meanwhile
      if (!deadB) {
        float4* w_loc = reinterpret_cast<float4*>(P.peer_w[me]);
        const int64_t lo = P.arena_n4 * me / G, hi = P.arena_n4 * (me + 1) / G;
        const int64_t others = P.arena_n4 - (hi - lo);
        float4* g_me = reinterpret_cast<float4*>(P.peer_g[me]);             // the zeroing stores go first: they do not wait for
        for (int64_t i = tid; i < P.arena_n4; i += nthr) g_me[i] = make_float4(0.f, 0.f, 0.f, 0.f);   // the NVLink round trip below
        for (int64_t j = tid; j < others; j += nthr) {
          const int64_t i = j < lo ? j : j + (hi - lo);          // skip my own slice
          int owner = int((i * G) / P.arena_n4);
          while (P.arena_n4 * owner / G > i) --owner;
          while (P.arena_n4 * (owner + 1) / G <= i) ++owner;
          w_loc[i] = __ldcg(reinterpret_cast<const float4*>(P.peer_w[owner]) + i);
        }
      }
    }
    if (tid == nthr - 1) {
      if (P.losses) P.losses[s] = float(P.loss_acc[s & 1] / double(batch));
      P.loss_acc[s & 1] = 0.0;
    }
    if (P.world == 1) coop_stamp(P, s, 3);              // Adam done in block 0
    // The barrier orders this step's Adam stores before the next step's gathers.  After the last step kernel completion
    // does that for whatever follows on the stream, so a single-GPU launch ends without it: the barrier counter then gets
    // one arrival round fewer, and bar_target (written to bar[2] below) counts exactly the rounds that ran.
    if (P.world > 1 || s + 1 < P.n_steps || P.last_sync) brk_grid_barrier(P.bar, bar_target);
    coop_stamp(P, s, 6);
    if (P.world > 1 && *reinterpret_cast<volatile uint32_t*>(P.dp_sync + 4) != 0u) break;   // aborted (uniform after the barrier)
  }
  if (smem_adam) {                                      // m and v back to global memory, one bulk store per array slice
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // this thread's shared stores -> visible to the copies
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t nb[2];
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int64_t bytes = tabs[k].rows * tabs[k].d * 4, off = int64_t(blockIdx.x) * P.slice4[k] * 16;
        nb[k] = off < bytes ? uint32_t(bytes - off < int64_t(P.slice4[k]) * 16 ? bytes - off : int64_t(P.slice4[k]) * 16) : 0u;
      }
      const uint32_t base = uint32_t(__cvta_generic_to_shared(adam_smem)), tx = nb[0] + nb[1];
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        if (nb[k] == 0) continue;
        const int64_t off = int64_t(blockIdx.x) * P.slice4[k] * 16;
        float* dsts[2] = {tabs[k].m, tabs[k].v};
#pragma unroll
        for (int a = 0; a < 2; ++a)
          asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                       ::"l"(reinterpret_cast<char*>(dsts[a]) + off), "r"(base + (a + 1) * tx + (k ? nb[0] : 0u)), "r"(nb[k])
                       : "memory");
      }
      asm volatile("cp.async.bulk.commit_group;\n\tcp.async.bulk.wait_group 0;" ::: "memory");
    }
  }
  if (tid == 0 && !(P.world > 1 && *reinterpret_cast<volatile uint32_t*>(P.dp_sync + 4) != 0u)) {
    double* pwo = reinterpret_cast<double*>(P.state);
    P.state[0] += P.n_steps; pwo[1] = beta_pow[P.n_steps & 1][0]; pwo[2] = beta_pow[P.n_steps & 1][1];
    if (P.world > 1) P.dp_sync[3] += uint32_t(P.n_steps);
    P.bar[2] = bar_target;
  }
}

template <bool TRAIN>
int launch_bpr(brk_ctx* ctx, const float* Wu, const float* Wi, float* Gu, float* Gi, uint32_t* Tu, uint32_t* Ti,
               int d, const int32_t* u, const int32_t* p, const int32_t* n, int64_t batch, int64_t global_batch,
               float* out, cudaStream_t st) {
  // gradients are scaled by 1/global_batch (data-parallel replicas sum their accumulators); the
  // reported loss is the mean over the local batch
  const float inv_batch = 1.0f / float(global_batch > 0 ? global_batch : batch);
  const double inv_local = 1.0 / double(batch);
  double* acc = ctx->loss_acc + 0;
  unsigned int* ticket = ctx->tickets + 0;
  const int64_t cap = int64_t(ctx->sm_count) * (2048 / kThreads);
  const bool vec = (d & 3) == 0 && d <= 512 && brk_aligned16(Wu) && brk_aligned16(Wi) &&
                   (!TRAIN || (brk_aligned16(Gu) && brk_aligned16(Gi)));
  if (vec) {
    const int d4 = d >> 2;
    const int lpr = brk_lanes_per_row(d4);
    const int nch = (d4 + lpr - 1) / lpr;
    int64_t need = (batch * lpr + kThreads - 1) / kThreads;
    const int grid = int(need < 1 ? 1 : (need < cap ? need : cap));
#define BRK_BPR_CASE(L, N)                                                                          \
  bpr_vec<L, N, TRAIN><<<grid, kThreads, 0, st>>>(Wu, Wi, Gu, Gi, Tu, Ti, d4, u, p, n, batch, inv_batch, \
                                                  inv_local, acc, ticket, out)
    if (lpr == 1) BRK_BPR_CASE(1, 1);
    else if (lpr == 2) BRK_BPR_CASE(2, 1);
    else if (lpr == 4) BRK_BPR_CASE(4, 1);
    else if (lpr == 8) BRK_BPR_CASE(8, 1);
    else if (lpr == 16) BRK_BPR_CASE(16, 1);
    else if (nch == 1) BRK_BPR_CASE(32, 1);
    else if (nch == 2) BRK_BPR_CASE(32, 2);
    else if (nch == 3) BRK_BPR_CASE(32, 3);
    else BRK_BPR_CASE(32, 4);
#undef BRK_BPR_CASE
  } else {
    int64_t need = (batch * 32 + kThreads - 1) / kThreads;
    const int grid = int(need < 1 ? 1 : (need < cap ? need : cap));
    bpr_scalar<TRAIN><<<grid, kThreads, 0, st>>>(Wu, Wi, Gu, Gi, Tu, Ti, d, u, p, n, batch, inv_batch, inv_local,
                                                 acc, ticket, out);
  }
  BRK_LAUNCH_CHECK();
  return 0;
}

}  // namespace

extern "C" int brk_bpr_fwd_bwd(brk_ctx* ctx, const brk_table* user, const brk_table* item,
                               const int32_t* u, const int32_t* p, const int32_t* n, int64_t batch,
                               int64_t global_batch, float* loss_out, void* stream) {
  BRK_REQUIRE(ctx && user && item && u && p && n, BRK_E_ARG, "brk_bpr_fwd_bwd: null argument");
  BRK_REQUIRE(user->w && user->g && item->w && item->g, BRK_E_ARG, "brk_bpr_fwd_bwd: table w/g missing");
  BRK_REQUIRE(user->d == item->d && user->d > 0, BRK_E_ARG, "brk_bpr_fwd_bwd: user d=%d item d=%d", user->d,
              item->d);
  BRK_REQUIRE(batch > 0, BRK_E_ARG, "brk_bpr_fwd_bwd: batch=%lld", (long long)batch);
  return launch_bpr<true>(ctx, user->w, item->w, user->g, item->g, user->touched, item->touched, user->d, u, p,
                          n, batch, global_batch, loss_out, (cudaStream_t)stream);
}

extern "C" int brk_bpr_scores(brk_ctx* ctx, const float* user_w, const float* item_w, int32_t d,
                              const int32_t* u, const int32_t* p, const int32_t* n, int64_t batch,
                              float* x_out, void* stream) {
  BRK_REQUIRE(ctx && user_w && item_w && u && p && n && x_out, BRK_E_ARG, "brk_bpr_scores: null argument");
  BRK_REQUIRE(d > 0 && batch > 0, BRK_E_ARG, "brk_bpr_scores: d=%d batch=%lld", d, (long long)batch);
  return launch_bpr<false>(ctx, user_w, item_w, nullptr, nullptr, nullptr, nullptr, d, u, p, n, batch, 0, x_out,
                           (cudaStream_t)stream);
}

static bool coop_eligible(const brk_table* user, const brk_table* item, int lazy_adam) {
  const int d = user->d;
  return !lazy_adam && (d & 3) == 0 && d <= 128 && user->m && user->v && item->m && item->v &&
         brk_aligned16(user->w) && brk_aligned16(item->w) && brk_aligned16(user->g) && brk_aligned16(item->g) &&
         ((user->rows * d) & 3) == 0 && ((item->rows * d) & 3) == 0 && getenv("BRK_NO_COOP") == nullptr;
}

static unsigned long long* g_coop_trace = nullptr;   // BRK_COOP_TRACE=1: per-step phase stamps of the last launch

struct CoopSampler {                 // fused negative sampling for launch_coop_steps (n == nullptr)
  const int64_t* csr_indptr; const int32_t* csr_items;
  uint32_t seed, epoch, num_items;
};

static int ensure_scratch(brk_ctx* ctx, size_t need) {
  if (ctx->scratch_bytes < need) {
    if (ctx->scratch) BRK_CUDA(cudaFree(ctx->scratch));      // cudaFree waits for the device: no kernel still uses it
    ctx->scratch = nullptr; ctx->scratch_bytes = 0;
    BRK_CUDA(cudaMalloc(&ctx->scratch, need));
    ctx->scratch_bytes = need;
  }
  return 0;
}

// steps_host[k]: off / count / sample_index of step k inside u, p (and n).  max_count: largest step.
static int launch_coop_steps(brk_ctx* ctx, const brk_table* user, const brk_table* item, const int32_t* u,
                             const int32_t* p, const int32_t* n, const BprStep* steps_host, int32_t n_steps,
                             int64_t max_count, brk_adam_hyper h, int64_t* step_dev, float* losses, cudaStream_t st,
                             const CoopSampler* smp = nullptr, const brk_dp_peer* dp = nullptr) {
  const int d = user->d;
  BprCoopParams P;
  P.use_inline = n_steps <= kInlineSteps;
  const size_t steps_bytes = P.use_inline ? 0 : ((size_t(n_steps) * sizeof(BprStep) + 255) & ~size_t(255));
  const int64_t pitch = (max_count + 3) & ~int64_t(3);
  const size_t stage_bytes = smp ? size_t(2) * 3 * pitch * sizeof(int32_t) : 0;
  if (steps_bytes + stage_bytes) { if (int rc = ensure_scratch(ctx, steps_bytes + stage_bytes)) return rc; }
  if (P.use_inline) {
    for (int k = 0; k < n_steps; ++k) P.inline_steps[k] = steps_host[k];
  } else {
    BRK_CUDA(cudaMemcpyAsync(ctx->scratch, steps_host, size_t(n_steps) * sizeof(BprStep), cudaMemcpyHostToDevice, st));
  }
  P.user = *user; P.item = *item; P.u = u; P.p = p; P.n = n;
  P.steps = reinterpret_cast<const BprStep*>(ctx->scratch);
  P.n_steps = n_steps; P.h = h; P.state = step_dev; P.losses = losses;
  P.loss_acc = ctx->loss_acc + 2;
  if (smp) {
    P.stage = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(ctx->scratch) + steps_bytes);
    P.stage_pitch = pitch;
    P.csr_indptr = smp->csr_indptr; P.csr_items = smp->csr_items;
    P.seed = smp->seed; P.epoch = smp->epoch; P.num_items = smp->num_items;
  } else {
    BRK_REQUIRE(n != nullptr, BRK_E_ARG, "brk_bpr_train_steps: negatives missing");
    P.stage = nullptr; P.stage_pitch = 0; P.csr_indptr = nullptr; P.csr_items = nullptr;
    P.seed = P.epoch = P.num_items = 0;
  }
  if (dp && dp->world > 1) {
    P.peer_w = dp->peer_w; P.peer_g = dp->peer_g; P.peer_flags = dp->peer_flags; P.dp_m = dp->m; P.dp_v = dp->v;
    P.dp_sync = dp->local_sync; P.arena_n4 = dp->n / 4; P.rank = dp->rank; P.world = dp->world;
    P.inv_global = 1.0f / float(int64_t(dp->world) * max_count);
  } else {
    P.peer_w = nullptr; P.peer_g = nullptr; P.peer_flags = nullptr; P.dp_m = nullptr; P.dp_v = nullptr; P.dp_sync = nullptr;
    P.arena_n4 = 0; P.rank = 0; P.world = 1; P.inv_global = 0.f;
  }
  if (getenv("BRK_COOP_TRACE") && !g_coop_trace) {
    BRK_CUDA(cudaMalloc(&g_coop_trace, 4096 * 8 * sizeof(unsigned long long)));
    BRK_CUDA(cudaMemset(g_coop_trace, 0, 4096 * 8 * sizeof(unsigned long long)));
  }
  P.dbg = (g_coop_trace && n_steps <= 4096) ? g_coop_trace : nullptr;
  P.bar = ctx->bar[BRK_BAR_BPR];
  {
    const char* e = getenv("BRK_PEER_SPIN_MS");              // budget of one cross-GPU wait; default ~30 s at 2 GHz
    const long long ms = e ? atoll(e) : 0;
    P.spin_budget = ms > 0 ? ms * 2000000LL : 60000000000LL;
  }
  const int lpr = brk_lanes_per_row(d >> 2);
  void* fn = nullptr;
  int slot = 0;
  switch (lpr) {
    case 1: fn = (void*)bpr_steps_coop<1, 1>; slot = 0; break;
    case 2: fn = (void*)bpr_steps_coop<2, 1>; slot = 1; break;
    case 4: fn = (void*)bpr_steps_coop<4, 1>; slot = 2; break;
    case 8: fn = (void*)bpr_steps_coop<8, 1>; slot = 3; break;
    case 16: fn = (void*)bpr_steps_coop<16, 1>; slot = 4; break;
    default: fn = (void*)bpr_steps_coop<32, 1>; slot = 5; break;
  }
  // Occupancy is a property of the kernel: queried once per instance.  `per_sm` CTAs of it fit an SM without dynamic shared
  // memory, and `smem_cap` is the dynamic shared memory a CTA may take while still `per_sm` of them fit: the shared-memory
  // Adam is only used within that budget, so it never shrinks the grid.
  static int per_sm_cache[6] = {0, 0, 0, 0, 0, 0};
  static size_t smem_cap_cache[6] = {0, 0, 0, 0, 0, 0};
  int per_sm = per_sm_cache[slot];
  if (per_sm == 0) {
    BRK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kThreads, 0));
    BRK_REQUIRE(per_sm > 0, BRK_E_STATE, "brk_bpr_train_steps: cooperative kernel does not fit");
    size_t cap_bytes = 0;
    BRK_CUDA(cudaOccupancyAvailableDynamicSMemPerBlock(&cap_bytes, fn, per_sm, kThreads));
    per_sm_cache[slot] = per_sm;
    smem_cap_cache[slot] = cap_bytes;
  }
  int64_t want = (max_count * lpr + kThreads - 1) / kThreads;
  const int64_t cap = int64_t(per_sm) * ctx->sm_count;
  const int grid = int(want < cap ? (want < 1 ? 1 : want) : cap);
  // CTA slices of the tables (the same cut as the bulk L2 prefetch): w, m and v of both take 3 * (slice_u + slice_i) float4
  size_t smem = 0;
  const brk_table* tabs[2] = {user, item};
  for (int k = 0; k < 2; ++k) {
    const int64_t n4 = tabs[k]->rows * d / 4;
    const int64_t s4 = (n4 + grid - 1) / grid;
    P.slice4[k] = int32_t(s4 < (int64_t(1) << 20) ? s4 : 0);
    smem += 3 * size_t(s4) * 16;
  }
  const bool smem_ok = P.world == 1 && !getenv("BRK_BPR_NO_SMEM_ADAM") && smem <= smem_cap_cache[slot] &&
                       P.slice4[0] > 0 && P.slice4[1] > 0 && brk_aligned16(user->m) && brk_aligned16(user->v) &&
                       brk_aligned16(item->m) && brk_aligned16(item->v);
  if (!smem_ok) { P.slice4[0] = P.slice4[1] = 0; smem = 0; }
  P.last_sync = getenv("BRK_BPR_NO_SMEM_ADAM") ? 1 : 0;
  // above the default 48 KB a kernel needs the opt-in attribute, which is per device: set it for the current one
  if (smem > 48 * 1024) BRK_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  void* args[] = {(void*)&P};
  BRK_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(kThreads), args, smem, st));
  return 0;
}

// step descriptors of batches `batch_index[k]` of arrays cut into batches of `batch`
static void make_steps(BprStep* out, const int64_t* batch_index, int n_steps, int64_t total, int64_t batch) {
  for (int k = 0; k < n_steps; ++k) {
    const int64_t off = batch_index[k] * batch;
    out[k].off = off; out[k].sample_index = off;
    out[k].count = int32_t((off + batch <= total) ? batch : total - off);
    out[k]._pad = 0;
  }
}

// Multi-step driver: one C call enqueues n_steps x (fused fwd/bwd + optimizer) so that the host
// cost per step is two kernel launches and nothing else (model.fit's inner loop,
// /root/reference/src/models/BPRModel.py:109).  batch_index_host[k] selects which batch of the
// device-resident triplet arrays step k consumes (Keras shuffles batches per epoch).
extern "C" int brk_bpr_train_steps(brk_ctx* ctx, const brk_table* user, const brk_table* item,
                                   const int32_t* u, const int32_t* p, const int32_t* n, int64_t total,
                                   int64_t batch, const int64_t* batch_index_host, int32_t n_steps,
                                   brk_adam_hyper h, int32_t lazy_adam, int64_t* step_dev, float* losses,
                                   void* stream) {
  BRK_REQUIRE(ctx && user && item && u && p && n && batch_index_host && step_dev, BRK_E_ARG,
              "brk_bpr_train_steps: null argument");
  BRK_REQUIRE(total > 0 && batch > 0 && n_steps >= 0, BRK_E_ARG, "brk_bpr_train_steps: total=%lld batch=%lld",
              (long long)total, (long long)batch);
  const int64_t n_batches = (total + batch - 1) / batch;
  for (int k = 0; k < n_steps; ++k)
    BRK_REQUIRE(batch_index_host[k] >= 0 && batch_index_host[k] < n_batches, BRK_E_ARG,
                "brk_bpr_train_steps: batch index %lld of %lld", (long long)batch_index_host[k], (long long)n_batches);
  if (n_steps == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const bool coop_ok = coop_eligible(user, item, lazy_adam);
  if (coop_ok) {
    std::vector<BprStep> steps(n_steps);
    make_steps(steps.data(), batch_index_host, n_steps, total, batch);
    return launch_coop_steps(ctx, user, item, u, p, n, steps.data(), n_steps, batch < total ? batch : total, h, step_dev,
                             losses, st);
  }
  brk_table tabs[2] = {*user, *item};
  for (int k = 0; k < n_steps; ++k) {
    const int64_t bi = batch_index_host[k];
    const int64_t off = bi * batch;
    const int64_t cnt = (off + batch <= total) ? batch : total - off;
    int rc = brk_bpr_fwd_bwd(ctx, user, item, u + off, p + off, n + off, cnt, 0, losses ? losses + k : nullptr, stream);
    if (rc) return rc;
    rc = lazy_adam ? brk_adam_rows(ctx, tabs, 2, h, step_dev, 1, stream)
                   : brk_adam_dense_keras(ctx, tabs, 2, h, step_dev, 1, stream);
    if (rc) return rc;
  }
  return 0;
}

// End-to-end steps from HOST buffers in one call (the public-API path bench.py's `e2e` times):
// every step's user / positive ids go H2D with their own cudaMemcpyAsync from the caller's page-locked
// arrays (ONE copy per step when the host layout is batch-major [n_batches][2][batch], i.e.
// p_host == u_host + batch and host_batch_stride == 2*batch), the step runs, and the losses come back D2H
// once per chunk.  Steps are launched in
// chunks of kChunk: one cooperative kernel runs kChunk steps (sampling its own Philox negatives, see
// bpr_steps_coop), so launch latency and the up-front staging of the first step are paid once per chunk.
// Copies run on a second stream through a ring of 2*kChunk staging slots (two chunks in flight):
//   copy stream,    chunk j : wait done[j-2] ; D2H losses of chunk j-2 (one copy) ; H2D ids of chunk j ; record ready[j]
//   compute stream, chunk j : wait ready[j] ; cooperative kernel (kChunk steps) ; record done[j]
// d_stage: device int32 scratch of BRK_BPR_STAGE_INTS(batch) = 4*kChunk*batch; d_losses: device [n_steps].
constexpr int kChunk = 16;

extern "C" int64_t brk_bpr_host_stage_ints(int64_t batch) { return int64_t(4) * kChunk * batch; }

extern "C" int brk_bpr_train_steps_host(brk_ctx* ctx, const brk_table* user, const brk_table* item,
                                        const int32_t* u_host, const int32_t* p_host, int64_t total, int64_t batch,
                                        int64_t host_batch_stride, const int64_t* batch_index_host, int32_t n_steps, uint32_t seed, uint32_t epoch,
                                        int32_t num_items, const int64_t* csr_indptr, const int32_t* csr_items,
                                        brk_adam_hyper h, int32_t lazy_adam, int64_t* step_dev, int32_t* d_stage,
                                        float* d_losses, float* losses_host, const brk_dp_peer* dp, void* stream) {
  BRK_REQUIRE(ctx && user && item && u_host && p_host && batch_index_host && step_dev && d_stage && d_losses &&
                  csr_indptr && csr_items, BRK_E_ARG, "brk_bpr_train_steps_host: null argument");
  BRK_REQUIRE(total > 0 && batch > 0 && n_steps >= 0 && num_items > 0, BRK_E_ARG,
              "brk_bpr_train_steps_host: total=%lld batch=%lld", (long long)total, (long long)batch);
  if (host_batch_stride <= 0) host_batch_stride = batch;
  BRK_REQUIRE(host_batch_stride >= batch, BRK_E_ARG, "brk_bpr_train_steps_host: host_batch_stride=%lld < batch",
              (long long)host_batch_stride);
  // batch-major host layout [n_batches][2][batch] (a loader that writes each batch's user ids then its item
  // ids): the step's inputs are ONE contiguous block -> one DMA per step instead of two
  const bool packed = host_batch_stride == 2 * batch && p_host == u_host + batch;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n_batches = (total + batch - 1) / batch;
  for (int k = 0; k < n_steps; ++k)
    BRK_REQUIRE(batch_index_host[k] >= 0 && batch_index_host[k] < n_batches, BRK_E_ARG,
                "brk_bpr_train_steps_host: batch index %lld of %lld", (long long)batch_index_host[k], (long long)n_batches);
  if (n_steps == 0) return 0;
  if (int rc = brk_ctx_ensure_copy(ctx)) return rc;
  cudaStream_t cs = ctx->copy_stream;
  const bool use_dp = dp != nullptr && dp->world > 1;
  // data-parallel mode: the tables are views into the peer arenas (their Adam moments live in `dp`, sharded)
  const bool coop_ok = use_dp ? ((user->d & 3) == 0 && user->d <= 128 && !lazy_adam) : coop_eligible(user, item, lazy_adam);
  BRK_REQUIRE(!use_dp || (coop_ok && item->w == user->w + user->rows * user->d && item->g == user->g + user->rows * user->d),
              BRK_E_ARG, "brk_bpr_train_steps_host: data-parallel mode needs adjacent arena views, d %% 4 == 0, d <= 128");
  brk_table tabs[2] = {*user, *item};
  // Chunk plan: 2, 4, 8 steps, then kChunk each.  The first launch waits for its whole chunk's ids, so a call of a few
  // steps (the bench's default --steps 20) used to spend ~150 us on 16 steps' worth of DMA before the first kernel; with a
  // short first chunk the kernels start after two steps' ids (256 KB) and every later copy hides behind compute.
  std::vector<int> starts;                          // chunk j = steps [starts[j], starts[j + 1])
  for (int k = 0, c = 2; k < n_steps; k += c, c = (c * 2 < kChunk ? c * 2 : kChunk)) starts.push_back(k);
  const int n_chunks = int(starts.size());
  starts.push_back(n_steps);
  std::vector<int> chunk_of(n_steps);
  for (int j = 0; j < n_chunks; ++j)
    for (int k = starts[j]; k < starts[j + 1]; ++k) chunk_of[k] = j;
  auto count_of = [&](int k) { const int64_t off = batch_index_host[k] * batch; return (off + batch <= total) ? batch : total - off; };
  // slot of step k: two chunk halves of kChunk slots, each slot = [u: batch][p: batch]
  auto slot_of = [&](int k) { const int j = chunk_of[k]; return d_stage + (int64_t(j & 1) * kChunk + (k - starts[j])) * 2 * batch; };
  auto copy_chunk = [&](int j) -> int {            // on the copy stream: results of chunk j-2 back, ids of chunk j in
    if (j >= 2) {
      BRK_CUDA(cudaStreamWaitEvent(cs, ctx->ev_done[j & 1], 0));
      if (losses_host)                               // the step losses of chunk j-2, one DMA
        BRK_CUDA(cudaMemcpyAsync(losses_host + starts[j - 2], d_losses + starts[j - 2], (starts[j - 1] - starts[j - 2]) * sizeof(float),
                                 cudaMemcpyDeviceToHost, cs));
    }
    // the chunk's H2D copies are spread over kCopyLanes streams so that several DMAs are in flight at once (a
    // single 128 KiB copy costs 10-35 us of latency on virtualised hosts); everything rejoins on `cs`
    BRK_CUDA(cudaEventRecord(ctx->ev_go, cs));
    for (int a = 0; a < BRK_COPY_AUX; ++a) BRK_CUDA(cudaStreamWaitEvent(ctx->copy_aux[a], ctx->ev_go, 0));
    for (int k = starts[j]; k < starts[j + 1]; ++k) {
      const int64_t hoff = batch_index_host[k] * host_batch_stride, cnt = count_of(k);
      const int lane = k % (BRK_COPY_AUX + 1);
      cudaStream_t cl = lane == 0 ? cs : ctx->copy_aux[lane - 1];
      if (packed) {
        BRK_CUDA(cudaMemcpyAsync(slot_of(k), u_host + hoff, 2 * batch * sizeof(int32_t), cudaMemcpyHostToDevice, cl));
      } else {
        BRK_CUDA(cudaMemcpyAsync(slot_of(k), u_host + hoff, cnt * sizeof(int32_t), cudaMemcpyHostToDevice, cl));
        BRK_CUDA(cudaMemcpyAsync(slot_of(k) + batch, p_host + hoff, cnt * sizeof(int32_t), cudaMemcpyHostToDevice, cl));
      }
    }
    for (int a = 0; a < BRK_COPY_AUX; ++a) {
      BRK_CUDA(cudaEventRecord(ctx->ev_aux[a], ctx->copy_aux[a]));
      BRK_CUDA(cudaStreamWaitEvent(cs, ctx->ev_aux[a], 0));
    }
    BRK_CUDA(cudaEventRecord(ctx->ev_ready[j & 1], cs));
    return 0;
  };
  // the copy stream must not run ahead of work already queued on `st` that may still use the staging slots
  BRK_CUDA(cudaEventRecord(ctx->ev_done[2], st));
  BRK_CUDA(cudaStreamWaitEvent(cs, ctx->ev_done[2], 0));
  if (int rc = copy_chunk(0)) return rc;
  for (int j = 0; j < n_chunks; ++j) {
    if (j + 1 < n_chunks) { if (int rc = copy_chunk(j + 1)) return rc; }
    const int k0 = starts[j], k1 = starts[j + 1];
    BRK_CUDA(cudaStreamWaitEvent(st, ctx->ev_ready[j & 1], 0));
    if (coop_ok) {
      BprStep steps[kChunk];
      for (int k = k0; k < k1; ++k) {
        steps[k - k0].off = slot_of(k) - d_stage;                     // u at off, p at off + batch (see P.p below)
        steps[k - k0].sample_index = batch_index_host[k] * batch;
        steps[k - k0].count = int32_t(count_of(k)); steps[k - k0]._pad = 0;
      }
      CoopSampler smp{csr_indptr, csr_items, seed, epoch, uint32_t(num_items)};
      int rc = launch_coop_steps(ctx, user, item, d_stage, d_stage + batch, nullptr, steps, k1 - k0, batch, h, step_dev,
                                 d_losses + k0, st, &smp, use_dp ? dp : nullptr);
      if (rc) return rc;
    } else {
      // generic widths / lazy Adam: separate sampler, fused fwd/bwd and optimizer launches (negatives in the
      // context scratch; steps are ordered on `st`, so one buffer serves all of them)
      if (int rc = ensure_scratch(ctx, size_t(batch) * sizeof(int32_t))) return rc;
      int32_t* dn = reinterpret_cast<int32_t*>(ctx->scratch);
      for (int k = k0; k < k1; ++k) {
        const int64_t off = batch_index_host[k] * batch, cnt = count_of(k);
        int32_t* du = slot_of(k);
        int rc = brk_philox_bpr_negatives(ctx, du, cnt, off, seed, epoch, num_items, csr_indptr, csr_items, dn, stream);
        if (rc) return rc;
        rc = brk_bpr_fwd_bwd(ctx, user, item, du, du + batch, dn, cnt, 0, d_losses + k, stream);
        if (rc) return rc;
        rc = lazy_adam ? brk_adam_rows(ctx, tabs, 2, h, step_dev, 1, stream)
                       : brk_adam_dense_keras(ctx, tabs, 2, h, step_dev, 1, stream);
        if (rc) return rc;
      }
    }
    BRK_CUDA(cudaEventRecord(ctx->ev_done[j & 1], st));
  }
  // results of the last two chunks, then rejoin: everything the copy stream did is ordered before
  // whatever follows on `st`
  if (losses_host) {
    const int first = starts[n_chunks >= 2 ? n_chunks - 2 : 0];
    BRK_CUDA(cudaStreamWaitEvent(cs, ctx->ev_done[(n_chunks - 1) & 1], 0));
    BRK_CUDA(cudaMemcpyAsync(losses_host + first, d_losses + first, (n_steps - first) * sizeof(float),
                             cudaMemcpyDeviceToHost, cs));
  }
  BRK_CUDA(cudaEventRecord(ctx->ev_ready[2], cs));
  BRK_CUDA(cudaStreamWaitEvent(st, ctx->ev_ready[2], 0));
  return 0;
}

// The same loop with the ids left in page-locked (mapped) HOST memory and no copy engine involved: ONE
// cooperative launch runs all n_steps; each step's kernel phase pulls that step's ids over PCIe
// (8*batch bytes), draws the negatives, trains, and stores the step's loss straight into
// losses_host.  u_host / p_host / losses_host must be device-accessible page-locked memory
// (cudaHostAlloc / torch pin_memory under unified addressing).
extern "C" int brk_bpr_train_steps_mapped(brk_ctx* ctx, const brk_table* user, const brk_table* item,
                                          const int32_t* u_host, const int32_t* p_host, int64_t total, int64_t batch,
                                          const int64_t* batch_index_host, int32_t n_steps, uint32_t seed,
                                          uint32_t epoch, int32_t num_items, const int64_t* csr_indptr,
                                          const int32_t* csr_items, brk_adam_hyper h, int64_t* step_dev,
                                          float* losses_host, void* stream) {
  BRK_REQUIRE(ctx && user && item && u_host && p_host && batch_index_host && step_dev && csr_indptr && csr_items,
              BRK_E_ARG, "brk_bpr_train_steps_mapped: null argument");
  BRK_REQUIRE(total > 0 && batch > 0 && n_steps >= 0 && num_items > 0, BRK_E_ARG,
              "brk_bpr_train_steps_mapped: total=%lld batch=%lld", (long long)total, (long long)batch);
  const int64_t n_batches = (total + batch - 1) / batch;
  for (int k = 0; k < n_steps; ++k)
    BRK_REQUIRE(batch_index_host[k] >= 0 && batch_index_host[k] < n_batches, BRK_E_ARG,
                "brk_bpr_train_steps_mapped: batch index %lld of %lld", (long long)batch_index_host[k], (long long)n_batches);
  BRK_REQUIRE(coop_eligible(user, item, 0), BRK_E_ARG,
              "brk_bpr_train_steps_mapped: needs the cooperative path (d %% 4 == 0, d <= 128, Adam slots, 16-byte aligned tables)");
  if (n_steps == 0) return 0;
  // device-visible aliases of the caller's buffers (mapped page-locked host memory, or plain device memory)
  auto dev_alias = [](const void* hp, const void** out) -> int {
    cudaPointerAttributes a;
    BRK_CUDA(cudaPointerGetAttributes(&a, hp));
    BRK_REQUIRE((a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) &&
                    a.devicePointer, BRK_E_ARG,
                "brk_bpr_train_steps_mapped: buffer %p is not device-accessible (page-lock it: cudaHostAlloc / pin_memory)", hp);
    *out = a.devicePointer;
    return 0;
  };
  const void *du = nullptr, *dp = nullptr, *dl = nullptr;
  if (int rc = dev_alias(u_host, &du)) return rc;
  if (int rc = dev_alias(p_host, &dp)) return rc;
  if (losses_host) { if (int rc = dev_alias(losses_host, &dl)) return rc; }
  CoopSampler smp{csr_indptr, csr_items, seed, epoch, uint32_t(num_items)};
  std::vector<BprStep> steps(n_steps);
  make_steps(steps.data(), batch_index_host, n_steps, total, batch);
  return launch_coop_steps(ctx, user, item, reinterpret_cast<const int32_t*>(du), reinterpret_cast<const int32_t*>(dp),
                           nullptr, steps.data(), n_steps, batch < total ? batch : total, h, step_dev,
                           reinterpret_cast<float*>(const_cast<void*>(dl)), (cudaStream_t)stream, &smp);
}

// Mirrored data-parallel training steps (one process per GPU; the reference's MultiWorkerMirroredStrategy,
// src/models/RModel.py:119-121) in ONE cooperative launch per rank: every step is this rank's fused fwd/bwd on
// its slice of the global batch, a cross-GPU barrier, reduce-scatter + Adam + all-gather over NVLink peer memory
// and a second barrier -- no NCCL call, no kernel launch and no host involvement between steps.  user / item
// must be views into this rank's arenas of `dp` (user first, item right behind it, w and g alike); all ranks call
// with the same n_steps and batch; gradients are scaled by 1 / (world * batch).
extern "C" int brk_bpr_train_steps_dp(brk_ctx* ctx, const brk_table* user, const brk_table* item, const int32_t* u,
                                      const int32_t* p, const int32_t* n, int64_t total, int64_t batch,
                                      const int64_t* batch_index_host, int32_t n_steps, brk_adam_hyper h,
                                      const brk_dp_peer* dp, int64_t* step_dev, float* losses, void* stream) {
  BRK_REQUIRE(ctx && user && item && u && p && n && batch_index_host && step_dev && dp, BRK_E_ARG,
              "brk_bpr_train_steps_dp: null argument");
  BRK_REQUIRE(total > 0 && batch > 0 && n_steps >= 0, BRK_E_ARG, "brk_bpr_train_steps_dp: total=%lld batch=%lld",
              (long long)total, (long long)batch);
  BRK_REQUIRE(dp->world >= 1 && dp->world <= 64 && dp->rank >= 0 && dp->rank < dp->world && dp->n > 0 && (dp->n & 3) == 0 &&
                  dp->peer_w && dp->peer_g && dp->peer_flags && dp->m && dp->v && dp->local_sync, BRK_E_ARG,
              "brk_bpr_train_steps_dp: descriptor incomplete");
  const int d = user->d;
  BRK_REQUIRE(d == item->d && (d & 3) == 0 && d <= 128 && item->w == user->w + user->rows * d &&
                  item->g == user->g + user->rows * d && (user->rows + item->rows) * d <= dp->n &&
                  brk_aligned16(user->w) && brk_aligned16(user->g), BRK_E_ARG,
              "brk_bpr_train_steps_dp: tables must be adjacent views into the peer arenas (d %% 4 == 0, d <= 128)");
  const int64_t n_batches = (total + batch - 1) / batch;
  for (int k = 0; k < n_steps; ++k)
    BRK_REQUIRE(batch_index_host[k] >= 0 && batch_index_host[k] < n_batches && (batch_index_host[k] + 1) * batch <= total,
                BRK_E_ARG, "brk_bpr_train_steps_dp: batch index %lld (full batches only: every rank must run the same count)",
                (long long)batch_index_host[k]);
  if (n_steps == 0) return 0;
  std::vector<BprStep> steps(n_steps);
  make_steps(steps.data(), batch_index_host, n_steps, total, batch);
  return launch_coop_steps(ctx, user, item, u, p, n, steps.data(), n_steps, batch, h, step_dev, losses,
                           (cudaStream_t)stream, nullptr, dp);
}

// Debug hook (profiles/dp_trace.py): copies the phase stamps of the last traced cooperative launch to the host.
extern "C" int brk_coop_trace_read(unsigned long long* out_host, int32_t n_words) {
  if (!g_coop_trace) return BRK_E_STATE;
  BRK_CUDA(cudaMemcpy(out_host, g_coop_trace, size_t(n_words) * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return 0;
}

// Fused BPR forward/backward on row-sharded tables (see brk_neumf_step_sharded for the protocol around it: a
// brk_peer_barrier, then every owner applies its optimizer to its shards, then another barrier).
extern "C" int brk_bpr_fwd_bwd_sharded(brk_ctx* ctx, const brk_shards* user, const brk_shards* item, int32_t d,
                                       const int32_t* u, const int32_t* p, const int32_t* n, int64_t batch,
                                       int64_t global_batch, float* loss_out, void* stream) {
  BRK_REQUIRE(ctx && user && item && u && p && n, BRK_E_ARG, "brk_bpr_fwd_bwd_sharded: null argument");
  BRK_REQUIRE(d > 0 && (d & 3) == 0 && d <= 512 && batch > 0, BRK_E_ARG, "brk_bpr_fwd_bwd_sharded: d=%d batch=%lld (d %% 4 == 0)",
              d, (long long)batch);
  BRK_REQUIRE(user->world >= 1 && user->world <= BRK_MAX_PEERS && item->world == user->world, BRK_E_ARG,
              "brk_bpr_fwd_bwd_sharded: world=%d/%d", user->world, item->world);
  v2::TabRef TU, TI;
  const brk_shards* sh[2] = {user, item};
  v2::TabRef* T[2] = {&TU, &TI};
  for (int k = 0; k < 2; ++k) {
    for (int q = 0; q < BRK_MAX_PEERS; ++q) { T[k]->w[q] = nullptr; T[k]->g[q] = nullptr; T[k]->t[q] = nullptr; }
    T[k]->world = sh[k]->world;
    for (int q = 0; q < sh[k]->world; ++q) {
      BRK_REQUIRE(sh[k]->w[q] && sh[k]->g[q] && brk_aligned16(sh[k]->w[q]) && brk_aligned16(sh[k]->g[q]), BRK_E_ARG,
                  "brk_bpr_fwd_bwd_sharded: shard %d of table %d missing or not 16-byte aligned", q, k);
      T[k]->w[q] = sh[k]->w[q]; T[k]->g[q] = sh[k]->g[q]; T[k]->t[q] = sh[k]->touched[q];
    }
  }
  const float inv_batch = 1.0f / float(global_batch > 0 ? global_batch : batch);
  const double inv_local = 1.0 / double(batch);
  const int d4 = d >> 2, lpr = brk_lanes_per_row(d4), nch = (d4 + lpr - 1) / lpr;
  const int64_t cap = int64_t(ctx->sm_count) * (2048 / kThreads);
  int64_t need = (batch * lpr + kThreads - 1) / kThreads;
  const int grid = int(need < 1 ? 1 : (need < cap ? need : cap));
  cudaStream_t st = (cudaStream_t)stream;
#define BRK_BPRS_CASE(L, N)                                                                                         \
  bpr_vec_sharded<L, N><<<grid, kThreads, 0, st>>>(TU, TI, d4, u, p, n, batch, inv_batch, inv_local, ctx->loss_acc + 0, \
                                                   ctx->tickets + 0, loss_out)
  if (lpr == 1) BRK_BPRS_CASE(1, 1);
  else if (lpr == 2) BRK_BPRS_CASE(2, 1);
  else if (lpr == 4) BRK_BPRS_CASE(4, 1);
  else if (lpr == 8) BRK_BPRS_CASE(8, 1);
  else if (lpr == 16) BRK_BPRS_CASE(16, 1);
  else if (nch == 1) BRK_BPRS_CASE(32, 1);
  else if (nch == 2) BRK_BPRS_CASE(32, 2);
  else if (nch == 3) BRK_BPRS_CASE(32, 3);
  else BRK_BPRS_CASE(32, 4);
#undef BRK_BPRS_CASE
  BRK_LAUNCH_CHECK();
  return 0;
}
