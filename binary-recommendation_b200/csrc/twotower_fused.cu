// The in-batch-softmax two-tower training step (trainers/twoTower.py:77-102) as ONE cooperative launch.
//
// The multi-kernel step (twotower.cu + gemm_tc.cu) is a chain of 8 dependent launches of ~6 us each at the reference's
// batch of 1000 (twoTower.py:292), and it writes the [B,B] score matrix to memory three times.  Here a CTA owns one
// 128 x 128 tile of the score matrix for the whole step -- flash-attention style, the scores never leave the SM:
//
//   phase F  (2T CTAs: tower x row block)   e = Emb[ids] (gathered straight into the operand tile), z = e W + b -> q / c
//   ---- grid barrier ----
//   phase S  (T^2 CTAs: score tile i, j)    S_ij = q_i c_j^T in TMEM; accidental-hit mask; per row (max, sum exp) of the tile
//   ---- grid barrier ----                  lse of a row = the T tile partials combined; loss from the diagonal tiles
//                                           P_ij = exp(S_ij - lse) - I stays in REGISTERS; written once K-major, once
//                                           MN-major into shared memory: dq_i += P_ij c_j, dc_j += P_ij^T q_i (REDs)
//   ---- grid barrier ----
//   phase G  (4T CTAs: tower x row block x {rows, weights})   de = dz W^T -> row-contiguous REDs into the table
//                                           accumulators;  dW += e^T dz, db += column sums of dz
//   ---- grid barrier ----                  (brk_twotower_train_step only)
//   phase O  (all CTAs)                     Keras Adagrad on the Dense blocks and on the rows this batch touched
//
// Operand loads that do not depend on a barrier (the MN-major re-staging of q_i / c_j, phase G's Dense kernel and
// re-gathered embedding rows) are issued in front of it and land while the grid waits.
//
// All six products are tcgen05.mma kind::tf32 (operands = fp32 bits truncated by the tensor core, fp32 accumulation in
// TMEM) on 128 x 128 tiles staged by cp.async in the swizzle of the view that reads them (tc_tiles.cuh); no operand is
// transposed in memory.  T = ceil(B / 128); the launch needs max(T^2, 4T) <= SM count co-resident CTAs (B <= 1536 on
// a B200); larger batches, other modes (rdZero) and widths above 128 take the multi-kernel step.
// The grid barrier (brk_grid_barrier, common.cuh) keeps its base in device memory (bar[2]), so the launch can be captured
// into a CUDA graph and replayed (TwoTowerModel.fit does).
//
// fused_step<false, true> is the step with TFRS Retrieval's options (brk_twotower_step_retrieval): temperature, candidate
// sampling probabilities (caller-supplied or the streaming frequency estimate), sample weights.  Phase F's item-tower CTAs
// update the estimator for their rows; phase S turns each column's probability into a log2-domain term in shared memory
// (after the F -> S barrier, so a column sees the update of its id whichever CTA made it), folds 1/tau into the
// read-out FFMA and w/tau into the P scale, and weighs the diagonal loss.
//
// fused_step<true> is the same step on row-sharded tables (brk_twotower_step_sharded): row r of a table lives on rank
// r % G at local row r / G.  The ids are split into (owner, local row) once, where they are staged in shared memory; the
// gathers of phases F and G read the owner's shard (NVLink peer memory across GPUs) and phase G's row-gradient REDs and
// touched bits go to the owner's accumulator and bitmask.  Phase O does not run: an owner's accumulator is complete only
// after a cross-GPU barrier and the Dense gradients only after their all-reduce, so the launch ends after phase G.
//
// fused_step<false, true, true> / fused_step<true, true, true> are the two steps with sampled negatives (brk_tt_sampled,
// drawn by tt_sample_negatives_kernel ahead of the launch): the item side has n = B + M rows (the batch's, then the draws)
// in Tc = ceil(n / 128) row blocks.  Phase F runs T + Tc row blocks, phase S T * Tc score tiles (the identity of P only in
// tiles with j < T -- the diagonal tiles -- and columns >= n dropped), phase G 2 (T + Tc) tower blocks, and phase O also
// walks the sampled rows.  Temperature and weights go where fused_step<false, true> puts them; no probabilities.  The
// launch needs max(T * Tc, 2 (T + Tc)) <= SM count.
//
// fused_step<true, true> is the row-sharded step with the options (brk_twotower_step_sharded_retrieval).  The estimator's
// state is sharded like the item table and only read here: its update is brk_tt_estimator_update_sharded, a launch of its
// own that every rank runs before a cross-GPU barrier.  Phase S reads the gap of column j's item row y at its owner,
// gap[y % G][y / G], with an L2-only load (the row may have been updated through NVLink by another GPU).
#include "common.cuh"
#include "tc.cuh"
#include "tc_tiles.cuh"
#include <math_constants.h>
#include <stdlib.h>
#include <type_traits>

namespace ttf {

using ntc::issue_gemm;
using ntc::km_off16;
using ntc::mn_off16;
using ntc::pad32;

constexpr int NT = 256, TS = 128;
constexpr uint32_t TILE = TS * 128 * 4;                             // one 128 x 128 fp32 operand tile
constexpr float kMinFloatOver100 = -3.4028234663852886e36f;          // np.finfo(np.float32).min / 100 (TFRS RemoveAccidentalHits)
constexpr float kLog2e = 1.4426950408889634f, kLn2 = 0.6931471805599453f;
__device__ __forceinline__ float ex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

struct Params {
  brk_table eu, ei;                                                  // embedding tables (w, g, touched)
  const float* W[2]; float* gW[2];                                   // Dense blocks: kernel [E][S], then bias [S]
  int E[2], S;
  const int32_t* ids[2]; const int32_t* cand;
  int B, T, training;
  float* z[2];                                                       // q, c   [B][S]
  float* dz[2];                                                      // dq, dc [B][S]
  float2* part;                                                      // [T * 128][T]: (max, sum exp) of row x column tile
  double* acc; float* loss_out;
  unsigned int* bar;                                                 // grid-barrier words {count, error, base} (common.cuh)
  unsigned long long* trace;                                         // BRK_TT_TRACE: %globaltimer stamps of block 0
  // Keras Adagrad in the same launch (brk_twotower_train_step): touched rows of the two tables + the two Dense blocks
  int do_opt; float lr, eps;
  brk_table dn[2];
};
// fused_step<true> (row-sharded tables): the same block followed by the two tables' shards.  A separate type keeps the
// parameter block of fused_step<false> as it was (its size changes ptxas' schedule).
struct ShardedParams : Params {
  brk_shards su, si;
};
template <bool SH> using ParamsT = typename std::conditional<SH, ShardedParams, Params>::type;
// fused_step<false, true>: the retrieval options (brk_tt_retrieval) behind the same block
struct RetrievalParams : Params {
  const float* cand_prob; const float* row_weight;                   // [B] or null
  long long* last; float* gap; long long* step;                      // streaming estimator (last == null: off)
  float inv_tau, alpha;
};
// fused_step<true, true>: the options behind the sharded block; gap[p] is rank p's shard of the estimator's gap
struct ShardedRetrievalParams : ShardedParams {
  const float* cand_prob; const float* row_weight;                   // [B] or null
  const float* gap[BRK_MAX_PEERS];                                   // gap[0] == null: no estimator
  float inv_tau;
};
// fused_step<SH, true, true>: sampled negatives (brk_tt_sampled) behind the options block (no probabilities, no estimator):
// the item side has n = B + M rows, item row x is ids[1][x] for x < B and smp[x - B] after, Tc = ceil(n / 128)
struct SampledParams : RetrievalParams { const int32_t* smp; int M, n, Tc; };
struct ShardedSampledParams : ShardedRetrievalParams { const int32_t* smp; int M, n, Tc; };
template <bool SH, bool RT, bool SM = false> using KParamsT = typename std::conditional<SM,
    typename std::conditional<SH, ShardedSampledParams, SampledParams>::type,
    typename std::conditional<RT, typename std::conditional<SH, ShardedRetrievalParams, RetrievalParams>::type, ParamsT<SH>>::type>::type;
// the estimator's gap of item row y as phase S reads it (after the F -> S barrier, past L1)
__device__ __forceinline__ bool has_estimator(const RetrievalParams& P) { return P.last != nullptr; }
__device__ __forceinline__ bool has_estimator(const ShardedRetrievalParams& P) { return P.gap[0] != nullptr; }
__device__ __forceinline__ float estimator_gap(const RetrievalParams& P, int32_t y) { return __ldcg(P.gap + y); }
__device__ __forceinline__ float estimator_gap(const ShardedRetrievalParams& P, int32_t y) {
  const int G = P.si.world;
  return __ldcg(P.gap[y % G] + y / G);
}

__device__ __forceinline__ void adagrad4(float4* w, float4* a, float4* g, float lr, float eps) {
  float4 w4 = *w, a4 = *a;
  const float4 g4 = *g;
  a4.x += g4.x * g4.x; w4.x -= lr * g4.x / (sqrtf(a4.x) + eps);
  a4.y += g4.y * g4.y; w4.y -= lr * g4.y / (sqrtf(a4.y) + eps);
  a4.z += g4.z * g4.z; w4.z -= lr * g4.z / (sqrtf(a4.z) + eps);
  a4.w += g4.w * g4.w; w4.w -= lr * g4.w / (sqrtf(a4.w) + eps);
  *w = w4; *a = a4; *g = make_float4(0.f, 0.f, 0.f, 0.f);
}

__device__ __forceinline__ void stamp(const Params& P, int k) {
  if (P.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    P.trace[k] = t;
  }
}

__device__ __forceinline__ void cp_async16(uint8_t* dst, const void* src, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(tc::smem_u32(dst)), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// 128 x 128 operand tile <- rows [r0, r0 + 128) x columns [0, ncols) of a row-major matrix (zero outside), or the table
// rows named by ids_s (gather).  MN = 0: K-major swizzle, 1: MN-major swizzle (tc_tiles.cuh).
// Thread (w = t / 32, c4 = t % 32) copies chunk c4 of rows w, w + 8, ..., w + 120: in both swizzles 8 rows further is
// +1024 bytes, so the offsets are one constant per thread plus an immediate.
template <int MN>
__device__ __forceinline__ void load_tile(uint8_t* dst, const float* __restrict__ src, int ld, int r0, int r_end, int ncols) {
  const int w = threadIdx.x >> 5, c4 = threadIdx.x & 31;
  int cb = (ncols - c4 * 4) * 4;
  cb = cb < 0 ? 0 : (cb > 16 ? 16 : cb);
  uint8_t* d = dst + (MN ? mn_off16(TS, w, c4) : km_off16(TS, w, c4));
  const float* p = src + int64_t(r0 + w) * ld + c4 * 4;
#pragma unroll
  for (int k = 0; k < TS / 8; ++k) {
    const int nb = (r0 + w + 8 * k < r_end) ? cb : 0;
    cp_async16(d + k * 1024, nb ? (const void*)(p + int64_t(8 * k) * ld) : (const void*)src, nb);
  }
}
// SH: ids_s holds local rows and own_s their owners; the row is read from shard own_s[.] of tower `tw`'s table (`table`
// is then unused: the zero-byte copies past `valid` name shard 0).
template <int MN, bool SH, class PT>
__device__ __forceinline__ void gather_tile(uint8_t* dst, const float* __restrict__ table, const PT& P, int tw, int d_,
                                            const int32_t* ids_s, const int32_t* own_s, int valid) {
  const int w = threadIdx.x >> 5, c4 = threadIdx.x & 31;
  int cb = (d_ - c4 * 4) * 4;
  cb = cb < 0 ? 0 : (cb > 16 ? 16 : cb);
  uint8_t* d = dst + (MN ? mn_off16(TS, w, c4) : km_off16(TS, w, c4));
  if constexpr (SH) table = (tw == 0 ? P.su : P.si).w[0];
#pragma unroll
  for (int k = 0; k < TS / 8; ++k) {
    const int nb = (w + 8 * k < valid) ? cb : 0;
    const float* src = table;
    if constexpr (SH) src = (tw == 0 ? P.su : P.si).w[own_s[w + 8 * k]];
    cp_async16(d + k * 1024, nb ? (const void*)(src + int64_t(ids_s[w + 8 * k]) * d_ + c4 * 4) : (const void*)table, nb);
  }
}


// 64 accumulator columns [c0, c0 + 64) of this thread's TMEM lane
__device__ __forceinline__ void tmem_load64(uint32_t tmem, int warp, int c0, float (&v)[64]) {
  uint32_t r0[32], r1[32];
  const uint32_t a = tmem + (uint32_t((warp & 3) * 32) << 16) + uint32_t(c0);
  tc::tmem_ld_32x32_issue(a, r0);
  tc::tmem_ld_32x32_issue(a + 32u, r1);
  tc::tmem_ld_wait(r0);
  tc::tmem_ld_wait(r1);
#pragma unroll
  for (int j = 0; j < 32; ++j) { v[j] = __uint_as_float(r0[j]); v[32 + j] = __uint_as_float(r1[j]); }
}

// The accumulator tile [128 rows x 128 columns] at TMEM column `col0` -> shared staging (row r at r * 512 bytes, 16-byte
// chunk c4 at (c4 ^ (r & 7)): conflict-free for lane = row writes and for row-contiguous reads)
__device__ __forceinline__ void tmem_to_staging(uint32_t tmem, int col0, uint8_t* stg) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, r = (warp & 3) * 32 + lane, h = warp >> 2;
  float v[64];
  tmem_load64(tmem, warp, col0 + h * 64, v);
#pragma unroll
  for (int j = 0; j < 64; j += 4)
    *reinterpret_cast<float4*>(stg + r * 512 + (((h * 16 + (j >> 2)) ^ (r & 7)) << 4)) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
}
__device__ __forceinline__ float4 staging_ld(const uint8_t* stg, int r, int c4) {
  return *reinterpret_cast<const float4*>(stg + r * 512 + ((c4 ^ (r & 7)) << 4));
}

#define TTF_OPERANDS_READY() do { cp_async_wait_all(); tc::fence_proxy_async_smem(); __syncthreads(); tc::fence_after_sync(); } while (0)

// ids_s[t] <- id r0 + t of tower k (threads t < TS); SH: the local row, and own_s[t] its owner (the one division per id)
template <bool SH>
__device__ __forceinline__ void stage_ids(const ParamsT<SH>& P, int k, int r0, int valid, int32_t* ids_s, int32_t* own_s) {
  const int t = threadIdx.x;
  if (t < TS) {
    const int32_t id = t < valid ? __ldg(P.ids[k] + r0 + t) : 0;
    if constexpr (SH) { ids_s[t] = id / P.su.world; own_s[t] = id % P.su.world; }
    else ids_s[t] = id;
  }
}

// ids_s[t] <- item row r0 + t of the sampled step's n = B + M item rows (the batch's, then the draws)
template <bool SH, class PT>
__device__ __forceinline__ void stage_item_ids(const PT& P, int r0, int valid, int32_t* ids_s, int32_t* own_s) {
  const int t = threadIdx.x;
  if (t < TS) {
    const int x = r0 + t;
    const int32_t id = t < valid ? (x < P.B ? __ldg(P.ids[1] + x) : __ldg(P.smp + (x - P.B))) : 0;
    if constexpr (SH) { ids_s[t] = id / P.su.world; own_s[t] = id % P.su.world; }
    else ids_s[t] = id;
  }
}

template <bool SH, bool RT = false, bool SM = false>
__global__ void __launch_bounds__(NT, 1) fused_step(const KParamsT<SH, RT, SM> P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* buf0 = sm; uint8_t* buf1 = sm + TILE; uint8_t* buf2 = sm + 2 * TILE;
  __shared__ uint64_t mbar;
  __shared__ uint32_t tmem_slot;
  __shared__ int32_t ids_s[TS], cand_r[TS];
  __shared__ int32_t own_s[SH ? TS : 1];                                // SH: owner rank of the row in ids_s
  __shared__ __align__(16) int32_t cand_c[TS];
  __shared__ float pm[2][TS], ps[2][TS], diag_s[TS], lse_s[TS];
  __shared__ __align__(16) float lq_s[RT ? TS : 1];                    // RT: log2 of the column's clipped probability
  __shared__ double red[32];
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int T = P.T, B = P.B, S = P.S;
  int n = B, Tc = T;                                                    // item-side rows and row blocks
  if constexpr (SM) { n = P.n; Tc = P.Tc; }
  const int b = blockIdx.x;
  stamp(P, 0);
  if (t == 0) { tc::mbar_init(tc::smem_u32(&mbar), 1); tc::fence_barrier_init(); }
  if (t < 32) tc::tmem_alloc<256>(tc::smem_u32(&tmem_slot));
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = tmem_slot;
  uint32_t phase = 0;
  unsigned int bar_target = *reinterpret_cast<volatile unsigned int*>(P.bar + 2);
  auto wait_mma = [&]() { tc::mbar_wait(tc::smem_u32(&mbar), phase); phase ^= 1u; tc::fence_after_sync(); };
  long long tstep = 0;                                                  // RT: this training step's estimator time
  if constexpr (RT && !SH) {
    if (P.last && P.training) tstep = *reinterpret_cast<volatile long long*>(P.step) + 1;   // written back after barrier 1
  }

  // ---------------- phase F: the two towers ----------------
  if (P.training) {                                                     // RED targets of phase S
    const int64_t n4 = int64_t(B) * S / 4;
    if constexpr (SM) {
      for (int k = 0; k < 2; ++k) {
        const int64_t nk4 = int64_t(k ? n : B) * S / 4;
        for (int64_t x = int64_t(b) * NT + t; x < nk4; x += int64_t(gridDim.x) * NT) reinterpret_cast<float4*>(P.dz[k])[x] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    } else {
      for (int k = 0; k < 2; ++k)
        for (int64_t x = int64_t(b) * NT + t; x < n4; x += int64_t(gridDim.x) * NT) reinterpret_cast<float4*>(P.dz[k])[x] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  if (b < (SM ? T + Tc : 2 * T)) {
    int k, r0, valid;
    if constexpr (SM) { k = b < T ? 0 : 1; r0 = (b - k * T) * TS; valid = min(TS, (k ? n : B) - r0); }
    else { k = b / T; r0 = (b % T) * TS; valid = min(TS, B - r0); }
    const int E = P.E[k];
    const brk_table& tab = k == 0 ? P.eu : P.ei;
    if constexpr (SM) { if (k == 1) stage_item_ids<SH>(P, r0, valid, ids_s, own_s); else stage_ids<SH>(P, k, r0, valid, ids_s, own_s); }
    else stage_ids<SH>(P, k, r0, valid, ids_s, own_s);
    if constexpr (RT && !SH) {                                          // Yi et al. Algorithm 2: the thread whose exchange
      if (k == 1 && P.last && P.training && t < valid) {                // saw another step is the sole updater of y
        const int32_t y = ids_s[t];
        const long long prev = (long long)atomicExch(reinterpret_cast<unsigned long long*>(P.last + y), (unsigned long long)tstep);
        if (prev != tstep)
          P.gap[y] = __fadd_rn(__fmul_rn(__fsub_rn(1.f, P.alpha), P.gap[y]), __fmul_rn(P.alpha, __ll2float_rn(tstep - prev)));
      }
    }
    load_tile<1>(buf1, P.W[k], S, 0, E, S);                             // W [K = E][N = S]: MN-major B operand
    __syncthreads();
    gather_tile<0, SH>(buf0, tab.w, P, k, E, ids_s, own_s, valid);   // e [M = samples][K = E]: K-major A operand
    cp_async_commit();
    TTF_OPERANDS_READY();
    if (t == 0) {
      issue_gemm<128, 128, 0, 1>(tmem, tc::smem_u32(buf0), TS, tc::smem_u32(buf1), TS, pad32(E), false);
      tc::mma_commit(tc::smem_u32(&mbar));
    }
    wait_mma();
    tmem_to_staging(tmem, 0, buf2);
    __syncthreads();
    const float* bias = P.W[k] + int64_t(E) * S;
    for (int idx = t; idx < TS * 32; idx += NT) {                       // z = e W + b, whole 512-byte rows per warp
      const int r = idx >> 5, c4 = idx & 31;
      if (r < valid && c4 * 4 < S) {
        float4 v = staging_ld(buf2, r, c4);
        const float4 bb = __ldg(reinterpret_cast<const float4*>(bias) + c4);
        v.x += bb.x; v.y += bb.y; v.z += bb.z; v.w += bb.w;
        *reinterpret_cast<float4*>(P.z[k] + int64_t(r0 + r) * S + c4 * 4) = v;
      }
    }
    tc::fence_before_sync();
  }
  stamp(P, 1);
  brk_grid_barrier(P.bar, bar_target);
  stamp(P, 2);
  if constexpr (RT && !SH) {
    if (P.last && P.training && b == 0 && t == 0) *P.step = tstep;      // every CTA read the counter before the barrier
  }

  // ---------------- phase S: one score tile per CTA ----------------
  const bool tile_cta = b < T * Tc;
  const int ti = b / Tc, tj = b % Tc;
  const int r = (warp & 3) * 32 + lane, h = warp >> 2;                  // this thread's tile row and column half
  const int ig = ti * TS + r;
  float pv[64];                                                         // S_ij, then P_ij: row r, columns [h * 64, h * 64 + 64)
  float mloc = -CUDART_INF_F;                                           // log2-domain maximum of those 64 scores
  const int diag_k = (ti == tj) ? r - h * 64 : -1;                      // this thread's diagonal column, if it has one
  if (tile_cta) {
    load_tile<0>(buf0, P.z[0], S, ti * TS, B, S);                       // q_i [M][K = S]
    load_tile<0>(buf1, P.z[1], S, tj * TS, n, S);                       // c_j [N][K = S]
    cp_async_commit();
    if (t < TS) {
      cand_r[t] = (P.cand && ti * TS + t < B) ? __ldg(P.cand + ti * TS + t) : -1;
      cand_c[t] = (P.cand && tj * TS + t < B) ? __ldg(P.cand + tj * TS + t) : -2;
      if constexpr (SM) { const int j = tj * TS + t; if (P.cand && j >= B && j < n) cand_c[t] = __ldg(P.smp + (j - B)); }
      if constexpr (RT) {                                               // the estimator's gap is read after the F -> S barrier
        const int j = tj * TS + t;
        float l2 = 0.f;
        if (j < B && (P.cand_prob || has_estimator(P))) {
          float p = 1.f;
          if (P.cand_prob) p = __ldg(P.cand_prob + j);
          else { const float gp = estimator_gap(P, __ldg(P.ids[1] + j)); if (gp >= 1.f) p = __frcp_rn(gp); }
          l2 = __log2f(fminf(fmaxf(p, 1e-6f), 1.f));
        }
        lq_s[t] = l2;
      }
    }
    TTF_OPERANDS_READY();
    stamp(P, 8);
    if (t == 0) {
      issue_gemm<128, 128, 0, 0>(tmem, tc::smem_u32(buf0), TS, tc::smem_u32(buf1), TS, pad32(S), false);
      tc::mma_commit(tc::smem_u32(&mbar));
    }
    wait_mma();
    __syncthreads();                                                    // every thread knows the operand tiles are free
    stamp(P, 9);
    // Read-out in the log2 domain (one FFMA + one MUFU.EX2 per score).  pv[k] ends up holding e_k = 2^(s_k - m) with m the
    // maximum of this thread's 64 columns, so that the gradient phase needs ONE scale per thread, not a second exponential
    // per score: P_k = e_k * 2^(m - lse).
    tmem_load64(tmem, warp, h * 64, pv);
    const int32_t my_id = cand_r[r];
    const int ncol = n - tj * TS - h * 64;                              // valid columns of this half (<= 0: none)
    const bool check = P.cand != nullptr;
    float m4[4] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
#pragma unroll
    for (int k = 0; k < 64; k += 4) {
      const int4 cc = *reinterpret_cast<const int4*>(&cand_c[h * 64 + k]);
      const int32_t c4v[4] = {cc.x, cc.y, cc.z, cc.w};
      float l4[4] = {0.f, 0.f, 0.f, 0.f};
      if constexpr (RT) { const float4 lv = *reinterpret_cast<const float4*>(&lq_s[h * 64 + k]); l4[0] = lv.x; l4[1] = lv.y; l4[2] = lv.z; l4[3] = lv.w; }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float v;
        if constexpr (RT) v = fmaf(pv[k + q], kLog2e * P.inv_tau, -l4[q]);     // s / tau - log p, log2 domain
        else v = pv[k + q] * kLog2e;
        if (check && c4v[q] == my_id && k + q != diag_k) v += kMinFloatOver100;
        if (k + q >= ncol) v = -CUDART_INF_F;
        if (k + q == diag_k) diag_s[r] = v;
        pv[k + q] = v;
        m4[q] = fmaxf(m4[q], v);
      }
    }
    mloc = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
    const float msub = mloc == -CUDART_INF_F ? 0.f : mloc;
    float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < 64; ++k) { pv[k] = ex2(pv[k] - msub); s4[k & 3] += pv[k]; }
    pm[h][r] = mloc; ps[h][r] = (s4[0] + s4[1]) + (s4[2] + s4[3]);
    __syncthreads();
    stamp(P, 10);
    if (h == 0) {
      const float m0 = pm[0][r], m1 = pm[1][r], M = fmaxf(m0, m1);
      const float Ms = M == -CUDART_INF_F ? 0.f : M;
      P.part[int64_t(ig) * Tc + tj] = make_float2(M, ps[0][r] * ex2(m0 - Ms) + ps[1][r] * ex2(m1 - Ms));
    }
    if (P.training) {                                                   // the gradient products' B operands travel while the grid
      load_tile<1>(buf0, P.z[1], S, tj * TS, n, S);                     // waits at the barrier: c_j [K = j][N = S]
      load_tile<1>(buf1, P.z[0], S, ti * TS, B, S);                     // q_i [K = i][N = S]
      cp_async_commit();
    }
  }
  stamp(P, 3);
  brk_grid_barrier(P.bar, bar_target);
  stamp(P, 4);
  if (tile_cta) {
    if (SM && h == 0) {                                                 // Tc may exceed 12: two passes over the partials
      float M = -CUDART_INF_F;
      for (int k = 0; k < Tc; ++k) M = fmaxf(M, __ldcg(&P.part[int64_t(ig) * Tc + k]).x);
      float sum = 0.f;
      for (int k = 0; k < Tc; ++k) {
        const float2 pk = __ldcg(&P.part[int64_t(ig) * Tc + k]);
        if (pk.x != -CUDART_INF_F) sum += pk.y * ex2(pk.x - M);
      }
      lse_s[r] = M + __log2f(sum);
    } else if (h == 0) {                                                // log-sum-exp of the row over its T tiles (log2 domain)
      float2 pp[12];                                                    // T <= 12 (T^2 <= SM count): one round trip for all of them
#pragma unroll
      for (int k = 0; k < 12; ++k) pp[k] = k < T ? __ldcg(&P.part[int64_t(ig) * T + k]) : make_float2(-CUDART_INF_F, 0.f);
      float M = -CUDART_INF_F;
#pragma unroll
      for (int k = 0; k < 12; ++k) M = fmaxf(M, pp[k].x);
      float sum = 0.f;
#pragma unroll
      for (int k = 0; k < 12; ++k) if (pp[k].x != -CUDART_INF_F) sum += pp[k].y * ex2(pp[k].x - M);
      lse_s[r] = M + __log2f(sum);
    }
    __syncthreads();
    stamp(P, 11);
    const float lse2 = lse_s[r];
    float wrow = 1.f;                                                   // RT: the row's sample weight
    if constexpr (RT) { if (P.row_weight && ig < B) wrow = __ldg(P.row_weight + ig); }
    if (ti == tj) {                                                     // loss = sum over rows of lse - S[row][row]
      double mine = (h == 0 && ig < B) ? double((lse2 - diag_s[r]) * kLn2) : 0.0;
      if constexpr (RT) mine *= double(wrow);
      const double tot = block_sum_double(mine, red);
      if (t == 0) atomicAdd(P.acc, tot);
    }
    if (P.training) {
      float scale = (ig < B && mloc != -CUDART_INF_F) ? ex2(mloc - lse2) : 0.f;
      float one = 1.f;                                                  // RT: d loss / d logit = w (P - I) / tau
      if constexpr (RT) { one = wrow * P.inv_tau; scale *= one; }
#pragma unroll
      for (int k = 0; k < 64; ++k) pv[k] *= scale;
      if (ig < B && diag_k >= 0 && diag_k < 64) {
#pragma unroll
        for (int k = 0; k < 64; ++k) if (k == diag_k) pv[k] -= one;
      }
      // dq_i += P_ij c_j : A = P [M = i][K = j] K-major, B = c_j [K = j][N = S] MN-major
#pragma unroll
      for (int k = 0; k < 64; k += 4)
        *reinterpret_cast<float4*>(buf2 + km_off16(TS, r, h * 16 + (k >> 2))) = make_float4(pv[k], pv[k + 1], pv[k + 2], pv[k + 3]);
      TTF_OPERANDS_READY();
      stamp(P, 12);
      if (t == 0) {
        issue_gemm<128, 128, 0, 1>(tmem + 128u, tc::smem_u32(buf2), TS, tc::smem_u32(buf0), TS, TS, false);
        tc::mma_commit(tc::smem_u32(&mbar));
      }
      wait_mma();
      __syncthreads();
      stamp(P, 13);
      // dc_j += P_ij^T q_i : A = P [K = i][M = j] MN-major, B = q_i [K = i][N = S] MN-major
#pragma unroll
      for (int k = 0; k < 64; k += 4)
        *reinterpret_cast<float4*>(buf2 + mn_off16(TS, r, h * 16 + (k >> 2))) = make_float4(pv[k], pv[k + 1], pv[k + 2], pv[k + 3]);
      tc::fence_proxy_async_smem();
      __syncthreads();
      tc::fence_after_sync();
      if (t == 0) {
        issue_gemm<128, 128, 1, 1>(tmem, tc::smem_u32(buf2), TS, tc::smem_u32(buf1), TS, TS, false);
        tc::mma_commit(tc::smem_u32(&mbar));
      }
      tmem_to_staging(tmem, 128, buf0);                                  // the dq partial leaves TMEM while that product runs (c_j is consumed)
      __syncthreads();
      for (int idx = t; idx < TS * 32; idx += NT) {                      // row-contiguous REDs of the dq partial
        const int rr = idx >> 5, c4 = idx & 31;
        if (ti * TS + rr < B && c4 * 4 < S) red_add_f4(P.dz[0] + int64_t(ti * TS + rr) * S + c4 * 4, staging_ld(buf0, rr, c4));
      }
      wait_mma();
      __syncthreads();
      stamp(P, 14);
      tmem_to_staging(tmem, 0, buf0);
      __syncthreads();
      for (int idx = t; idx < TS * 32; idx += NT) {
        const int rr = idx >> 5, c4 = idx & 31;
        if (tj * TS + rr < n && c4 * 4 < S) red_add_f4(P.dz[1] + int64_t(tj * TS + rr) * S + c4 * 4, staging_ld(buf0, rr, c4));
      }
      tc::fence_before_sync();
    }
  }
  // phase G's operands that do not depend on the barrier travel across it: the Dense kernel (rows job) or the embedding rows,
  // gathered again straight into the MN-major view (weights job)
  const bool g_cta = P.training && b < (SM ? 2 * (T + Tc) : 4 * T);
  int gk, g_r0, g_valid;
  if constexpr (SM) { gk = b < 2 * T ? 0 : 1; g_r0 = ((b - gk * 2 * T) >> 1) * TS; g_valid = min(TS, (gk ? n : B) - g_r0); }
  else { gk = b / (2 * T); g_r0 = ((b % (2 * T)) >> 1) * TS; g_valid = min(TS, B - g_r0); }
  const int g_job = b & 1;
  if (g_cta) {
    __syncthreads();                                                    // staging and operand tiles of the phase above are done with
    if constexpr (SM) { if (gk == 1) stage_item_ids<SH>(P, g_r0, g_valid, ids_s, own_s); else stage_ids<SH>(P, gk, g_r0, g_valid, ids_s, own_s); }
    else stage_ids<SH>(P, gk, g_r0, g_valid, ids_s, own_s);
    if (g_job == 0) {
      load_tile<0>(buf1, P.W[gk], S, 0, P.E[gk], S);
    } else {
      __syncthreads();
      gather_tile<1, SH>(buf0, (gk == 0 ? P.eu : P.ei).w, P, gk, P.E[gk], ids_s, own_s, g_valid);
    }
    cp_async_commit();
  }
  stamp(P, 5);
  brk_grid_barrier(P.bar, bar_target);
  stamp(P, 6);
  if (b == 0 && t == 0) {                                               // every loss contribution was added before the barrier
    if (P.loss_out) P.loss_out[0] = float(*reinterpret_cast<volatile double*>(P.acc));
    *P.acc = 0.0;
    if (SH || !(P.training && P.do_opt)) P.bar[2] = bar_target;         // base of the next launch
  }

  // ---------------- phase G: gradients of the tower parameters ----------------
  if (g_cta) {
    const int k = gk, job = g_job, r0 = g_r0, valid = g_valid, E = P.E[k];
    const brk_table& tab = k == 0 ? P.eu : P.ei;
    if (job == 0) {
      // de = dz W^T : A = dz [M = samples][K = S] K-major, B = W [N = E][K = S] K-major -> REDs into the rows' accumulators
      load_tile<0>(buf0, P.dz[k], S, r0, SM && k ? n : B, S);
      cp_async_commit();
      TTF_OPERANDS_READY();
      if (t == 0) {
        issue_gemm<128, 128, 0, 0>(tmem, tc::smem_u32(buf0), TS, tc::smem_u32(buf1), TS, pad32(S), false);
        tc::mma_commit(tc::smem_u32(&mbar));
      }
      wait_mma();
      tmem_to_staging(tmem, 0, buf2);
      __syncthreads();
      for (int idx = t; idx < TS * 32; idx += NT) {
        const int rr = idx >> 5, c4 = idx & 31;
        if (rr < valid) {
          const int64_t row = ids_s[rr];
          if constexpr (SH) {                                           // the owner's accumulator and bitmask (never null)
            const brk_shards& sh = k == 0 ? P.su : P.si;
            const int o = own_s[rr];
            if (c4 * 4 < E) red_add_f4(sh.g[o] + row * E + c4 * 4, staging_ld(buf2, rr, c4));
            if (c4 == 0) asm volatile("red.global.or.b32 [%0], %1;" ::"l"(sh.touched[o] + (row >> 5)), "r"(1u << (row & 31)) : "memory");
          } else {
            if (c4 * 4 < E) red_add_f4(tab.g + row * E + c4 * 4, staging_ld(buf2, rr, c4));
            if (c4 == 0 && tab.touched) asm volatile("red.global.or.b32 [%0], %1;" ::"l"(tab.touched + (row >> 5)), "r"(1u << (row & 31)) : "memory");
          }
        }
      }
    } else {
      // dW += e^T dz : A = e [K = samples][M = E] MN-major (gathered again, straight into that view), B = dz [K][N = S] MN-major
      load_tile<1>(buf1, P.dz[k], S, r0, SM && k ? n : B, S);
      cp_async_commit();
      TTF_OPERANDS_READY();
      if (t == 0) {
        issue_gemm<128, 128, 1, 1>(tmem, tc::smem_u32(buf0), TS, tc::smem_u32(buf1), TS, TS, false);
        tc::mma_commit(tc::smem_u32(&mbar));
      }
      if (t < S) {                                                      // db = column sums of dz, on the CUDA cores meanwhile
        float sacc = 0.f;
        for (int rr = 0; rr < TS; ++rr) sacc += *reinterpret_cast<const float*>(buf1 + mn_off16(TS, rr, t >> 2) + (t & 3) * 4);
        atomicAdd(P.gW[k] + int64_t(E) * S + t, sacc);
      }
      wait_mma();
      tmem_to_staging(tmem, 0, buf2);
      __syncthreads();
      for (int idx = t; idx < TS * 32; idx += NT) {
        const int e = idx >> 5, c4 = idx & 31;
        if (e < E && c4 * 4 < S) red_add_f4(P.gW[k] + int64_t(e) * S + c4 * 4, staging_ld(buf2, e, c4));
      }
    }
    tc::fence_before_sync();
  }
  stamp(P, 7);
  // ---------------- phase O: Keras Adagrad (optim.cu AdagradOp) on what this step touched ----------------
  if (!SH && P.training && P.do_opt) {
    brk_grid_barrier(P.bar, bar_target);
    if (b == 0 && t == 0) P.bar[2] = bar_target;
    // rows: every warp takes a run of `per` (tower, sample) pairs, one per lane: the ids are loaded and the touched bits
    // cleared in ONE round trip each (the lane whose atomicAnd saw the bit set owns the row -- ids repeat in a batch); then
    // the warp walks its run, two rows' loads in flight, E/4 lanes per row
    {
      const int nwarps = int(gridDim.x) * (NT / 32), gw = b * (NT / 32) + warp;
      const int npairs = SM ? B + n : 2 * B;                            // SM: the sampled rows after the batch's
      const int per = (npairs + nwarps - 1) / nwarps;                   // <= 32: 2B <= 8 * 32 * max(T^2, 4T)
      const int x = gw * per + lane;
      const bool mine = lane < per && x < npairs;
      const int k = x >= B ? 1 : 0;
      int64_t row = 0;
      uint32_t own = 0u;
      if (mine) {
        const brk_table& tab = k == 0 ? P.eu : P.ei;
        if constexpr (SM) row = x < 2 * B ? __ldg(P.ids[k] + (x - k * B)) : __ldg(P.smp + (x - 2 * B));
        else row = __ldg(P.ids[k] + (x - k * B));
        const uint32_t bit = 1u << (row & 31);
        own = atomicAnd(tab.touched + (row >> 5), ~bit) & bit;
      }
      float* base = nullptr;                                            // this lane's row, if it owns one
      float* accb = nullptr; float* grdb = nullptr;
      if (own) { const brk_table& tab = k == 0 ? P.eu : P.ei; base = tab.w + row * P.E[k]; accb = tab.m + row * P.E[k]; grdb = tab.g + row * P.E[k]; }
      const int Ek = P.E[k];
      for (int j0 = 0; j0 < per; j0 += 2) {
        float4 w4[2], a4[2], g4[2];
        float4* wp[2]; float4* ap[2]; float4* gp[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int j = j0 + q < 32 ? j0 + q : 31;
          float* bj = reinterpret_cast<float*>(__shfl_sync(0xffffffffu, reinterpret_cast<unsigned long long>(base), j));
          float* aj = reinterpret_cast<float*>(__shfl_sync(0xffffffffu, reinterpret_cast<unsigned long long>(accb), j));
          float* gj = reinterpret_cast<float*>(__shfl_sync(0xffffffffu, reinterpret_cast<unsigned long long>(grdb), j));
          const int Ej = __shfl_sync(0xffffffffu, Ek, j);
          const bool go = j0 + q < per && bj != nullptr && lane * 4 < Ej;
          wp[q] = go ? reinterpret_cast<float4*>(bj) + lane : nullptr;
          ap[q] = reinterpret_cast<float4*>(aj) + lane; gp[q] = reinterpret_cast<float4*>(gj) + lane;
          if (go) { w4[q] = *wp[q]; a4[q] = *ap[q]; g4[q] = *gp[q]; }
        }
#pragma unroll
        for (int q = 0; q < 2; ++q)
          if (wp[q] != nullptr) {
            float4 w = w4[q], a = a4[q];
            const float4 g = g4[q];
            a.x += g.x * g.x; w.x -= P.lr * g.x / (sqrtf(a.x) + P.eps);
            a.y += g.y * g.y; w.y -= P.lr * g.y / (sqrtf(a.y) + P.eps);
            a.z += g.z * g.z; w.z -= P.lr * g.z / (sqrtf(a.z) + P.eps);
            a.w += g.w * g.w; w.w -= P.lr * g.w / (sqrtf(a.w) + P.eps);
            *wp[q] = w; *ap[q] = a; *gp[q] = make_float4(0.f, 0.f, 0.f, 0.f);
          }
      }
    }
    for (int k = 0; k < 2; ++k) {
      const int64_t n4 = P.dn[k].rows * P.dn[k].d / 4;
      for (int64_t x = int64_t(b) * NT + t; x < n4; x += int64_t(gridDim.x) * NT)
        adagrad4(reinterpret_cast<float4*>(P.dn[k].w) + x, reinterpret_cast<float4*>(P.dn[k].m) + x, reinterpret_cast<float4*>(P.dn[k].g) + x,
                 P.lr, P.eps);
    }
    stamp(P, 15);
  }
  __syncthreads();
  if (t < 32) tc::tmem_dealloc<256>(tmem);
}

}  // namespace ttf

// Internal entry (twotower.cu): *handled = 0 when the shape is not this kernel's (the caller then takes the multi-kernel step).
// sh != nullptr: the tables are row-sharded (brk_twotower_step_sharded, training only, do_opt = 0); the embedding
// tables of user / item are then not read.  rt: the options on unsharded tables, srt: on sharded ones (null: none).
int brk_twotower_step_fused(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u, const int32_t* i,
                            const int32_t* cand_ids, int64_t batch, int32_t training, const brk_twotower_workspace* ws,
                            float* loss_out, cudaStream_t st, int* handled, int do_opt, float lr, float eps,
                            const brk_twotower_shards* sh, const brk_tt_retrieval* rt, const brk_tt_retrieval_sharded* srt,
                            const brk_tt_sampled* smp) {
  using namespace ttf;
  *handled = 0;
  const int S = user->S, B = int(batch), T = (B + TS - 1) / TS;
  // sampled negatives: the item side has n = B + M rows in Tc row blocks; T * Tc score tiles, 2 (T + Tc) tower blocks
  const int n = smp ? B + int(smp->count) : B, Tc = (n + TS - 1) / TS;
  const int need = smp ? (T * Tc > 2 * (T + Tc) ? T * Tc : 2 * (T + Tc)) : (T * T > 4 * T ? T * T : 4 * T);
  const int grid = need > ctx->sm_count ? need : ctx->sm_count;   // the CTAs without a tile share the zeroing and the optimizer phase
  if (getenv("BRK_TT_NO_FUSED")) return 0;
  if (S > 128 || user->E > 128 || item->E > 128 || (S & 3) || (user->E & 3) || (item->E & 3) || need > ctx->sm_count || T > 12) return 0;
  const brk_tower* tw[2] = {user, item};
  if (sh != nullptr) {
    if (!training || do_opt) return 0;
    const brk_shards* s2[2] = {&sh->user, &sh->item};
    for (int k = 0; k < 2; ++k)
      for (int p = 0; p < s2[k]->world; ++p)
        if (!brk_aligned16(s2[k]->w[p]) || !brk_aligned16(s2[k]->g[p])) return 0;
  }
  for (int k = 0; k < 2; ++k)
    if ((!sh && !brk_aligned16(tw[k]->emb.w)) || !brk_aligned16(tw[k]->dense.w) ||
        (training && ((!sh && !brk_aligned16(tw[k]->emb.g)) || !brk_aligned16(tw[k]->dense.g))))
      return 0;
  if (!brk_aligned16(ws->q) || !brk_aligned16(ws->c) || (training && (!brk_aligned16(ws->dq) || !brk_aligned16(ws->dc)))) return 0;
  const size_t smem = 3 * size_t(TILE) + 1024;
  if (sh && rt) return 0;                                          // unsharded options on sharded tables: not a caller's call
  if (smp && !training) return 0;
  const int kv = smp ? (sh ? 5 : 4) : (sh ? (srt ? 3 : 1) : (rt ? 2 : 0));
  const void* kern = smp ? (sh ? (const void*)fused_step<true, true, true> : (const void*)fused_step<false, true, true>)
                   : sh ? (srt ? (const void*)fused_step<true, true> : (const void*)fused_step<true>)
                        : (rt ? (const void*)fused_step<false, true> : (const void*)fused_step<false>);
  // the shared-memory opt-in is per device: set it for the current one; occupancy is a property of each instantiation,
  // queried once
  BRK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  static int per_sm[6] = {-1, -1, -1, -1, -1, -1};
  int& occ = per_sm[kv];
  if (occ < 0) BRK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NT, smem));
  if (grid > occ * ctx->sm_count) return 0;
  const size_t part_floats = size_t(T) * TS * Tc * 2;
  if (ctx->tt_part_floats < part_floats) {
    if (ctx->tt_part) BRK_CUDA(cudaFree(ctx->tt_part));
    ctx->tt_part = nullptr; ctx->tt_part_floats = 0;
    BRK_CUDA(cudaMalloc(&ctx->tt_part, part_floats * sizeof(float)));
    ctx->tt_part_floats = part_floats;
  }
  ShardedParams P;                                    // fused_step<false> reads its Params base (at offset 0)
  memset(&P, 0, sizeof(P));
  P.eu = user->emb; P.ei = item->emb;
  for (int k = 0; k < 2; ++k) { P.W[k] = tw[k]->dense.w; P.gW[k] = tw[k]->dense.g; P.E[k] = tw[k]->E; }
  P.S = S; P.ids[0] = u; P.ids[1] = i; P.cand = cand_ids;
  P.B = B; P.T = T; P.training = training;
  P.z[0] = ws->q; P.z[1] = ws->c; P.dz[0] = ws->dq; P.dz[1] = ws->dc;
  P.part = reinterpret_cast<float2*>(ctx->tt_part);
  P.acc = ws->acc; P.loss_out = loss_out; P.bar = ctx->bar[BRK_BAR_TT];
  const char* tr = getenv("BRK_TT_TRACE");
  P.trace = tr ? reinterpret_cast<unsigned long long*>(strtoull(tr, nullptr, 16)) : nullptr;
  if (do_opt && training) {                           // in-kernel Adagrad needs the touched bitmasks (row ownership) and float4 blocks
    bool ok = true;
    for (int k = 0; k < 2; ++k) {
      const brk_table& e = tw[k]->emb; const brk_table& d = tw[k]->dense;
      ok = ok && e.touched && e.m && d.m && brk_aligned16(e.m) && brk_aligned16(d.m) && ((d.rows * d.d) & 3) == 0;
    }
    if (!ok) return 0;
    P.do_opt = 1; P.lr = lr; P.eps = eps;
    P.dn[0] = user->dense; P.dn[1] = item->dense;
  }
  if (sh) { P.su = sh->user; P.si = sh->item; }
  RetrievalParams R;
  memset(&R, 0, sizeof(R));
  if (rt) {
    static_cast<Params&>(R) = static_cast<const Params&>(P);
    R.cand_prob = rt->cand_prob; R.row_weight = rt->row_weight;
    R.last = reinterpret_cast<long long*>(rt->last); R.gap = rt->gap; R.step = reinterpret_cast<long long*>(rt->step);
    R.inv_tau = rt->inv_temperature; R.alpha = rt->alpha;
  }
  ShardedRetrievalParams SR;
  memset(&SR, 0, sizeof(SR));
  if (sh && srt) {
    static_cast<ShardedParams&>(SR) = P;
    SR.cand_prob = srt->cand_prob; SR.row_weight = srt->row_weight; SR.inv_tau = srt->inv_temperature;
    if (srt->est)
      for (int p = 0; p < srt->est->world; ++p) SR.gap[p] = srt->est->gap[p];
  }
  // sampled negatives: the options block with no probabilities or estimator (rejected by the callers), then the draws
  SampledParams SM_;
  ShardedSampledParams SSM;
  memset(&SM_, 0, sizeof(SM_));
  memset(&SSM, 0, sizeof(SSM));
  if (smp) {
    if (sh) {
      static_cast<ShardedParams&>(SSM) = P;
      SSM.row_weight = srt ? srt->row_weight : nullptr; SSM.inv_tau = srt ? srt->inv_temperature : 1.f;
      SSM.smp = smp->ids; SSM.M = int(smp->count); SSM.n = n; SSM.Tc = Tc;
    } else {
      static_cast<Params&>(SM_) = static_cast<const Params&>(P);
      SM_.row_weight = rt ? rt->row_weight : nullptr; SM_.inv_tau = rt ? rt->inv_temperature : 1.f;
      SM_.smp = smp->ids; SM_.M = int(smp->count); SM_.n = n; SM_.Tc = Tc;
    }
  }
  void* args[] = {smp ? (sh ? (void*)&SSM : (void*)&SM_)
                      : sh ? (srt ? (void*)&SR : (void*)&P) : (rt ? (void*)&R : (void*)static_cast<Params*>(&P))};
  BRK_CUDA(cudaLaunchCooperativeKernel(kern, dim3(grid), dim3(NT), args, smem, st));
  *handled = 1;
  return 0;
}
