// Two-tower training step with GLOBAL in-batch negatives (brk_twotower_step_global, include/brk_b200.h): every rank's
// queries are scored against the candidates of the whole global batch.  The step is split at its two cross-GPU
// dependencies into three launches on the caller's stream, with a brk_peer_barrier between them issued by the caller:
//   phase 0  towers (twotower.cu's tower_forward); the candidate vectors go straight into this rank's symmetric block,
//            its ids and header {count, S} beside them;
//   phase 1  gather of the world candidate blocks (16-byte peer loads) into one local [n, S] buffer, scores Q C^T
//            [b, n], the rectangular masked softmax, dq = (P - Y) C and this rank's dc partial (P - Y)^T Q [n, S] into
//            its slot buffer;
//   phase 2  the owner sums rows [o_r, o_r + b_r) of every rank's slot in rank order (fixed order: reproducible), then
//            the Dense / row gradients of both towers as in the one-replica step.
// No launch spans a cross-GPU wait, so one process can issue the phases of G emulated ranks in turn on one GPU.
// One slot buffer per rank is enough: a rank writes its slot in phase 1 of step s + 1 only after the phase-0 barrier
// of that step, which no rank passes before every rank has issued (stream order) its phase 2 of step s, the last
// reader of the slots; the candidate blocks are likewise last read in phase 1 and next written after the phase-1
// barrier.  Everything runs on `stream` (no fork): the barriers then order all of a phase's work.
// Algorithmic work per rank and step: 3 * 2 b n S FLOP for the products (b = this rank's rows), 4 n S bytes gathered
// from the peers and 4 G b S bytes read by the owner reduce.
#include "common.cuh"
#include <math_constants.h>

int brk_tt_gemm(brk_ctx* ctx, cudaStream_t st, int tcore, const float* A, const float* B, float* C, int M, int N, int K, int lda,
                int ldb, int ldc, int ta, int tb, int accumulate, bool allow_split);                           // twotower.cu
int brk_tt_tower_forward(brk_ctx* ctx, const brk_tower* t, const int32_t* ids, int64_t n, float* emb_out, float* out, int tcore,
                         cudaStream_t st, const brk_shards* sh);
int brk_tt_colsum(cudaStream_t st, const float* X, int M, int N, float* out);
int brk_tt_check_shards(const brk_shards* s, int32_t E, const char* which, const char* fn);

namespace {

constexpr float kMinFloatOver100 = -3.4028234663852886e36f;     // np.finfo(np.float32).min / 100
constexpr int kHeader = 4;                                      // int32 words ahead of the ids: {count, S, 0, 0}

struct Blocks {                                                 // the peer blocks a launch reads, by value
  const float* cand[BRK_MAX_PEERS];
  const int32_t* ids[BRK_MAX_PEERS];
  const float* slot[BRK_MAX_PEERS];
  int offset[BRK_MAX_PEERS], count[BRK_MAX_PEERS];
};

// Header and ids of this rank's slice (phase 0).
__global__ void publish_ids_kernel(const int32_t* __restrict__ ids, int n, int S, int32_t* __restrict__ out) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < kHeader) out[j] = j == 0 ? n : (j == 1 ? S : 0);
  if (j < n) out[kHeader + j] = __ldg(ids + j);
}

// c_all rows [o_p, o_p + b_p) <- block p (blockIdx.y = p), 16-byte loads; ids likewise.  A header that disagrees with
// the caller's split sets *err = 1 + p (the first such p wins); the copy still stays inside the blocks' capacity.
__global__ void __launch_bounds__(256)
gather_blocks_kernel(Blocks b, int S4, float4* __restrict__ c_all, int32_t* __restrict__ ids_all, int32_t* __restrict__ err) {
  const int p = blockIdx.y, n = b.count[p];
  if (n == 0) return;
  const int32_t* ids = b.ids[p];
  if (blockIdx.x == 0 && threadIdx.x == 0 && (ids[0] != n || ids[1] != 4 * S4)) atomicCAS(err, 0, 1 + p);
  const float4* src = reinterpret_cast<const float4*>(b.cand[p]);
  float4* dst = c_all + int64_t(b.offset[p]) * S4;
  const int64_t total = int64_t(n) * S4;
  for (int64_t e = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; e < total; e += int64_t(gridDim.x) * blockDim.x) {
    dst[e] = ldg_nc_f4(src + e);
    if (e < n) ids_all[b.offset[p] + e] = ids[kHeader + e];
  }
}

// One CTA per query row of the [b, n] score matrix: label column off + row, accidental hits (another candidate with
// the row's positive id) masked, log-sum-exp, loss, and in place P - Y.  inbatch_softmax_kernel (twotower.cu) is the
// square case off = 0, n = b.
__global__ void __launch_bounds__(256)
global_softmax_kernel(float* __restrict__ Sc, const int32_t* __restrict__ ids_all, int n, int off, double* __restrict__ loss_acc) {
  __shared__ float redf[32];
  __shared__ double redd[32];
  __shared__ float lse_sm;
  const int row = blockIdx.x, t = threadIdx.x, label = off + row;
  float* s = Sc + int64_t(row) * n;
  const int32_t pos_id = __ldg(ids_all + label);
  float mx = -CUDART_INF_F;
  for (int j = t; j < n; j += 256) {
    float v = s[j];
    if (j != label && __ldg(ids_all + j) == pos_id) { v += kMinFloatOver100; s[j] = v; }
    mx = fmaxf(mx, v);
  }
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((t & 31) == 0) redf[t >> 5] = mx;
  __syncthreads();
  mx = redf[0];
#pragma unroll
  for (int w = 1; w < 8; ++w) mx = fmaxf(mx, redf[w]);
  double sum = 0.0;
  for (int j = t; j < n; j += 256) sum += double(expf(s[j] - mx));
  sum = block_sum_double(sum, redd);
  if (t == 0) {
    const float lse = mx + logf(float(sum));
    lse_sm = lse;
    atomicAdd(loss_acc, double(lse - s[label]));
  }
  __syncthreads();
  const float lse = lse_sm;
  for (int j = t; j < n; j += 256) s[j] = expf(s[j] - lse) - (j == label ? 1.f : 0.f);
}

__global__ void finish_loss_kernel(double* acc, float* loss_out) {
  if (loss_out) loss_out[0] = float(acc[0]);
  acc[0] = 0.0;
}

// dc [b, S] = sum over p = 0, 1, ..., G - 1 of slot_p rows [off, off + b): the owner's fixed-order reduce (phase 2).
__global__ void __launch_bounds__(256)
owner_reduce_kernel(Blocks bl, int G, int off, int b, int S4, float4* __restrict__ dc) {
  const int64_t total = int64_t(b) * S4, base = int64_t(off) * S4;
  for (int64_t e = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; e < total; e += int64_t(gridDim.x) * blockDim.x) {
    float4 s = ldg_nc_f4(reinterpret_cast<const float4*>(bl.slot[0]) + base + e);
    for (int p = 1; p < G; ++p) {
      const float4 v = ldg_nc_f4(reinterpret_cast<const float4*>(bl.slot[p]) + base + e);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    dc[e] = s;
  }
}

int grid_for(brk_ctx* ctx, int64_t work) {
  const int64_t want = (work + 255) / 256, cap = int64_t(ctx->sm_count) * 8;
  return int(want < 1 ? 1 : (want < cap ? want : cap));
}

// Dense and embedding-row gradients of one tower from dz [b, S], in twotower_step's order: dW += e^T dz, db += column
// sums of dz, de = dz W^T, then the rows' scatter (local table with touched bits, or REDs into the owners' shards).
int tower_backward(brk_ctx* ctx, cudaStream_t st, int tcore, const brk_tower* t, const float* e, const float* dz, float* de,
                   const int32_t* ids, int b, const brk_shards* sh) {
  const int E = t->E, S = t->S;
  int rc;
  float* gW = t->dense.g;
  if ((rc = brk_tt_gemm(ctx, st, tcore, e, dz, gW, E, S, b, E, S, S, 1, 0, 1, true))) return rc;
  if ((rc = brk_tt_colsum(st, dz, b, S, gW + int64_t(E) * S))) return rc;
  if ((rc = brk_tt_gemm(ctx, st, tcore, dz, t->dense.w, de, b, E, S, S, S, E, 0, 1, 0, false))) return rc;
  return sh ? brk_scatter_add_rows_sharded(ctx, sh, E, ids, b, de, (void*)st)
            : brk_scatter_add_rows(ctx, t->emb.g, t->emb.rows, E, ids, b, de, t->emb.touched, 0, (void*)st);
}

}  // namespace

extern "C" int brk_twotower_step_global(brk_ctx* ctx, int32_t phase, const brk_tower* user, const brk_tower* item,
                                        const brk_twotower_shards* sh, const brk_twotower_global* g, const int32_t* u,
                                        const int32_t* i, int32_t mode, const brk_twotower_workspace* ws, float* loss_out,
                                        void* stream) {
  static const char* fn = "brk_twotower_step_global";
  BRK_REQUIRE(ctx && user && item && g && ws, BRK_E_ARG, "%s: null argument", fn);
  BRK_REQUIRE(phase >= 0 && phase <= 2, BRK_E_ARG, "%s: phase %d (0..2)", fn, phase);
  BRK_REQUIRE((mode & ~0x100) == 0, BRK_E_ARG, "%s: mode 0x%x (0 or 0x100; rdZero has no in-batch negatives)", fn, mode);
  const int G = g->world, r = g->rank;
  BRK_REQUIRE(G >= 1 && G <= BRK_MAX_PEERS, BRK_E_ARG, "%s: world=%d (1..%d)", fn, G, BRK_MAX_PEERS);
  BRK_REQUIRE(r >= 0 && r < G, BRK_E_ARG, "%s: rank=%d world=%d", fn, r, G);
  const int S = user->S;
  BRK_REQUIRE(user->S == item->S && S > 0 && (S & 3) == 0, BRK_E_ARG,
              "%s: S %d vs %d (equal positive multiples of 4)", fn, user->S, item->S);
  BRK_REQUIRE(user->E > 0 && item->E > 0, BRK_E_ARG, "%s: E %d / %d", fn, user->E, item->E);
  int64_t n = 0;
  for (int p = 0; p < G; ++p) {
    BRK_REQUIRE(g->offset[p] == n && g->count[p] >= 0 && g->count[p] <= g->cap, BRK_E_ARG,
                "%s: rank %d's slice [%lld, +%lld) does not continue [0, %lld) (or exceeds cap %lld)", fn, p,
                (long long)g->offset[p], (long long)g->count[p], (long long)n, (long long)g->cap);
    n += g->count[p];
  }
  BRK_REQUIRE(n <= g->n_cap && n < (1 << 30), BRK_E_ARG, "%s: n=%lld (n_cap %lld)", fn, (long long)n, (long long)g->n_cap);
  const int b = int(g->count[r]), off = int(g->offset[r]);
  BRK_REQUIRE(int64_t(b) * n < (int64_t(1) << 31), BRK_E_ARG, "%s: score matrix [%d, %lld] too large", fn, b, (long long)n);
  int rc;
  if (sh) {
    if ((rc = brk_tt_check_shards(&sh->user, user->E, "user", fn))) return rc;
    if ((rc = brk_tt_check_shards(&sh->item, item->E, "item", fn))) return rc;
    BRK_REQUIRE(sh->user.world == G && sh->item.world == G && sh->user.rank == r && sh->item.rank == r, BRK_E_ARG,
                "%s: shards of world %d / %d, rank %d / %d, not %d / %d", fn, sh->user.world, sh->item.world, sh->user.rank,
                sh->item.rank, G, r);
  }
  if (n == 0) return 0;
  for (int p = 0; p < G; ++p) {
    BRK_REQUIRE(g->slot[p] && (g->count[p] == 0 || (g->cand[p] && g->ids[p])), BRK_E_ARG,
                "%s: rank %d's candidate / id / slot buffer is null", fn, p);
  }
  BRK_REQUIRE(g->ids[r] && g->c_all && g->ids_all && g->err, BRK_E_ARG, "%s: ids / c_all / ids_all / err is null", fn);
  if (b > 0) {
    BRK_REQUIRE(u && i, BRK_E_ARG, "%s: null ids", fn);
    BRK_REQUIRE(ws->eu && ws->ei && ws->q && ws->dq && ws->dc && ws->scores && ws->acc && ws->deu && ws->dei, BRK_E_ARG,
                "%s: workspace missing", fn);
    BRK_REQUIRE(user->dense.w && item->dense.w && user->dense.g && item->dense.g, BRK_E_ARG,
                "%s: Dense blocks or their gradients missing", fn);
    BRK_REQUIRE(sh || (user->emb.w && item->emb.w && user->emb.g && item->emb.g), BRK_E_ARG,
                "%s: tables or their gradients missing (no shards given)", fn);
  }
  const int tcore = (mode & 0x100) ? 1 : 0;
  cudaStream_t st = (cudaStream_t)stream;
  const brk_shards* tsh[2] = {sh ? &sh->user : nullptr, sh ? &sh->item : nullptr};
  Blocks bl;
  for (int p = 0; p < BRK_MAX_PEERS; ++p) {
    const bool in = p < G;
    bl.cand[p] = in ? g->cand[p] : nullptr; bl.ids[p] = in ? g->ids[p] : nullptr; bl.slot[p] = in ? g->slot[p] : nullptr;
    bl.offset[p] = in ? int(g->offset[p]) : 0; bl.count[p] = in ? int(g->count[p]) : 0;
  }
  const int S4 = S / 4;
  if (phase == 0) {
    if (b > 0) {
      if ((rc = brk_tt_tower_forward(ctx, item, i, b, ws->ei, g->cand[r], tcore, st, tsh[1]))) return rc;
      if ((rc = brk_tt_tower_forward(ctx, user, u, b, ws->eu, ws->q, tcore, st, tsh[0]))) return rc;
    }
    publish_ids_kernel<<<(b + kHeader + 255) / 256, 256, 0, st>>>(i, b, S, g->ids[r]);
    BRK_LAUNCH_CHECK();
    return 0;
  }
  if (phase == 1) {
    float* slot = g->slot[r];
    if (b == 0) {                                    // no queries: this rank's partial is zero for every candidate
      BRK_CUDA(cudaMemsetAsync(slot, 0, size_t(n) * S * sizeof(float), st));
      if (loss_out) BRK_CUDA(cudaMemsetAsync(loss_out, 0, sizeof(float), st));
      return 0;
    }
    int maxc = 0;
    for (int p = 0; p < G; ++p) maxc = bl.count[p] > maxc ? bl.count[p] : maxc;
    const int gx = (grid_for(ctx, int64_t(maxc) * S4) + G - 1) / G;
    gather_blocks_kernel<<<dim3(gx, G), 256, 0, st>>>(bl, S4, reinterpret_cast<float4*>(g->c_all), g->ids_all, g->err);
    BRK_LAUNCH_CHECK();
    const int N = int(n);
    BRK_CUDA(cudaMemsetAsync(ws->dq, 0, size_t(b) * S * sizeof(float), st));     // RED target of the split-K product
    // scores = q C_all^T [b, n]
    if ((rc = brk_tt_gemm(ctx, st, tcore, ws->q, g->c_all, ws->scores, b, N, S, S, S, N, 0, 1, 0, false))) return rc;
    global_softmax_kernel<<<b, 256, 0, st>>>(ws->scores, g->ids_all, N, off, ws->acc);
    BRK_LAUNCH_CHECK();
    finish_loss_kernel<<<1, 1, 0, st>>>(ws->acc, loss_out);
    BRK_LAUNCH_CHECK();
    // dq = (P - Y) C_all [b, S]: few output tiles, long K = n -> split-K with REDs
    if ((rc = brk_tt_gemm(ctx, st, tcore, ws->scores, g->c_all, ws->dq, b, S, N, N, S, S, 0, 0, 1, true))) return rc;
    // this rank's partial (P - Y)^T q [n, S]: row j is candidate j's share from these queries
    return brk_tt_gemm(ctx, st, tcore, ws->scores, ws->q, slot, N, S, b, N, S, S, 1, 0, 0, false);
  }
  if (b == 0) return 0;
  owner_reduce_kernel<<<grid_for(ctx, int64_t(b) * S4), 256, 0, st>>>(bl, G, off, b, S4, reinterpret_cast<float4*>(ws->dc));
  BRK_LAUNCH_CHECK();
  if ((rc = tower_backward(ctx, st, tcore, user, ws->eu, ws->dq, ws->deu, u, b, tsh[0]))) return rc;
  return tower_backward(ctx, st, tcore, item, ws->ei, ws->dc, ws->dei, i, b, tsh[1]);
}
