// Two-tower training step: /root/reference/trainers/twoTower.py:19-111.
//   towers   : Embedding[E] -> Dense(S) linear (twoTower.py:40-41; StringLookup indices come from the host)
//   loss     : tfrs.tasks.Retrieval as called at :82-83 -- scores = Q C^T [B,B], labels = identity,
//              accidental hits (another row's candidate id equals this row's positive id) get
//              finfo(float32).min/100 added, categorical cross-entropy from logits, reduction SUM;
//              or (rdZero, :85-87) sigmoid(<q,c>) against RATING_TYPE with mean BCE.
//   backward : P = softmax(scores) - I;  dQ = P C, dC = P^T Q;  Dense and embedding gradients.
// fp32 throughout (this is the exact-parity path): the products are a register-tiled CUDA-core SGEMM
// (64x64x16 tiles, 4x4 per thread, transposes folded into the tile loads, optional split-K with RED
// accumulation for the weight gradients whose output is a single 128x128 tile); the row softmax +
// loss + gradient-of-logits is one fused kernel over the materialised score matrix.
// Algorithmic work per step: 3 * 2 B^2 S FLOP for the in-batch products + 6 * 2 B E S for the towers;
// bytes: 2 rows gathered + 2 row gradients per interaction (8E B each way) + 12 B^2 for the scores.
#include "common.cuh"
#include <math_constants.h>
#include <cmath>

namespace {

constexpr int TM = 64, TN = 64, TK = 16, kGemmThreads = 256;

// C[M,N] (op)= alpha * opA(A) * opB(B) (+ bias[N])
//   ta == 0: A is [M,K] row-major (lda = K-stride);  ta == 1: A is stored [K,M] (A^T used)
//   tb == 0: B is [K,N] row-major;                    tb == 1: B is stored [N,K]
//   accumulate != 0: C += (RED.ADD when split-K > 1, plain += otherwise); bias added by split 0 only
//   grid: x = row tile * column tiles + column tile (gridDim.y would cap M at 65535 row tiles), z = K split
__global__ void __launch_bounds__(kGemmThreads)
sgemm_kernel(const float* __restrict__ A, const float* __restrict__ Bm, float* __restrict__ C,
             const float* __restrict__ bias, int M, int N, int K, int lda, int ldb, int ldc, int ta, int tb,
             float alpha, int accumulate, int k_per_split) {
  __shared__ __align__(16) float As[TK][TM + 4];
  __shared__ __align__(16) float Bs[TK][TN + 4];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;       // 16 x 16 threads, 4x4 outputs each
  const unsigned col_tiles = unsigned(N + TN - 1) / TN;
  const int m0 = int(blockIdx.x / col_tiles) * TM, n0 = int(blockIdx.x % col_tiles) * TN;
  const int kbeg = blockIdx.z * k_per_split, kend = min(K, kbeg + k_per_split);
  float acc[4][4] = {};
  for (int k0 = kbeg; k0 < kend; k0 += TK) {
    // stage A tile as As[k][m] and B tile as Bs[k][n]; 1024 elements each, 4 per thread
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int idx = threadIdx.x + e * kGemmThreads;
      int m, k;
      if (ta == 0) { m = idx / TK; k = idx % TK; } else { k = idx / TM; m = idx % TM; }
      const int gm = m0 + m, gk = k0 + k;
      float v = 0.f;
      if (gm < M && gk < kend) v = ta == 0 ? __ldg(A + int64_t(gm) * lda + gk) : __ldg(A + int64_t(gk) * lda + gm);
      As[k][m] = v;
      int n, kk;
      if (tb == 0) { kk = idx / TN; n = idx % TN; } else { n = idx / TK; kk = idx % TK; }
      const int gn = n0 + n, gk2 = k0 + kk;
      float w = 0.f;
      if (gn < N && gk2 < kend) w = tb == 0 ? __ldg(Bm + int64_t(gk2) * ldb + gn) : __ldg(Bm + int64_t(gn) * ldb + gk2);
      Bs[kk][n] = w;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TK; ++k) {
      const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
  const bool split = gridDim.z > 1;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gm = m0 + ty * 4 + i;
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gn = n0 + tx * 4 + j;
      if (gn >= N) continue;
      float v = alpha * acc[i][j];
      if (bias != nullptr && blockIdx.z == 0) v += __ldg(bias + gn);
      float* dst = C + int64_t(gm) * ldc + gn;
      if (split) atomicAdd(dst, v);
      else if (accumulate) *dst += v;
      else *dst = v;
    }
  }
}

int sgemm(brk_ctx* ctx, cudaStream_t st, const float* A, const float* B, float* C, const float* bias, int M, int N,
          int K, int lda, int ldb, int ldc, int ta, int tb, float alpha, int accumulate, bool allow_split) {
  const int gx = (N + TN - 1) / TN, gy = (M + TM - 1) / TM;
  int splits = 1;
  if (allow_split && accumulate) {                      // few output tiles, long K: split K across CTAs
    const int want = (2 * ctx->sm_count) / (gx * gy);
    const int max_by_k = (K + 4 * TK - 1) / (4 * TK);
    splits = want < 1 ? 1 : (want < max_by_k ? want : max_by_k);
    if (splits > 64) splits = 64;
    if (splits < 1) splits = 1;
  }
  int kps = ((K + splits - 1) / splits + TK - 1) / TK * TK;
  splits = (K + kps - 1) / kps;
  sgemm_kernel<<<dim3(unsigned(gx) * unsigned(gy), 1, splits), kGemmThreads, 0, st>>>(A, B, C, bias, M, N, K, lda, ldb, ldc,
                                                                                      ta, tb, alpha, accumulate, kps);
  BRK_LAUNCH_CHECK();
  return 0;
}

// out[n] += sum_m X[m][n]: bias gradients (ones^T dz) without a degenerate M = 1 product.  A block sums the 64-row chunks
// blockIdx.y, blockIdx.y + gridDim.y, ... and adds its sum once; gridDim.y is capped at 65535, below which a block has
// one chunk.
__global__ void __launch_bounds__(128) colsum_kernel(const float* __restrict__ X, int M, int N, int ld, float* __restrict__ out) {
  const int n = blockIdx.x * 128 + threadIdx.x;
  if (n >= N) return;
  float s = 0.f;
  for (int64_t m0 = int64_t(blockIdx.y) * 64; m0 < M; m0 += int64_t(gridDim.y) * 64)
    for (int m = int(m0), m1 = int(min(int64_t(M), m0 + 64)); m < m1; ++m) s += __ldg(X + int64_t(m) * ld + n);
  atomicAdd(out + n, s);
}

int colsum(cudaStream_t st, const float* X, int M, int N, float* out) {
  const int chunks = (M + 63) / 64;
  colsum_kernel<<<dim3((N + 127) / 128, chunks < 65535 ? chunks : 65535), 128, 0, st>>>(X, M, N, N, out);
  BRK_LAUNCH_CHECK();
  return 0;
}

}  // namespace
int brk_twotower_step_fused(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u, const int32_t* i,
                            const int32_t* cand_ids, int64_t batch, int32_t training, const brk_twotower_workspace* ws,
                            float* loss_out, cudaStream_t st, int* handled, int do_opt, float lr, float eps,
                            const brk_twotower_shards* sh, const brk_tt_retrieval* rt,
                            const brk_tt_retrieval_sharded* srt, const brk_tt_sampled* smp);                      // twotower_fused.cu
int brk_gemm_tf32_impl(brk_ctx* ctx, const float* A, const float* B, float* C, const float* bias, int M, int N, int K, int lda,
                       int ldb, int ldc, int trans_a, int trans_b, float alpha, int accumulate, bool allow_split,
                       cudaStream_t st);
namespace {

// product dispatcher: tensor cores (TF32 operands) when asked for and the operands allow 16-byte loads, else fp32 SGEMM
int gemm(brk_ctx* ctx, cudaStream_t st, int tcore, const float* A, const float* B, float* C, const float* bias, int M, int N,
         int K, int lda, int ldb, int ldc, int ta, int tb, float alpha, int accumulate, bool allow_split) {
  if (tcore) {
    const int rc = brk_gemm_tf32_impl(ctx, A, B, C, bias, M, N, K, lda, ldb, ldc, ta, tb, alpha, accumulate, allow_split, st);
    if (rc != BRK_E_ALIGN) return rc;
  }
  return sgemm(ctx, st, A, B, C, bias, M, N, K, lda, ldb, ldc, ta, tb, alpha, accumulate, allow_split);
}

// One CTA per row of the [B,B] score matrix: accidental-hit masking, log-sum-exp, loss, and in place
// P = softmax - I (the gradient of the SUM-reduced cross-entropy w.r.t. the logits).
// RT (brk_twotower_step_retrieval): logits s * inv_tau - logq[j] (logq null: no correction), the row's loss and gradient
// weighted by w[row] (null: 1), P = w (softmax - I) * inv_tau.
constexpr float kMinFloatOver100 = -3.4028234663852886e36f;     // np.finfo(np.float32).min / 100
struct SoftmaxOptions { float inv_tau; const float* logq; const float* w; };
template <bool RT = false>
__global__ void __launch_bounds__(256)
inbatch_softmax_kernel(float* __restrict__ S, const int32_t* __restrict__ cand_ids, int B, int training,
                       double* __restrict__ loss_acc, SoftmaxOptions o = {}) {
  __shared__ float redf[32];
  __shared__ double redd[32];
  const int row = blockIdx.x, t = threadIdx.x;
  float* s = S + int64_t(row) * B;
  const int32_t pos_id = cand_ids ? __ldg(cand_ids + row) : -1;
  float mx = -CUDART_INF_F;
  for (int j = t; j < B; j += 256) {
    float v = s[j];
    if constexpr (RT) {
      v *= o.inv_tau;
      if (o.logq) v -= __ldg(o.logq + j);
      if (cand_ids && j != row && __ldg(cand_ids + j) == pos_id) v += kMinFloatOver100;
      s[j] = v;
    } else {
      if (cand_ids && j != row && __ldg(cand_ids + j) == pos_id) { v += kMinFloatOver100; s[j] = v; }
    }
    mx = fmaxf(mx, v);
  }
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((t & 31) == 0) redf[t >> 5] = mx;
  __syncthreads();
  mx = redf[0];
#pragma unroll
  for (int w = 1; w < 8; ++w) mx = fmaxf(mx, redf[w]);
  double sum = 0.0;
  for (int j = t; j < B; j += 256) sum += double(expf(s[j] - mx));
  sum = block_sum_double(sum, redd);
  __shared__ float lse_sm;
  if (t == 0) {
    const float lse = mx + logf(float(sum));
    lse_sm = lse;
    if constexpr (RT) atomicAdd(loss_acc, double(o.w ? __ldg(o.w + row) : 1.f) * double(lse - s[row]));
    else atomicAdd(loss_acc, double(lse - s[row]));       // -log softmax_row[row]
  }
  __syncthreads();
  if (!training) return;
  const float lse = lse_sm;
  if constexpr (RT) {
    const float wt = (o.w ? __ldg(o.w + row) : 1.f) * o.inv_tau;
    for (int j = t; j < B; j += 256) s[j] = (expf(s[j] - lse) - (j == row ? 1.f : 0.f)) * wt;
  } else {
    for (int j = t; j < B; j += 256) s[j] = expf(s[j] - lse) - (j == row ? 1.f : 0.f);
  }
}

// The log-probability term of every column for inbatch_softmax_kernel<true>: logq[j] = log(clip(p_j, 1e-6, 1)), p_j =
// cand_prob[j] or the streaming frequency estimate of item row ids[j].  With the estimator and training, first the
// update of Yi et al.'s Algorithm 2 at t = *step + 1: the thread whose exchange of last[y] returned another step is the
// sole updater of y, so duplicates update once; then *step = t.  One CTA: the update must be complete before any
// column reads gap, and a batch is a few thousand ids.
__global__ void __launch_bounds__(1024)
tt_logq_kernel(const int32_t* __restrict__ ids, int B, const float* __restrict__ cand_prob, long long* last, float* gap,
               long long* step, float alpha, int training, float* __restrict__ logq) {
  const int t = threadIdx.x;
  if (last && training) {
    const long long ts = *step + 1;
    for (int j = t; j < B; j += 1024) {
      const int32_t y = __ldg(ids + j);
      const long long prev = (long long)atomicExch(reinterpret_cast<unsigned long long*>(last + y), (unsigned long long)ts);
      if (prev != ts) gap[y] = __fadd_rn(__fmul_rn(__fsub_rn(1.f, alpha), gap[y]), __fmul_rn(alpha, __ll2float_rn(ts - prev)));
    }
    __syncthreads();
    if (t == 0) *step = ts;
  }
  for (int j = t; j < B; j += 1024) {
    float p = 1.f;
    if (cand_prob) p = __ldg(cand_prob + j);
    else { const float gp = gap[__ldg(ids + j)]; if (gp >= 1.f) p = __frcp_rn(gp); }
    logq[j] = logf(fminf(fmaxf(p, 1e-6f), 1.f));
  }
}

// Every rank's shard of the sharded estimator (brk_tt_estimator_sharded) as a kernel argument: row y at [y % world][y / world]
struct EstimatorShards {
  long long* last[BRK_MAX_PEERS];
  float* gap[BRK_MAX_PEERS];
  int world;
};

// The estimator's update on row-sharded state (brk_tt_estimator_update_sharded), one thread per id of this rank's slice.
// Every CTA reads t = *step + 1 first; the last CTA to take a ticket -- every other CTA has read the counter by then --
// writes t back and resets the ticket, so graph replays advance the counter too.  The exchange is system-scope: ranks on
// other GPUs exchange the same last[y] in the same step, and the one thread that sees another step is y's sole updater.
// gap is read past L1: its last writer may have been another GPU.
__global__ void __launch_bounds__(256)
tt_estimator_update_sharded_kernel(const int32_t* __restrict__ ids, int n, EstimatorShards e, float alpha, long long* step,
                                   unsigned int* ticket) {
  __shared__ long long ts_s;
  if (threadIdx.x == 0) ts_s = *reinterpret_cast<volatile long long*>(step) + 1;
  __syncthreads();
  const long long ts = ts_s;
  const int j = blockIdx.x * 256 + threadIdx.x;
  if (j < n) {
    const int32_t y = __ldg(ids + j);
    const int o = y % e.world;
    const int64_t l = y / e.world;
    const long long prev = (long long)atomicExch_system(reinterpret_cast<unsigned long long*>(e.last[o] + l), (unsigned long long)ts);
    if (prev != ts) {
      float* g = e.gap[o] + l;
      *g = __fadd_rn(__fmul_rn(__fsub_rn(1.f, alpha), __ldcg(g)), __fmul_rn(alpha, __ll2float_rn(ts - prev)));
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(ticket, 1u) == gridDim.x - 1) {
      *step = ts;
      *ticket = 0u;
      __threadfence();
    }
  }
}

// The column terms of inbatch_softmax_kernel<true> on row-sharded state (brk_twotower_step_sharded_retrieval): logq[j] =
// log(clip(p_j, 1e-6, 1)), p_j = cand_prob[j] or 1 / gap of item row ids[j] at its owner.  Reads only.
__global__ void __launch_bounds__(256)
tt_logq_sharded_kernel(const int32_t* __restrict__ ids, int B, const float* __restrict__ cand_prob, EstimatorShards e,
                       float* __restrict__ logq) {
  const int j = blockIdx.x * 256 + threadIdx.x;
  if (j >= B) return;
  float p = 1.f;
  if (cand_prob) p = __ldg(cand_prob + j);
  else {
    const int32_t y = __ldg(ids + j);
    const float gp = __ldcg(e.gap[y % e.world] + y / e.world);
    if (gp >= 1.f) p = __frcp_rn(gp);
  }
  logq[j] = logf(fminf(fmaxf(p, 1e-6f), 1.f));
}

// The draws of brk_tt_sampled at t = *step + 1: ids[k] = lo + mulshift(philox((k, t, t >> 32, tag), (seed, replica)).x,
// range).  One CTA: every thread has read the counter before thread 0 writes t back, so graph replays draw the next step.
__global__ void __launch_bounds__(1024)
tt_sample_negatives_kernel(int32_t* __restrict__ ids, int M, int32_t lo, uint32_t range, uint32_t seed, uint32_t replica,
                           long long* step) {
  __shared__ long long ts_s;
  if (threadIdx.x == 0) ts_s = *step + 1;
  __syncthreads();
  const unsigned long long ts = (unsigned long long)ts_s;
  for (int k = threadIdx.x; k < M; k += 1024) {
    const uint4 w = philox4x32_10(make_uint4(uint32_t(k), uint32_t(ts), uint32_t(ts >> 32), kBrkTagTwoTowerNeg), seed, replica);
    ids[k] = lo + int32_t(__umulhi(w.x, range));
  }
  if (threadIdx.x == 0) *step = (long long)ts;
}

// One CTA per query row of the [B, n] scores of the sampled-negatives step (n = B + M): columns j < B are the batch's
// candidates (item rows ids[j]), columns B + k the draws smp[k].  Logits s * inv_tau, a column j != row whose item row
// equals the row's positive masked, loss w_row (lse - s_row,row), in place P = w_row (softmax - Y) * inv_tau.
__global__ void __launch_bounds__(256)
sampled_softmax_kernel(float* __restrict__ Sc, const int32_t* __restrict__ ids, const int32_t* __restrict__ smp, int B, int n,
                       double* __restrict__ loss_acc, float inv_tau, const float* __restrict__ w) {
  __shared__ float redf[32];
  __shared__ double redd[32];
  __shared__ float lse_sm;
  const int row = blockIdx.x, t = threadIdx.x;
  float* s = Sc + int64_t(row) * n;
  const int32_t pos_id = __ldg(ids + row);
  float mx = -CUDART_INF_F;
  for (int j = t; j < n; j += 256) {
    float v = s[j] * inv_tau;
    const int32_t id = j < B ? __ldg(ids + j) : __ldg(smp + (j - B));
    if (j != row && id == pos_id) v += kMinFloatOver100;
    s[j] = v;
    mx = fmaxf(mx, v);
  }
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((t & 31) == 0) redf[t >> 5] = mx;
  __syncthreads();
  mx = redf[0];
#pragma unroll
  for (int k = 1; k < 8; ++k) mx = fmaxf(mx, redf[k]);
  double sum = 0.0;
  for (int j = t; j < n; j += 256) sum += double(expf(s[j] - mx));
  sum = block_sum_double(sum, redd);
  const float wr = w ? __ldg(w + row) : 1.f;
  if (t == 0) {
    const float lse = mx + logf(float(sum));
    lse_sm = lse;
    atomicAdd(loss_acc, double(wr) * double(lse - s[row]));
  }
  __syncthreads();
  const float lse = lse_sm, wt = wr * inv_tau;
  for (int j = t; j < n; j += 256) s[j] = (expf(s[j] - lse) - (j == row ? 1.f : 0.f)) * wt;
}

// rdZero mode: pred = sigmoid(<q_b, c_b>), mean BCE against labels; dq = g c, dc = g q, g = (p - y)/B.
__global__ void __launch_bounds__(256)
rowdot_bce_kernel(const float* __restrict__ q, const float* __restrict__ c, const float* __restrict__ y, int B, int S,
                  int training, float* __restrict__ dq, float* __restrict__ dc, double* __restrict__ loss_acc) {
  const int lane = threadIdx.x & 31;
  const int row = (blockIdx.x * 256 + threadIdx.x) >> 5;
  if (row >= B) return;
  float dot = 0.f;
  for (int k = lane; k < S; k += 32) dot = fmaf(q[int64_t(row) * S + k], c[int64_t(row) * S + k], dot);
  dot = warp_sum(dot);
  const float yv = y[row];
  const float p = 1.0f / (1.0f + expf(-dot));
  // Keras BCE on probabilities clips to [1e-7, 1 - 1e-7]; the from-logits form is used as Keras
  // back-tracks a sigmoid output to its logits
  const float l = fmaxf(dot, 0.f) - dot * yv + log1pf(expf(-fabsf(dot)));
  if (lane == 0) atomicAdd(loss_acc, double(l) / double(B));
  if (!training) return;
  const float g = (p - yv) / float(B);
  for (int k = lane; k < S; k += 32) {
    dq[int64_t(row) * S + k] = g * c[int64_t(row) * S + k];
    dc[int64_t(row) * S + k] = g * q[int64_t(row) * S + k];
  }
}

__global__ void finish_loss_kernel(double* acc, float* loss_out) {
  if (loss_out) loss_out[0] = float(acc[0]);
  acc[0] = 0.0;
}

}  // namespace

extern "C" int brk_sgemm(brk_ctx* ctx, const float* A, const float* B, float* C, const float* bias, int32_t M,
                         int32_t N, int32_t K, int32_t lda, int32_t ldb, int32_t ldc, int32_t trans_a, int32_t trans_b,
                         float alpha, int32_t accumulate, void* stream) {
  BRK_REQUIRE(ctx && A && B && C, BRK_E_ARG, "brk_sgemm: null argument");
  BRK_REQUIRE(M > 0 && N > 0 && K > 0, BRK_E_ARG, "brk_sgemm: M=%d N=%d K=%d", M, N, K);
  BRK_REQUIRE(lda >= (trans_a ? M : K) && ldb >= (trans_b ? K : N) && ldc >= N, BRK_E_ARG,
              "brk_sgemm: lda=%d ldb=%d ldc=%d below the stored row length (M=%d N=%d K=%d trans_a=%d trans_b=%d)", lda, ldb,
              ldc, M, N, K, trans_a, trans_b);
  return sgemm(ctx, (cudaStream_t)stream, A, B, C, bias, M, N, K, lda, ldb, ldc, trans_a, trans_b, alpha, accumulate,
               true);
}

// sh != nullptr: the rows come from the row-sharded table sh instead of t->emb.  extra [m]: rows gathered after ids[0..n)
// (the sampled negatives), the tower then runs over all n + m rows.
static int tower_forward(brk_ctx* ctx, const brk_tower* t, const int32_t* ids, int64_t n, float* emb_out, float* out,
                         int tcore, void* stream, const brk_shards* sh = nullptr, const int32_t* extra = nullptr,
                         int64_t m = 0) {
  int rc = sh ? brk_gather_rows_sharded(ctx, sh, t->E, ids, n, emb_out, stream)
              : brk_gather_rows(ctx, t->emb.w, t->emb.rows, t->E, ids, n, emb_out, stream);
  if (rc) return rc;
  if (m > 0) {
    float* dst = emb_out + n * t->E;
    rc = sh ? brk_gather_rows_sharded(ctx, sh, t->E, extra, m, dst, stream)
            : brk_gather_rows(ctx, t->emb.w, t->emb.rows, t->E, extra, m, dst, stream);
    if (rc) return rc;
  }
  const float* W = t->dense.w;                       // [E, S] Keras kernel, then bias [S]
  return gemm(ctx, (cudaStream_t)stream, tcore, emb_out, W, out, W + int64_t(t->E) * t->S, int(n + m), t->S, t->E, t->E,
              t->S, t->S, 0, 0, 1.f, 0, false);
}

extern "C" int brk_tower_forward(brk_ctx* ctx, const brk_tower* t, const int32_t* ids, int64_t n, float* emb_out,
                                 float* out, void* stream) {
  BRK_REQUIRE(ctx && t && ids && emb_out && out, BRK_E_ARG, "brk_tower_forward: null argument");
  BRK_REQUIRE(t->emb.w && t->dense.w && t->E > 0 && t->S > 0 && n > 0, BRK_E_ARG, "brk_tower_forward: bad tower");
  return tower_forward(ctx, t, ids, n, emb_out, out, 0, stream);
}

// The step after argument checks (brk_twotower_step, brk_twotower_step_sharded).  sh != nullptr: the embedding rows are
// gathered from and their gradients scattered into the row-sharded tables sh instead of user->emb / item->emb.
// rt != nullptr (unsharded, softmax mode only): the retrieval options, brk_twotower_step_retrieval; srt != nullptr
// (sharded, softmax mode only): brk_twotower_step_sharded_retrieval.
static int launch_sampler(const brk_tt_sampled* smp, cudaStream_t st) {
  tt_sample_negatives_kernel<<<1, 1024, 0, st>>>(smp->ids, int(smp->count), int32_t(smp->lo), uint32_t(smp->hi - smp->lo),
                                                 smp->seed, smp->replica, reinterpret_cast<long long*>(smp->step));
  BRK_LAUNCH_CHECK();
  return 0;
}

// smp != nullptr (softmax mode, training, no probabilities or estimator in rt / srt): sampled negatives -- the draws are
// made first, the item side of every buffer and product has n = B + M rows, the scores are [B, n].
// drawn: the caller has launched the sampler already (the train step, after its one-launch attempt).
static int twotower_step(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const brk_twotower_shards* sh,
                         const int32_t* u, const int32_t* i, const int32_t* cand_ids, const float* labels, int64_t batch,
                         int32_t mode, int32_t training, const brk_twotower_workspace* ws, float* loss_out, void* stream,
                         const brk_tt_retrieval* rt = nullptr, const brk_tt_retrieval_sharded* srt = nullptr,
                         const brk_tt_sampled* smp = nullptr, bool drawn = false) {
  // mode bit 8 (0x100): Dense / in-batch products on the tensor cores (TF32 operands, gemm_tc.cu)
  const int tcore = (mode & 0x100) ? 1 : 0;
  mode &= 0xFF;
  cudaStream_t st = (cudaStream_t)stream;
  const int B = int(batch), S = user->S, Eu = user->E, Ei = item->E;
  const int M = smp ? int(smp->count) : 0, n = B + M;
  const brk_shards* tsh[2] = {sh ? &sh->user : nullptr, sh ? &sh->item : nullptr};
  int rc;
  if (smp && !drawn && (rc = launch_sampler(smp, st))) return rc;
  if (mode == 0 && tcore) {                         // the whole step as one cooperative launch when the batch fits on chip
    int handled = 0;
    if ((rc = brk_twotower_step_fused(ctx, user, item, u, i, cand_ids, batch, training, ws, loss_out, st, &handled, 0, 0.f, 0.f,
                                      sh, rt, srt, smp))) return rc;
    if (handled) return 0;
  }
  // The user chain and the item chain are independent until the score product and again after the loss gradient, and
  // inside each chain the Dense gradients (dW, db) are independent of the embedding gradient (de -> scatter): the item
  // chain runs on fork stream 0, the Dense gradients on fork streams 1 / 2 (branches of the graph under stream
  // capture), the user chain on `st`.  At the reference's batch of 1000 (twoTower.py:292) every kernel is a few
  // microseconds, so the step is bound by the length of its dependency chain: 20 kernels in one line before, 8 now.
  // Outside a capture every fork/join costs four driver calls on the launching thread, which is what bounds the eager
  // step: there only the item chain is forked; the Dense-gradient side chains are used when the step is being captured.
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  BRK_CUDA(cudaStreamIsCapturing(st, &cap));
  const bool wide = cap == cudaStreamCaptureStatusActive;
  cudaStream_t fk = ctx->fork_stream[0];
  float* dz[2] = {ws->dq, ws->dc};
  // towers: q = Eu[u] Wu + bu, c = Ei[i] Wi + bi
  SoftmaxOptions so = {};
  if (rt || srt) {                                    // the column terms are ready before the score product is
    so.inv_tau = rt ? rt->inv_temperature : srt->inv_temperature; so.w = rt ? rt->row_weight : srt->row_weight;
    if (rt ? (rt->cand_prob || rt->last) : (srt->cand_prob || srt->est)) {
      if (ctx->tt_logq_floats < size_t(B)) {
        if (ctx->tt_logq) BRK_CUDA(cudaFree(ctx->tt_logq));
        ctx->tt_logq = nullptr; ctx->tt_logq_floats = 0;
        BRK_CUDA(cudaMalloc(&ctx->tt_logq, size_t(B) * sizeof(float)));
        ctx->tt_logq_floats = size_t(B);
      }
      if (rt) {
        tt_logq_kernel<<<1, 1024, 0, st>>>(i, B, rt->cand_prob, reinterpret_cast<long long*>(rt->last), rt->gap,
                                            reinterpret_cast<long long*>(rt->step), rt->alpha, training, ctx->tt_logq);
      } else {
        EstimatorShards e = {};
        e.world = 1;
        if (srt->est) {
          e.world = srt->est->world;
          for (int p = 0; p < e.world; ++p) e.gap[p] = srt->est->gap[p];
        }
        tt_logq_sharded_kernel<<<(B + 255) / 256, 256, 0, st>>>(i, B, srt->cand_prob, e, ctx->tt_logq);
      }
      BRK_LAUNCH_CHECK();
      so.logq = ctx->tt_logq;
    }
  }
  BRK_FORK(ctx, st, 0);
  if (training && mode == 0) BRK_CUDA(cudaMemsetAsync(dz[1], 0, size_t(n) * S * sizeof(float), fk));   // RED targets of
  if ((rc = tower_forward(ctx, item, i, batch, ws->ei, ws->c, tcore, fk, tsh[1], smp ? smp->ids : nullptr, M)))
    return rc;                                                                                           // the split-K
  if (training && mode == 0) BRK_CUDA(cudaMemsetAsync(dz[0], 0, size_t(B) * S * sizeof(float), st));   // products below
  if ((rc = tower_forward(ctx, user, u, batch, ws->eu, ws->q, tcore, stream, tsh[0]))) return rc;
  BRK_JOIN(ctx, st, 0);
  if (mode == 0) {
    // scores = q c^T [B, n]; softmax CE (SUM) with accidental-hit removal; in place P = softmax - I
    if ((rc = gemm(ctx, st, tcore, ws->q, ws->c, ws->scores, nullptr, B, n, S, S, S, n, 0, 1, 1.f, 0, false))) return rc;
    if (smp) {
      const float* w = rt ? rt->row_weight : (srt ? srt->row_weight : nullptr);
      const float inv_tau = rt ? rt->inv_temperature : (srt ? srt->inv_temperature : 1.f);
      sampled_softmax_kernel<<<B, 256, 0, st>>>(ws->scores, i, smp->ids, B, n, ws->acc, inv_tau, w);
    } else if (rt || srt) {
      inbatch_softmax_kernel<true><<<B, 256, 0, st>>>(ws->scores, cand_ids, B, training, ws->acc, so);
    } else {
      inbatch_softmax_kernel<<<B, 256, 0, st>>>(ws->scores, cand_ids, B, training, ws->acc);
    }
    BRK_LAUNCH_CHECK();
  } else {
    rowdot_bce_kernel<<<(B * 32 + 255) / 256, 256, 0, st>>>(ws->q, ws->c, labels, B, S, training, ws->dq, ws->dc, ws->acc);
    BRK_LAUNCH_CHECK();
  }
  if (!training) {
    finish_loss_kernel<<<1, 1, 0, st>>>(ws->acc, loss_out);
    BRK_LAUNCH_CHECK();
    return 0;
  }
  BRK_FORK(ctx, st, 0);
  // Per tower k (user on st, item on fork stream 0):
  //   softmax mode: dz = P c [B,S] (user) / P^T q [B,S] (item): few output tiles (B/64 x S/64) and a long K = B, so
  //   the products are split along K across CTAs and accumulated with REDs into the zeroed outputs;
  //   embedding-row gradients: de = dz W^T [B,E], scattered into the table accumulators;
  //   beside them (fork stream 1 + k): dW = e^T dz [E,S] (split-K over the batch), db = column sums of dz.
  const brk_tower* tw[2] = {user, item};
  const float* e[2] = {ws->eu, ws->ei};
  float* de[2] = {ws->deu, ws->dei};
  const float* other[2] = {ws->c, ws->q};
  const int32_t* ids[2] = {u, i};
  const int E[2] = {Eu, Ei};
  const int rows[2] = {B, n};                      // the item side has the sampled rows after the batch's
  for (int k = 0; k < 2; ++k) {
    cudaStream_t sk = k == 0 ? st : fk;
    cudaStream_t sd = wide ? ctx->fork_stream[1 + k] : sk;
    const int R = rows[k];
    if (mode == 0) {   // k = 0: dq = P c [B, S] (K = n); k = 1: dc = P^T q [n, S] (K = B); P is [B, n], ld n
      if ((rc = gemm(ctx, sk, tcore, ws->scores, other[k], dz[k], nullptr, R, S, rows[1 - k], n, S, S, k, 0, 1.f, 1, true)))
        return rc;
    }
    if (wide) BRK_FORK(ctx, sk, 1 + k);
    float* gW = tw[k]->dense.g;
    float* gb = gW + int64_t(E[k]) * S;
    if ((rc = gemm(ctx, sd, tcore, e[k], dz[k], gW, nullptr, E[k], S, R, E[k], S, S, 1, 0, 1.f, 1, true))) return rc;
    if ((rc = colsum(sd, dz[k], R, S, gb))) return rc;
    if (k == 0) {                                  // the loss scalar rides on the user tower's side stream
      finish_loss_kernel<<<1, 1, 0, sd>>>(ws->acc, loss_out);
      BRK_LAUNCH_CHECK();
    }
    // de = dz W^T: W stored [E,S] = "B stored [N,K]" with N = E, K = S  (tb = 1); its own buffer: the dW product
    // beside it is still reading the gathered rows e
    if ((rc = gemm(ctx, sk, tcore, dz[k], tw[k]->dense.w, de[k], nullptr, R, E[k], S, S, S, E[k], 0, 1, 1.f, 0, false))) return rc;
    for (int part = 0; part < (k == 1 && smp ? 2 : 1); ++part) {   // the batch's rows, then the sampled rows
      const int32_t* pid = part ? smp->ids : ids[k];
      const int64_t cnt = part ? M : batch;
      const float* val = de[k] + (part ? int64_t(B) * E[k] : 0);
      rc = tsh[k] ? brk_scatter_add_rows_sharded(ctx, tsh[k], E[k], pid, cnt, val, (void*)sk)
                  : brk_scatter_add_rows(ctx, tw[k]->emb.g, tw[k]->emb.rows, E[k], pid, cnt, val, tw[k]->emb.touched, 0,
                                         (void*)sk);
      if (rc) return rc;
    }
    if (wide) BRK_JOIN(ctx, sk, 1 + k);
  }
  BRK_JOIN(ctx, st, 0);
  return 0;
}

static int check_retrieval(const brk_tower* item, int32_t mode, const brk_tt_retrieval* rt, const char* fn) {
  BRK_REQUIRE(std::isfinite(rt->inv_temperature) && rt->inv_temperature > 0.f, BRK_E_ARG,
              "%s: 1 / temperature = %g is not finite and > 0", fn, double(rt->inv_temperature));
  BRK_REQUIRE((mode & 0xFF) == 0, BRK_E_ARG, "%s: the retrieval options need the in-batch softmax (rdZero mode has no "
              "in-batch negatives)", fn);
  if (rt->last) {
    BRK_REQUIRE(!rt->cand_prob, BRK_E_ARG, "%s: candidate probabilities and the streaming estimator are exclusive", fn);
    BRK_REQUIRE(rt->gap && rt->step, BRK_E_ARG, "%s: the streaming estimator needs gap and a step counter", fn);
    BRK_REQUIRE(rt->rows >= item->emb.rows, BRK_E_ARG, "%s: estimator arrays of %lld rows, the item table has %lld", fn,
                (long long)rt->rows, (long long)item->emb.rows);
    BRK_REQUIRE(rt->alpha > 0.f && rt->alpha <= 1.f, BRK_E_ARG, "%s: estimator alpha = %g outside (0, 1]", fn, double(rt->alpha));
  }
  return 0;
}

// The checks that every sampled-negatives entry point shares (brk_tt_sampled).  item_rows < 0: the sharded step, which
// only has smp->rows.  cand_prob / has_est: what rt carries beside temperature and weights.
static int check_sampled(const brk_tt_sampled* smp, int32_t mode, int64_t batch, int64_t item_rows, const float* cand_prob,
                         bool has_est, float inv_temperature, const char* fn) {
  BRK_REQUIRE(smp, BRK_E_ARG, "%s: null sampled-negatives argument", fn);
  BRK_REQUIRE(smp->count >= 1 && smp->count < (1 << 30), BRK_E_ARG, "%s: sampled count M = %lld (at least 1)", fn,
              (long long)smp->count);
  BRK_REQUIRE(smp->ids && smp->step, BRK_E_ARG, "%s: sampled negatives need an ids buffer [M] and a step counter", fn);
  BRK_REQUIRE(item_rows < 0 || smp->rows == item_rows, BRK_E_ARG, "%s: sampled rows = %lld, the item table has %lld", fn,
              (long long)smp->rows, (long long)item_rows);
  BRK_REQUIRE(smp->lo >= 0 && smp->lo < smp->hi && smp->hi <= smp->rows && smp->rows < (int64_t(1) << 31), BRK_E_ARG,
              "%s: sampled range [%lld, %lld) is empty or outside the item table's %lld rows", fn, (long long)smp->lo,
              (long long)smp->hi, (long long)smp->rows);
  BRK_REQUIRE((mode & 0xFF) == 0, BRK_E_ARG, "%s: sampled negatives need the in-batch softmax (rdZero mode has no "
              "candidates)", fn);
  BRK_REQUIRE(!cand_prob && !has_est, BRK_E_ARG, "%s: candidate probabilities and the streaming estimator are not offered "
              "with sampled negatives (the logQ correction of a mixed pool needs both routes' probabilities)", fn);
  BRK_REQUIRE(std::isfinite(inv_temperature) && inv_temperature > 0.f, BRK_E_ARG,
              "%s: 1 / temperature = %g is not finite and > 0", fn, double(inv_temperature));
  BRK_REQUIRE(batch >= 0 && batch < (1 << 30) && batch * (batch + smp->count) < (int64_t(1) << 31), BRK_E_ARG,
              "%s: score matrix [%lld, %lld] has 2^31 or more entries", fn, (long long)batch,
              (long long)(batch + smp->count));
  return 0;
}

// batch == 0 with sampled negatives: the draws still advance the counter, the loss is 0
static int sampled_empty_step(const brk_tt_sampled* smp, float* loss_out, cudaStream_t st) {
  int rc;
  if ((rc = launch_sampler(smp, st))) return rc;
  if (loss_out) BRK_CUDA(cudaMemsetAsync(loss_out, 0, sizeof(float), st));
  return 0;
}

static int twotower_step_checked(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u,
                                 const int32_t* i, const int32_t* cand_ids, const float* labels, int64_t batch,
                                 int32_t mode, int32_t training, const brk_twotower_workspace* ws, float* loss_out,
                                 void* stream, const brk_tt_retrieval* rt, const brk_tt_sampled* smp = nullptr,
                                 bool drawn = false) {
  if (smp) {
    static const char* fn = "brk_twotower_step_sampled";
    BRK_REQUIRE(ctx && user && item && ws, BRK_E_ARG, "%s: null argument", fn);
    int rc;
    if ((rc = check_sampled(smp, mode, batch, item->emb.rows, rt ? rt->cand_prob : nullptr, rt && rt->last,
                            rt ? rt->inv_temperature : 1.f, fn))) return rc;
    if (batch == 0) return sampled_empty_step(smp, loss_out, (cudaStream_t)stream);
  }
  BRK_REQUIRE(ctx && user && item && u && i && ws, BRK_E_ARG, "brk_twotower_step: null argument");
  BRK_REQUIRE(user->S == item->S && batch > 0 && batch < (1 << 30), BRK_E_ARG, "brk_twotower_step: S %d vs %d, batch %lld",
              user->S, item->S, (long long)batch);
  BRK_REQUIRE((mode & 0xFF) == 0 || labels, BRK_E_ARG, "brk_twotower_step: rdZero mode needs labels");
  BRK_REQUIRE(ws->eu && ws->ei && ws->q && ws->c && ws->dq && ws->dc && ws->acc && ((mode & 0xFF) != 0 || ws->scores), BRK_E_ARG,
              "brk_twotower_step: workspace missing");
  BRK_REQUIRE(!training || (user->emb.g && item->emb.g && user->dense.g && item->dense.g && ws->deu && ws->dei), BRK_E_ARG,
              "brk_twotower_step: gradient accumulators / deu, dei workspace missing");
  if (rt) {
    int rc;
    if ((rc = check_retrieval(item, mode, rt, "brk_twotower_step_retrieval"))) return rc;
  }
  return twotower_step(ctx, user, item, nullptr, u, i, cand_ids, labels, batch, mode, training, ws, loss_out, stream, rt,
                       nullptr, smp, drawn);
}

extern "C" int brk_twotower_step_sampled(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u,
                                         const int32_t* i, int64_t batch, int32_t mode, const brk_twotower_workspace* ws,
                                         float* loss_out, void* stream, const brk_tt_sampled* smp, const brk_tt_retrieval* rt) {
  BRK_REQUIRE(smp, BRK_E_ARG, "brk_twotower_step_sampled: null sampled-negatives argument");
  return twotower_step_checked(ctx, user, item, u, i, i, nullptr, batch, mode, 1, ws, loss_out, stream, rt, smp);
}

extern "C" int brk_twotower_step(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u,
                                 const int32_t* i, const int32_t* cand_ids, const float* labels, int64_t batch,
                                 int32_t mode, int32_t training, const brk_twotower_workspace* ws, float* loss_out,
                                 void* stream) {
  return twotower_step_checked(ctx, user, item, u, i, cand_ids, labels, batch, mode, training, ws, loss_out, stream, nullptr);
}

extern "C" int brk_twotower_step_retrieval(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u,
                                           const int32_t* i, const int32_t* cand_ids, const float* labels, int64_t batch,
                                           int32_t mode, int32_t training, const brk_twotower_workspace* ws, float* loss_out,
                                           void* stream, const brk_tt_retrieval* rt) {
  return twotower_step_checked(ctx, user, item, u, i, cand_ids, labels, batch, mode, training, ws, loss_out, stream, rt);
}

static int check_shards(const brk_shards* s, int32_t E, const char* which, const char* fn = "brk_twotower_step_sharded") {
  BRK_REQUIRE(s->world >= 1 && s->world <= BRK_MAX_PEERS, BRK_E_ARG, "%s: %s world=%d (1..%d)", fn, which, s->world,
              BRK_MAX_PEERS);
  BRK_REQUIRE(s->rank >= 0 && s->rank < s->world, BRK_E_ARG, "%s: %s rank=%d world=%d", fn, which, s->rank, s->world);
  for (int p = 0; p < s->world; ++p)
    BRK_REQUIRE(s->w[p] && s->g[p] && s->touched[p], BRK_E_ARG, "%s: %s shard %d has a null w / g / touched", fn, which, p);
  BRK_REQUIRE(E > 0 && (E & 3) == 0, BRK_E_ARG, "%s: %s width %d is not a positive multiple of 4", fn, which, E);
  return 0;
}

static int check_estimator(const brk_tt_estimator_sharded* e, const char* fn) {
  BRK_REQUIRE(e->world >= 1 && e->world <= BRK_MAX_PEERS, BRK_E_ARG, "%s: estimator world=%d (1..%d)", fn, e->world,
              BRK_MAX_PEERS);
  BRK_REQUIRE(e->rank >= 0 && e->rank < e->world, BRK_E_ARG, "%s: estimator rank=%d world=%d", fn, e->rank, e->world);
  BRK_REQUIRE(e->rows >= 1, BRK_E_ARG, "%s: estimator shards of %lld rows", fn, (long long)e->rows);
  return 0;
}

static int twotower_step_sharded_checked(brk_ctx* ctx, const brk_tower* user, const brk_tower* item,
                                         const brk_twotower_shards* sh, const int32_t* u, const int32_t* i,
                                         const int32_t* cand_ids, const float* labels, int64_t batch, int32_t mode,
                                         const brk_twotower_workspace* ws, float* loss_out, void* stream,
                                         const brk_tt_retrieval_sharded* srt) {
  BRK_REQUIRE(ctx && user && item && ws, BRK_E_ARG, "brk_twotower_step_sharded: null argument");
  BRK_REQUIRE(sh, BRK_E_ARG, "brk_twotower_step_sharded: null shards");
  int rc;
  if ((rc = check_shards(&sh->user, user->E, "user"))) return rc;
  if ((rc = check_shards(&sh->item, item->E, "item"))) return rc;
  BRK_REQUIRE(sh->user.world == sh->item.world && sh->user.rank == sh->item.rank, BRK_E_ARG,
              "brk_twotower_step_sharded: user / item shards of different worlds or ranks");
  BRK_REQUIRE(user->S == item->S && batch >= 0 && batch < (1 << 30), BRK_E_ARG,
              "brk_twotower_step_sharded: S %d vs %d, batch %lld", user->S, item->S, (long long)batch);
  if (batch == 0) return 0;
  BRK_REQUIRE(u && i, BRK_E_ARG, "brk_twotower_step_sharded: null ids");
  BRK_REQUIRE((mode & 0xFF) == 0 || labels, BRK_E_ARG, "brk_twotower_step_sharded: rdZero mode needs labels");
  BRK_REQUIRE(ws->eu && ws->ei && ws->q && ws->c && ws->dq && ws->dc && ws->acc && ws->deu && ws->dei &&
              ((mode & 0xFF) != 0 || ws->scores), BRK_E_ARG, "brk_twotower_step_sharded: workspace missing");
  BRK_REQUIRE(user->dense.w && item->dense.w && user->dense.g && item->dense.g, BRK_E_ARG,
              "brk_twotower_step_sharded: Dense blocks or their gradients missing");
  return twotower_step(ctx, user, item, sh, u, i, cand_ids, labels, batch, mode, 1, ws, loss_out, stream, nullptr, srt);
}

extern "C" int brk_twotower_step_sharded(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const brk_twotower_shards* sh,
                                         const int32_t* u, const int32_t* i, const int32_t* cand_ids, const float* labels,
                                         int64_t batch, int32_t mode, const brk_twotower_workspace* ws, float* loss_out,
                                         void* stream) {
  return twotower_step_sharded_checked(ctx, user, item, sh, u, i, cand_ids, labels, batch, mode, ws, loss_out, stream, nullptr);
}

extern "C" int brk_twotower_step_sharded_retrieval(brk_ctx* ctx, const brk_tower* user, const brk_tower* item,
                                                   const brk_twotower_shards* sh, const int32_t* u, const int32_t* i,
                                                   const int32_t* cand_ids, const float* labels, int64_t batch, int32_t mode,
                                                   const brk_twotower_workspace* ws, float* loss_out, void* stream,
                                                   const brk_tt_retrieval_sharded* rt) {
  static const char* fn = "brk_twotower_step_sharded_retrieval";
  if (rt) {
    BRK_REQUIRE(std::isfinite(rt->inv_temperature) && rt->inv_temperature > 0.f, BRK_E_ARG,
                "%s: 1 / temperature = %g is not finite and > 0", fn, double(rt->inv_temperature));
    BRK_REQUIRE((mode & 0xFF) == 0, BRK_E_ARG, "%s: the retrieval options need the in-batch softmax (rdZero mode has no "
                "in-batch negatives)", fn);
    if (const brk_tt_estimator_sharded* e = rt->est) {
      BRK_REQUIRE(!rt->cand_prob, BRK_E_ARG, "%s: candidate probabilities and the streaming estimator are exclusive", fn);
      int rc;
      if ((rc = check_estimator(e, fn))) return rc;
      BRK_REQUIRE(sh && e->world == sh->item.world && e->rank == sh->item.rank, BRK_E_ARG,
                  "%s: estimator of world %d rank %d, item shards of another world or rank", fn, e->world, e->rank);
      for (int p = 0; p < e->world; ++p)
        BRK_REQUIRE(e->gap[p], BRK_E_ARG, "%s: estimator shard %d has a null gap", fn, p);
    }
  }
  return twotower_step_sharded_checked(ctx, user, item, sh, u, i, cand_ids, labels, batch, mode, ws, loss_out, stream, rt);
}

extern "C" int brk_twotower_step_sharded_sampled(brk_ctx* ctx, const brk_tower* user, const brk_tower* item,
                                                 const brk_twotower_shards* sh, const int32_t* u, const int32_t* i,
                                                 int64_t batch, int32_t mode, const brk_twotower_workspace* ws, float* loss_out,
                                                 void* stream, const brk_tt_sampled* smp, const brk_tt_retrieval_sharded* rt) {
  static const char* fn = "brk_twotower_step_sharded_sampled";
  int rc;
  if ((rc = check_sampled(smp, mode, batch, -1, rt ? rt->cand_prob : nullptr, rt && rt->est, rt ? rt->inv_temperature : 1.f,
                          fn))) return rc;
  BRK_REQUIRE(ctx && user && item && ws && sh, BRK_E_ARG, "%s: null argument", fn);
  if ((rc = check_shards(&sh->user, user->E, "user", fn))) return rc;
  if ((rc = check_shards(&sh->item, item->E, "item", fn))) return rc;
  if (batch == 0) return sampled_empty_step(smp, loss_out, (cudaStream_t)stream);
  BRK_REQUIRE(u && i, BRK_E_ARG, "%s: null ids", fn);
  BRK_REQUIRE(sh->user.world == sh->item.world && sh->user.rank == sh->item.rank, BRK_E_ARG,
              "%s: user / item shards of different worlds or ranks", fn);
  BRK_REQUIRE(user->S == item->S, BRK_E_ARG, "%s: S %d vs %d", fn, user->S, item->S);
  BRK_REQUIRE(ws->eu && ws->ei && ws->q && ws->c && ws->dq && ws->dc && ws->acc && ws->deu && ws->dei && ws->scores, BRK_E_ARG,
              "%s: workspace missing", fn);
  BRK_REQUIRE(user->dense.w && item->dense.w && user->dense.g && item->dense.g, BRK_E_ARG,
              "%s: Dense blocks or their gradients missing", fn);
  return twotower_step(ctx, user, item, sh, u, i, i, nullptr, batch, mode, 1, ws, loss_out, stream, nullptr, rt, smp);
}

extern "C" int brk_tt_estimator_update_sharded(brk_ctx* ctx, const brk_tt_estimator_sharded* est, const int32_t* ids,
                                               int64_t n, float alpha, int64_t* step, void* stream) {
  static const char* fn = "brk_tt_estimator_update_sharded";
  BRK_REQUIRE(ctx && est && step, BRK_E_ARG, "%s: null argument", fn);
  BRK_REQUIRE(n >= 0 && n < (1 << 30) && (n == 0 || ids), BRK_E_ARG, "%s: n = %lld, ids %p", fn, (long long)n, (const void*)ids);
  BRK_REQUIRE(alpha > 0.f && alpha <= 1.f, BRK_E_ARG, "%s: estimator alpha = %g outside (0, 1]", fn, double(alpha));
  int rc;
  if ((rc = check_estimator(est, fn))) return rc;
  EstimatorShards e = {};
  e.world = est->world;
  for (int p = 0; p < e.world; ++p) {
    BRK_REQUIRE(est->last[p] && est->gap[p], BRK_E_ARG, "%s: estimator shard %d has a null last / gap", fn, p);
    e.last[p] = reinterpret_cast<long long*>(est->last[p]); e.gap[p] = est->gap[p];
  }
  const int grid = n > 0 ? int((n + 255) / 256) : 1;          // an empty slice still advances the counter
  tt_estimator_update_sharded_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(ids, int(n), e, alpha,
                                                                              reinterpret_cast<long long*>(step), ctx->tickets + 7);
  BRK_LAUNCH_CHECK();
  return 0;
}

extern "C" int brk_tower_forward_sharded(brk_ctx* ctx, const brk_tower* t, const brk_shards* sh, const int32_t* ids, int64_t n,
                                         float* emb_out, float* out, void* stream) {
  BRK_REQUIRE(ctx && t && sh && ids && emb_out && out, BRK_E_ARG, "brk_tower_forward_sharded: null argument");
  BRK_REQUIRE(t->dense.w && t->E > 0 && t->S > 0 && n > 0, BRK_E_ARG, "brk_tower_forward_sharded: bad tower");
  return tower_forward(ctx, t, ids, n, emb_out, out, 0, stream, sh);
}

// Pieces of the step that the global-negatives phases (twotower_global.cu) run in their own order.
int brk_tt_gemm(brk_ctx* ctx, cudaStream_t st, int tcore, const float* A, const float* B, float* C, int M, int N, int K, int lda,
                int ldb, int ldc, int ta, int tb, int accumulate, bool allow_split) {
  return gemm(ctx, st, tcore, A, B, C, nullptr, M, N, K, lda, ldb, ldc, ta, tb, 1.f, accumulate, allow_split);
}
int brk_tt_tower_forward(brk_ctx* ctx, const brk_tower* t, const int32_t* ids, int64_t n, float* emb_out, float* out, int tcore,
                         cudaStream_t st, const brk_shards* sh) {
  return tower_forward(ctx, t, ids, n, emb_out, out, tcore, st, sh);
}
int brk_tt_colsum(cudaStream_t st, const float* X, int M, int N, float* out) { return colsum(st, X, M, N, out); }
int brk_tt_check_shards(const brk_shards* s, int32_t E, const char* which, const char* fn) {
  return check_shards(s, E, which, fn);
}

// Training step + Keras Adagrad (twoTower.py:89-102 with the optimizer of :278-279) in one call.  In-batch-softmax steps
// on the tensor cores whose batch fits on chip run as ONE launch (twotower_fused.cu: the optimizer is the last phase of the
// same cooperative kernel and only visits the rows the batch touched); everything else is brk_twotower_step followed by
// the dense or row-sparse Adagrad pass of optim.cu (row-sparse for tables above rows_threshold_bytes that carry a bitmask).
static int twotower_train_step(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u,
                               const int32_t* i, const int32_t* cand_ids, const float* labels, int64_t batch,
                               int32_t mode, const brk_twotower_workspace* ws, float lr, float eps,
                               int64_t rows_threshold_bytes, float* loss_out, void* stream, const brk_tt_retrieval* rt,
                               const brk_tt_sampled* smp = nullptr) {
  int rc;
  if (smp) {          // the draws, then the one launch with Adagrad when it fits, else the multi-kernel step
    static const char* fn = "brk_twotower_train_step_sampled";
    BRK_REQUIRE(ctx && user && item && ws, BRK_E_ARG, "%s: null argument", fn);
    if ((rc = check_sampled(smp, mode, batch, item->emb.rows, rt ? rt->cand_prob : nullptr, rt && rt->last,
                            rt ? rt->inv_temperature : 1.f, fn))) return rc;
    if (batch == 0) return sampled_empty_step(smp, loss_out, (cudaStream_t)stream);
    BRK_REQUIRE(u && i, BRK_E_ARG, "%s: null ids", fn);
    if ((rc = launch_sampler(smp, (cudaStream_t)stream))) return rc;
    if ((mode & 0x100) && user->S == item->S && ws->q && ws->c && ws->dq && ws->dc && ws->acc && user->emb.g && item->emb.g &&
        user->dense.g && item->dense.g) {
      int handled = 0;
      if ((rc = brk_twotower_step_fused(ctx, user, item, u, i, i, batch, 1, ws, loss_out, (cudaStream_t)stream, &handled, 1, lr,
                                        eps, nullptr, rt, nullptr, smp)))
        return rc;
      if (handled) return 0;
    }
    if ((rc = twotower_step_checked(ctx, user, item, u, i, i, labels, batch, mode, 1, ws, loss_out, stream, rt, smp, true)))
      return rc;
  } else {
    BRK_REQUIRE(ctx && user && item && u && i && ws, BRK_E_ARG, "brk_twotower_train_step: null argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (rt && (rc = check_retrieval(item, mode, rt, "brk_twotower_train_step_retrieval"))) return rc;
    if ((mode & 0xFF) == 0 && (mode & 0x100) && user->S == item->S && batch > 0 && batch < (1 << 30) && ws->q && ws->c &&
        ws->dq && ws->dc && ws->acc && user->emb.g && item->emb.g && user->dense.g && item->dense.g) {
      int handled = 0;
      if ((rc = brk_twotower_step_fused(ctx, user, item, u, i, cand_ids, batch, 1, ws, loss_out, st, &handled, 1, lr, eps,
                                        nullptr, rt, nullptr, nullptr)))
        return rc;
      if (handled) return 0;
    }
    if ((rc = twotower_step_checked(ctx, user, item, u, i, cand_ids, labels, batch, mode, 1, ws, loss_out, stream, rt)))
      return rc;
  }
  brk_table dense_pass[4], rows_pass[2];
  int nd = 0, nr = 0;
  const brk_tower* tw[2] = {user, item};
  for (int k = 0; k < 2; ++k) {
    const brk_table& e = tw[k]->emb;
    if (e.touched && int64_t(e.rows) * e.d * 4 > rows_threshold_bytes) rows_pass[nr++] = e;
    else dense_pass[nd++] = e;
  }
  dense_pass[nd++] = user->dense; dense_pass[nd++] = item->dense;
  if ((rc = brk_adagrad_dense(ctx, dense_pass, nd, lr, eps, stream))) return rc;
  if (nr && (rc = brk_adagrad_rows(ctx, rows_pass, nr, lr, eps, stream))) return rc;
  return 0;
}

extern "C" int brk_twotower_train_step(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u,
                                       const int32_t* i, const int32_t* cand_ids, const float* labels, int64_t batch,
                                       int32_t mode, const brk_twotower_workspace* ws, float lr, float eps,
                                       int64_t rows_threshold_bytes, float* loss_out, void* stream) {
  return twotower_train_step(ctx, user, item, u, i, cand_ids, labels, batch, mode, ws, lr, eps, rows_threshold_bytes, loss_out,
                             stream, nullptr);
}

extern "C" int brk_twotower_train_step_retrieval(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u,
                                                 const int32_t* i, const int32_t* cand_ids, const float* labels, int64_t batch,
                                                 int32_t mode, const brk_twotower_workspace* ws, float lr, float eps,
                                                 int64_t rows_threshold_bytes, float* loss_out, void* stream,
                                                 const brk_tt_retrieval* rt) {
  return twotower_train_step(ctx, user, item, u, i, cand_ids, labels, batch, mode, ws, lr, eps, rows_threshold_bytes, loss_out,
                             stream, rt);
}

extern "C" int brk_twotower_train_step_sampled(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u,
                                               const int32_t* i, int64_t batch, int32_t mode, const brk_twotower_workspace* ws,
                                               float lr, float eps, int64_t rows_threshold_bytes, float* loss_out, void* stream,
                                               const brk_tt_sampled* smp, const brk_tt_retrieval* rt) {
  BRK_REQUIRE(smp, BRK_E_ARG, "brk_twotower_train_step_sampled: null sampled-negatives argument");
  return twotower_train_step(ctx, user, item, u, i, i, nullptr, batch, mode, ws, lr, eps, rows_threshold_bytes, loss_out,
                             stream, rt, smp);
}
