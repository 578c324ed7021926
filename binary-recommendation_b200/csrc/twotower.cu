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

namespace {

constexpr int TM = 64, TN = 64, TK = 16, kGemmThreads = 256;

// C[M,N] (op)= alpha * opA(A) * opB(B) (+ bias[N])
//   ta == 0: A is [M,K] row-major (lda = K-stride);  ta == 1: A is stored [K,M] (A^T used)
//   tb == 0: B is [K,N] row-major;                    tb == 1: B is stored [N,K]
//   accumulate != 0: C += (RED.ADD when split-K > 1, plain += otherwise); bias added by split 0 only
__global__ void __launch_bounds__(kGemmThreads)
sgemm_kernel(const float* __restrict__ A, const float* __restrict__ Bm, float* __restrict__ C,
             const float* __restrict__ bias, int M, int N, int K, int lda, int ldb, int ldc, int ta, int tb,
             float alpha, int accumulate, int k_per_split) {
  __shared__ __align__(16) float As[TK][TM + 4];
  __shared__ __align__(16) float Bs[TK][TN + 4];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;       // 16 x 16 threads, 4x4 outputs each
  const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
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
  sgemm_kernel<<<dim3(gx, gy, splits), kGemmThreads, 0, st>>>(A, B, C, bias, M, N, K, lda, ldb, ldc, ta, tb, alpha,
                                                              accumulate, kps);
  BRK_LAUNCH_CHECK();
  return 0;
}

// out[n] += sum_m X[m][n]: bias gradients (ones^T dz) without a degenerate M = 1 product
__global__ void __launch_bounds__(128) colsum_kernel(const float* __restrict__ X, int M, int N, int ld, float* __restrict__ out) {
  const int n = blockIdx.x * 128 + threadIdx.x;
  const int m0 = blockIdx.y * 64, m1 = min(M, m0 + 64);
  if (n >= N) return;
  float s = 0.f;
  for (int m = m0; m < m1; ++m) s += __ldg(X + int64_t(m) * ld + n);
  atomicAdd(out + n, s);
}

}  // namespace
int brk_twotower_step_fused(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u, const int32_t* i,
                            const int32_t* cand_ids, int64_t batch, int32_t training, const brk_twotower_workspace* ws,
                            float* loss_out, cudaStream_t st, int* handled, int do_opt, float lr, float eps,
                            const brk_twotower_shards* sh);                                                       // twotower_fused.cu
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
constexpr float kMinFloatOver100 = -3.4028234663852886e36f;     // np.finfo(np.float32).min / 100
__global__ void __launch_bounds__(256)
inbatch_softmax_kernel(float* __restrict__ S, const int32_t* __restrict__ cand_ids, int B, int training,
                       double* __restrict__ loss_acc) {
  __shared__ float redf[32];
  __shared__ double redd[32];
  const int row = blockIdx.x, t = threadIdx.x;
  float* s = S + int64_t(row) * B;
  const int32_t pos_id = cand_ids ? __ldg(cand_ids + row) : -1;
  float mx = -CUDART_INF_F;
  for (int j = t; j < B; j += 256) {
    float v = s[j];
    if (cand_ids && j != row && __ldg(cand_ids + j) == pos_id) { v += kMinFloatOver100; s[j] = v; }
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
    atomicAdd(loss_acc, double(lse - s[row]));            // -log softmax_row[row]
  }
  __syncthreads();
  if (!training) return;
  const float lse = lse_sm;
  for (int j = t; j < B; j += 256) s[j] = expf(s[j] - lse) - (j == row ? 1.f : 0.f);
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
  return sgemm(ctx, (cudaStream_t)stream, A, B, C, bias, M, N, K, lda, ldb, ldc, trans_a, trans_b, alpha, accumulate,
               true);
}

// sh != nullptr: the rows come from the row-sharded table sh instead of t->emb
static int tower_forward(brk_ctx* ctx, const brk_tower* t, const int32_t* ids, int64_t n, float* emb_out, float* out,
                         int tcore, void* stream, const brk_shards* sh = nullptr) {
  int rc = sh ? brk_gather_rows_sharded(ctx, sh, t->E, ids, n, emb_out, stream)
              : brk_gather_rows(ctx, t->emb.w, t->emb.rows, t->E, ids, n, emb_out, stream);
  if (rc) return rc;
  const float* W = t->dense.w;                       // [E, S] Keras kernel, then bias [S]
  return gemm(ctx, (cudaStream_t)stream, tcore, emb_out, W, out, W + int64_t(t->E) * t->S, int(n), t->S, t->E, t->E, t->S,
              t->S, 0, 0, 1.f, 0, false);
}

extern "C" int brk_tower_forward(brk_ctx* ctx, const brk_tower* t, const int32_t* ids, int64_t n, float* emb_out,
                                 float* out, void* stream) {
  BRK_REQUIRE(ctx && t && ids && emb_out && out, BRK_E_ARG, "brk_tower_forward: null argument");
  BRK_REQUIRE(t->emb.w && t->dense.w && t->E > 0 && t->S > 0 && n > 0, BRK_E_ARG, "brk_tower_forward: bad tower");
  return tower_forward(ctx, t, ids, n, emb_out, out, 0, stream);
}

// The step after argument checks (brk_twotower_step, brk_twotower_step_sharded).  sh != nullptr: the embedding rows are
// gathered from and their gradients scattered into the row-sharded tables sh instead of user->emb / item->emb.
static int twotower_step(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const brk_twotower_shards* sh,
                         const int32_t* u, const int32_t* i, const int32_t* cand_ids, const float* labels, int64_t batch,
                         int32_t mode, int32_t training, const brk_twotower_workspace* ws, float* loss_out, void* stream) {
  // mode bit 8 (0x100): Dense / in-batch products on the tensor cores (TF32 operands, gemm_tc.cu)
  const int tcore = (mode & 0x100) ? 1 : 0;
  mode &= 0xFF;
  cudaStream_t st = (cudaStream_t)stream;
  const int B = int(batch), S = user->S, Eu = user->E, Ei = item->E;
  const brk_shards* tsh[2] = {sh ? &sh->user : nullptr, sh ? &sh->item : nullptr};
  int rc;
  if (mode == 0 && tcore) {                         // the whole step as one cooperative launch when the batch fits on chip
    int handled = 0;
    if ((rc = brk_twotower_step_fused(ctx, user, item, u, i, cand_ids, batch, training, ws, loss_out, st, &handled, 0, 0.f, 0.f,
                                      sh))) return rc;
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
  BRK_FORK(ctx, st, 0);
  if (training && mode == 0) BRK_CUDA(cudaMemsetAsync(dz[1], 0, size_t(B) * S * sizeof(float), fk));   // RED targets of
  if ((rc = tower_forward(ctx, item, i, batch, ws->ei, ws->c, tcore, fk, tsh[1]))) return rc;            // the split-K
  if (training && mode == 0) BRK_CUDA(cudaMemsetAsync(dz[0], 0, size_t(B) * S * sizeof(float), st));   // products below
  if ((rc = tower_forward(ctx, user, u, batch, ws->eu, ws->q, tcore, stream, tsh[0]))) return rc;
  BRK_JOIN(ctx, st, 0);
  if (mode == 0) {
    // scores = q c^T; softmax CE (SUM) with accidental-hit removal; in place P = softmax - I
    if ((rc = gemm(ctx, st, tcore, ws->q, ws->c, ws->scores, nullptr, B, B, S, S, S, B, 0, 1, 1.f, 0, false))) return rc;
    inbatch_softmax_kernel<<<B, 256, 0, st>>>(ws->scores, cand_ids, B, training, ws->acc);
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
  for (int k = 0; k < 2; ++k) {
    cudaStream_t sk = k == 0 ? st : fk;
    cudaStream_t sd = wide ? ctx->fork_stream[1 + k] : sk;
    if (mode == 0) {
      if ((rc = gemm(ctx, sk, tcore, ws->scores, other[k], dz[k], nullptr, B, S, B, B, S, S, k, 0, 1.f, 1, true))) return rc;
    }
    if (wide) BRK_FORK(ctx, sk, 1 + k);
    float* gW = tw[k]->dense.g;
    float* gb = gW + int64_t(E[k]) * S;
    if ((rc = gemm(ctx, sd, tcore, e[k], dz[k], gW, nullptr, E[k], S, B, E[k], S, S, 1, 0, 1.f, 1, true))) return rc;
    colsum_kernel<<<dim3((S + 127) / 128, (B + 63) / 64), 128, 0, sd>>>(dz[k], B, S, S, gb);
    BRK_LAUNCH_CHECK();
    if (k == 0) {                                  // the loss scalar rides on the user tower's side stream
      finish_loss_kernel<<<1, 1, 0, sd>>>(ws->acc, loss_out);
      BRK_LAUNCH_CHECK();
    }
    // de = dz W^T: W stored [E,S] = "B stored [N,K]" with N = E, K = S  (tb = 1); its own buffer: the dW product
    // beside it is still reading the gathered rows e
    if ((rc = gemm(ctx, sk, tcore, dz[k], tw[k]->dense.w, de[k], nullptr, B, E[k], S, S, S, E[k], 0, 1, 1.f, 0, false))) return rc;
    rc = tsh[k] ? brk_scatter_add_rows_sharded(ctx, tsh[k], E[k], ids[k], batch, de[k], (void*)sk)
                : brk_scatter_add_rows(ctx, tw[k]->emb.g, tw[k]->emb.rows, E[k], ids[k], batch, de[k], tw[k]->emb.touched, 0,
                                       (void*)sk);
    if (rc) return rc;
    if (wide) BRK_JOIN(ctx, sk, 1 + k);
  }
  BRK_JOIN(ctx, st, 0);
  return 0;
}

extern "C" int brk_twotower_step(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u,
                                 const int32_t* i, const int32_t* cand_ids, const float* labels, int64_t batch,
                                 int32_t mode, int32_t training, const brk_twotower_workspace* ws, float* loss_out,
                                 void* stream) {
  BRK_REQUIRE(ctx && user && item && u && i && ws, BRK_E_ARG, "brk_twotower_step: null argument");
  BRK_REQUIRE(user->S == item->S && batch > 0 && batch < (1 << 30), BRK_E_ARG, "brk_twotower_step: S %d vs %d, batch %lld",
              user->S, item->S, (long long)batch);
  BRK_REQUIRE((mode & 0xFF) == 0 || labels, BRK_E_ARG, "brk_twotower_step: rdZero mode needs labels");
  BRK_REQUIRE(ws->eu && ws->ei && ws->q && ws->c && ws->dq && ws->dc && ws->acc && ((mode & 0xFF) != 0 || ws->scores), BRK_E_ARG,
              "brk_twotower_step: workspace missing");
  BRK_REQUIRE(!training || (user->emb.g && item->emb.g && user->dense.g && item->dense.g && ws->deu && ws->dei), BRK_E_ARG,
              "brk_twotower_step: gradient accumulators / deu, dei workspace missing");
  return twotower_step(ctx, user, item, nullptr, u, i, cand_ids, labels, batch, mode, training, ws, loss_out, stream);
}

static int check_shards(const brk_shards* s, int32_t E, const char* which) {
  BRK_REQUIRE(s->world >= 1 && s->world <= BRK_MAX_PEERS, BRK_E_ARG, "brk_twotower_step_sharded: %s world=%d (1..%d)", which,
              s->world, BRK_MAX_PEERS);
  BRK_REQUIRE(s->rank >= 0 && s->rank < s->world, BRK_E_ARG, "brk_twotower_step_sharded: %s rank=%d world=%d", which, s->rank,
              s->world);
  for (int p = 0; p < s->world; ++p)
    BRK_REQUIRE(s->w[p] && s->g[p] && s->touched[p], BRK_E_ARG, "brk_twotower_step_sharded: %s shard %d has a null w / g / touched",
                which, p);
  BRK_REQUIRE(E > 0 && (E & 3) == 0, BRK_E_ARG, "brk_twotower_step_sharded: %s width %d is not a positive multiple of 4", which, E);
  return 0;
}

extern "C" int brk_twotower_step_sharded(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const brk_twotower_shards* sh,
                                         const int32_t* u, const int32_t* i, const int32_t* cand_ids, const float* labels,
                                         int64_t batch, int32_t mode, const brk_twotower_workspace* ws, float* loss_out,
                                         void* stream) {
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
  return twotower_step(ctx, user, item, sh, u, i, cand_ids, labels, batch, mode, 1, ws, loss_out, stream);
}

extern "C" int brk_tower_forward_sharded(brk_ctx* ctx, const brk_tower* t, const brk_shards* sh, const int32_t* ids, int64_t n,
                                         float* emb_out, float* out, void* stream) {
  BRK_REQUIRE(ctx && t && sh && ids && emb_out && out, BRK_E_ARG, "brk_tower_forward_sharded: null argument");
  BRK_REQUIRE(t->dense.w && t->E > 0 && t->S > 0 && n > 0, BRK_E_ARG, "brk_tower_forward_sharded: bad tower");
  return tower_forward(ctx, t, ids, n, emb_out, out, 0, stream, sh);
}

// Training step + Keras Adagrad (twoTower.py:89-102 with the optimizer of :278-279) in one call.  In-batch-softmax steps
// on the tensor cores whose batch fits on chip run as ONE launch (twotower_fused.cu: the optimizer is the last phase of the
// same cooperative kernel and only visits the rows the batch touched); everything else is brk_twotower_step followed by
// the dense or row-sparse Adagrad pass of optim.cu (row-sparse for tables above rows_threshold_bytes that carry a bitmask).
extern "C" int brk_twotower_train_step(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u,
                                       const int32_t* i, const int32_t* cand_ids, const float* labels, int64_t batch,
                                       int32_t mode, const brk_twotower_workspace* ws, float lr, float eps,
                                       int64_t rows_threshold_bytes, float* loss_out, void* stream) {
  BRK_REQUIRE(ctx && user && item && u && i && ws, BRK_E_ARG, "brk_twotower_train_step: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  int rc;
  if ((mode & 0xFF) == 0 && (mode & 0x100) && user->S == item->S && batch > 0 && batch < (1 << 30) && ws->q && ws->c && ws->dq &&
      ws->dc && ws->acc && user->emb.g && item->emb.g && user->dense.g && item->dense.g) {
    int handled = 0;
    if ((rc = brk_twotower_step_fused(ctx, user, item, u, i, cand_ids, batch, 1, ws, loss_out, st, &handled, 1, lr, eps, nullptr)))
      return rc;
    if (handled) return 0;
  }
  if ((rc = brk_twotower_step(ctx, user, item, u, i, cand_ids, labels, batch, mode, 1, ws, loss_out, stream))) return rc;
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
