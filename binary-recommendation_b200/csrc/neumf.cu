// Fused NeuMF forward + backward (K1+K2+K3+K4+K5): /root/reference/src/models/NeuMFModel.py:53-100
// (class spec) and /root/reference/trainers/NFC_plain.py:109-155 (script spec).
//
//   x0 = [uMLP[u], iMLP[i]] -> drop -> act(W1) -> BN1 -> drop -> act(W2) -> BN2 -> drop -> act(W3) = h3
//   out = sigmoid([h3, <uMF[u], iMF[i]>] W4 + b4);  loss = MSE | BCE
//
// Training-mode BatchNorm needs whole-batch statistics after layers 1 and 2 and, in the backward
// pass, whole-batch sums of dy and dy*xhat, so one step is five kernels separated exactly at those
// dependencies (A: fwd1, B: fwd2, C: fwd3 + head + loss + bwd head/3, D: bwd2, E: bwd1); the sums
// travel through a small double-precision accumulator block.  No activation is ever stored
// sample-major: the three intermediates that cross a kernel boundary (h1, h2 and the BN-output
// gradients) are feature-major [H, B] so that thread-per-sample accesses are coalesced.
//
// Inside a kernel a CTA owns a tile of 128 samples, one thread per sample:
//   * embedding rows are gathered cooperatively (consecutive threads read consecutive 16-byte pieces
//     of the same row -> full 128-byte segments) into a padded shared-memory tile;
//   * weights live in shared memory and are read as broadcast float4; accumulators in registers;
//   * weight gradients are a block-level GEMM  dW = X^T dZ  over the tile out of shared memory with a
//     4x4 register tile per thread, then one float RED per entry per CTA;
//   * embedding gradients leave as 16-byte vector REDs into the dense accumulators (as in bpr.cu);
//   * dropout masks are regenerated from Philox (never stored): stream defined in oracle/neumf.py.
// Algorithmic HBM/L2 traffic per interaction at E=32: 4 rows gathered (512 B) + 12 B ids/label +
// 4 B prediction (528 B, SURVEY.md 8d) + 4 row gradients (512 B) + 2x re-gather in the backward.
//
// These kernels serve the script spec (10;100,50,10): the tiled kernels of neumf2.cu need power-of-two widths.
#include "common.cuh"
#include "neumf_common.cuh"   // parameter / accumulator layouts, BatchNorm and dropout constants, activations
#include <math_constants.h>

namespace {

using v2::Acc; using v2::Layout;
using v2::act_f; using v2::act_grad; using v2::drop16;
using v2::kBnEps; using v2::kBnMomentum;

constexpr int kTile = 128;            // samples per CTA = threads per CTA

__host__ __device__ constexpr int pad4(int x) { return (x + 3) & ~3; }

struct NeumfArgs {
  brk_table uMLP, iMLP, uMF, iMF, dense;
  const int32_t* u; const int32_t* i; const float* y;
  int64_t B; int64_t first_index; int64_t global_B;   // global_B scales the loss gradient (data parallel)
  float* h1; float* h2; float* dy1; float* dy2;   // feature-major [H, B]
  float* out;                                      // [B] predictions
  double* acc;                                     // Acc<H1,H2>::total doubles, zero on entry
  float* bn_moving;                                // mm1[H1] mv1[H1] mm2[H2] mv2[H2]
  float* loss_out;
  uint32_t drop_seed, drop_epoch; int32_t dropout; // dropout != 0 -> Philox masks, keep 205/256
  int32_t loss_kind;                               // 0 mse, 1 bce
  int32_t training;
};

// In-place dropout on a shared-memory row of n features.
template <int N>
__device__ __forceinline__ void drop_row(float* row, uint64_t idx, int layer, uint32_t seed, uint32_t epoch) {
#pragma unroll 1
  for (int c = 0; c < (N + 15) / 16; ++c) {
    float m[16];
    drop16(idx, c, layer, seed, epoch, m);
#pragma unroll
    for (int j = 0; j < 16; ++j) if (c * 16 + j < N) row[c * 16 + j] *= m[j];
  }
}

// Cooperative coalesced gather of `rows_valid` embedding rows of width E into tile[s*pitch + col0 ...].
template <int E>
__device__ __forceinline__ void stage_rows(float* tile, int pitch, int col0, const float* __restrict__ table,
                                           const int32_t* ids_sm, int rows_valid) {
  if constexpr (E % 4 == 0) {
    constexpr int C = E / 4;
    for (int idx = threadIdx.x; idx < rows_valid * C; idx += kTile) {
      const int s = idx / C, c = idx - s * C;
      const float4 v = __ldg(reinterpret_cast<const float4*>(table + int64_t(ids_sm[s]) * E) + c);
      *reinterpret_cast<float4*>(tile + s * pitch + col0 + c * 4) = v;
    }
  } else {
    for (int idx = threadIdx.x; idx < rows_valid * E; idx += kTile) {
      const int s = idx / E, c = idx - s * E;
      tile[s * pitch + col0 + c] = __ldg(table + int64_t(ids_sm[s]) * E + c);
    }
  }
}

// Copy an [IN, OUT] row-major weight matrix into shared memory with the row padded to OUTP floats.
template <int IN, int OUT>
__device__ __forceinline__ void stage_weight(float* dst, const float* __restrict__ src) {
  constexpr int OUTP = pad4(OUT);
  for (int idx = threadIdx.x; idx < IN * OUTP; idx += kTile) {
    const int k = idx / OUTP, j = idx - k * OUTP;
    dst[idx] = j < OUT ? __ldg(src + k * OUT + j) : 0.f;
  }
}

// acc[j] = bias[j] + sum_k x[k] * W[k][j]   (x: this thread's shared-memory row; W, bias in smem)
template <int IN, int OUT>
__device__ __forceinline__ void dense_fwd(const float* xrow, const float* Wsm, const float* bsm, float (&acc)[pad4(OUT)]) {
  constexpr int OUTP = pad4(OUT);
#pragma unroll
  for (int j = 0; j < OUTP; ++j) acc[j] = j < OUT ? bsm[j] : 0.f;
#pragma unroll 2
  for (int k = 0; k < IN; ++k) {
    const float xk = xrow[k];
    const float4* wr = reinterpret_cast<const float4*>(Wsm + k * OUTP);
#pragma unroll
    for (int j4 = 0; j4 < OUTP / 4; ++j4) {
      const float4 w = wr[j4];
      acc[4 * j4 + 0] = fmaf(xk, w.x, acc[4 * j4 + 0]);
      acc[4 * j4 + 1] = fmaf(xk, w.y, acc[4 * j4 + 1]);
      acc[4 * j4 + 2] = fmaf(xk, w.z, acc[4 * j4 + 2]);
      acc[4 * j4 + 3] = fmaf(xk, w.w, acc[4 * j4 + 3]);
    }
  }
}
// dx[k] = sum_j dz[j] * W[k][j]
template <int IN, int OUT>
__device__ __forceinline__ float dense_bwd_one(int k, const float (&dz)[pad4(OUT)], const float* Wsm) {
  constexpr int OUTP = pad4(OUT);
  const float4* wr = reinterpret_cast<const float4*>(Wsm + k * OUTP);
  float s = 0.f;
#pragma unroll
  for (int j4 = 0; j4 < OUTP / 4; ++j4) {
    const float4 w = wr[j4];
    s = fmaf(dz[4 * j4 + 0], w.x, s); s = fmaf(dz[4 * j4 + 1], w.y, s);
    s = fmaf(dz[4 * j4 + 2], w.z, s); s = fmaf(dz[4 * j4 + 3], w.w, s);
  }
  return s;
}

// Block GEMM over the tile: gW[k][j] += sum_s X[s][k] * dZ[s][j], gb[j] += sum_s dZ[s][j].
// X: [kTile][xp] (first IN columns), dZ: [kTile][zp] (first OUT columns; padded columns are zero).
template <int IN, int OUT>
__device__ __forceinline__ void wgrad_block(const float* X, int xp, const float* dZ, int zp, float* __restrict__ gW,
                                            float* __restrict__ gb) {
  constexpr int OUTP = pad4(OUT), INP = pad4(IN);
  constexpr int TJ = OUTP / 4, TK = INP / 4, NT = TJ * TK;          // 4x4 register tiles
  for (int t = threadIdx.x; t < NT; t += kTile) {
    const int tk = t / TJ, tj = t - tk * TJ;
    float a[4][4] = {};
#pragma unroll 4
    for (int s = 0; s < kTile; ++s) {
      float xv[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) xv[q] = (4 * tk + q < IN) ? X[s * xp + 4 * tk + q] : 0.f;
      const float4 z = *reinterpret_cast<const float4*>(dZ + s * zp + 4 * tj);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        a[q][0] = fmaf(xv[q], z.x, a[q][0]); a[q][1] = fmaf(xv[q], z.y, a[q][1]);
        a[q][2] = fmaf(xv[q], z.z, a[q][2]); a[q][3] = fmaf(xv[q], z.w, a[q][3]);
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int r = 0; r < 4; ++r)
        if (4 * tk + q < IN && 4 * tj + r < OUT) atomicAdd(gW + (4 * tk + q) * OUT + 4 * tj + r, a[q][r]);
  }
  if (gb != nullptr) {
    for (int j = threadIdx.x; j < OUT; j += kTile) {
      float s = 0.f;
      for (int r = 0; r < kTile; ++r) s += dZ[r * zp + j];
      atomicAdd(gb + j, s);
    }
  }
}

// Per-feature block sums of a [kTile][pitch] tile (first H columns) and of its square (or of a product
// with a second tile): one double atomic per feature per CTA.
template <int H>
__device__ __forceinline__ void col_sums(const float* A, int ap, const float* Bm, int bp, double* sumA, double* sumAB) {
  // double accumulation: with sigmoid activations h ~ 0.5 +- 0.01, so E[h^2] - mean^2 cancels 3-4 digits;
  // fp32 partial sums here cost a 2.5e-4 relative error in the variance (measured against an fp64 oracle).
  for (int f = threadIdx.x; f < H; f += kTile) {
    double s = 0.0, q = 0.0;
    for (int r = 0; r < kTile; ++r) {
      const double a = double(A[r * ap + f]);
      s += a;
      q = fma(a, Bm ? double(Bm[r * bp + f]) : a, q);
    }
    atomicAdd(sumA + f, s);
    atomicAdd(sumAB + f, q);
  }
}

// mean / rstd per feature from the global sums (training) or the moving statistics (inference).
template <int H>
__device__ __forceinline__ void bn_prepare(float* mean_sm, float* rstd_sm, const double* sum, const double* sq,
                                           const float* mov_mean, const float* mov_var, int64_t B, bool training) {
  for (int f = threadIdx.x; f < H; f += kTile) {
    float mu, var;
    if (training) {
      const double m = sum[f] / double(B);
      mu = float(m);
      var = float(fmax(sq[f] / double(B) - m * m, 0.0));      // biased variance, as Keras
    } else {
      mu = mov_mean[f]; var = mov_var[f];
    }
    mean_sm[f] = mu;
    rstd_sm[f] = 1.0f / sqrtf(var + kBnEps);
  }
}

extern __shared__ __align__(16) float smem_f[];

// ------------------------------------------------------------------------------------------------
// A: gather MLP rows, dropout0, layer 1, store h1 (feature-major), accumulate BN1 sums
// ------------------------------------------------------------------------------------------------
template <int E, int H1, int H2, int H3, int ACT>
__global__ void __launch_bounds__(kTile) neumf_fwd1(const NeumfArgs A) {
  using L = Layout<E, H1, H2, H3>; using AC = Acc<H1, H2>;
  constexpr int XP = 2 * E + 4, HP = pad4(H1) + 4;
  float* X = smem_f;                         // [kTile][XP]
  float* W = X + kTile * XP;                 // [2E][pad4(H1)]
  float* bias = W + 2 * E * pad4(H1);        // [pad4(H1)]
  float* Hs = bias + pad4(H1);               // [kTile][HP]
  int32_t* ids = reinterpret_cast<int32_t*>(Hs + kTile * HP);   // [2][kTile]
  const int64_t b0 = int64_t(blockIdx.x) * kTile;
  const int valid = int((A.B - b0) < int64_t(kTile) ? (A.B - b0) : int64_t(kTile));
  const int t = threadIdx.x;
  if (t < valid) { ids[t] = __ldg(A.u + b0 + t); ids[kTile + t] = __ldg(A.i + b0 + t); }
  stage_weight<2 * E, H1>(W, A.dense.w + L::W1);
  for (int j = t; j < pad4(H1); j += kTile) bias[j] = j < H1 ? A.dense.w[L::b1 + j] : 0.f;
  __syncthreads();
  stage_rows<E>(X, XP, 0, A.uMLP.w, ids, valid);
  stage_rows<E>(X, XP, E, A.iMLP.w, ids + kTile, valid);
  __syncthreads();
  float acc[pad4(H1)];
  if (t < valid) {
    if (A.dropout && A.training) drop_row<2 * E>(X + t * XP, uint64_t(A.first_index + b0 + t), 0, A.drop_seed, A.drop_epoch);
    dense_fwd<2 * E, H1>(X + t * XP, W, bias, acc);
#pragma unroll
    for (int j = 0; j < pad4(H1); ++j) {
      acc[j] = j < H1 ? act_f<ACT>(acc[j]) : 0.f;
      if (j < H1) A.h1[int64_t(j) * A.B + b0 + t] = acc[j];
    }
  } else {
#pragma unroll
    for (int j = 0; j < pad4(H1); ++j) acc[j] = 0.f;
  }
  if (A.training) {
#pragma unroll
    for (int j = 0; j < pad4(H1); ++j) Hs[t * HP + j] = acc[j];
    __syncthreads();
    col_sums<H1>(Hs, HP, nullptr, 0, A.acc + AC::s1, A.acc + AC::q1);
  }
}

// ------------------------------------------------------------------------------------------------
// B: BN1, dropout1, layer 2, store h2, accumulate BN2 sums
// ------------------------------------------------------------------------------------------------
template <int E, int H1, int H2, int H3, int ACT>
__global__ void __launch_bounds__(kTile) neumf_fwd2(const NeumfArgs A) {
  using L = Layout<E, H1, H2, H3>; using AC = Acc<H1, H2>;
  constexpr int XP = pad4(H1) + 4, HP = pad4(H2) + 4;
  float* X = smem_f;                         // [kTile][XP]  d1 = dropout(bn1(h1))
  float* W = X + kTile * XP;                 // [H1][pad4(H2)]
  float* bias = W + H1 * pad4(H2);
  float* Hs = bias + pad4(H2);               // [kTile][HP]
  float* mean = Hs + kTile * HP; float* rstd = mean + H1; float* gam = rstd + H1; float* bet = gam + H1;
  const int64_t b0 = int64_t(blockIdx.x) * kTile;
  const int valid = int((A.B - b0) < int64_t(kTile) ? (A.B - b0) : int64_t(kTile));
  const int t = threadIdx.x;
  stage_weight<H1, H2>(W, A.dense.w + L::W2);
  for (int j = t; j < pad4(H2); j += kTile) bias[j] = j < H2 ? A.dense.w[L::b2 + j] : 0.f;
  bn_prepare<H1>(mean, rstd, A.acc + AC::s1, A.acc + AC::q1, A.bn_moving, A.bn_moving + H1, A.B, A.training);
  for (int f = t; f < H1; f += kTile) { gam[f] = A.dense.w[L::g1 + f]; bet[f] = A.dense.w[L::be1 + f]; }
  __syncthreads();
  float acc[pad4(H2)];
  if (t < valid) {
    float* row = X + t * XP;
#pragma unroll 4
    for (int f = 0; f < H1; ++f)
      row[f] = gam[f] * (A.h1[int64_t(f) * A.B + b0 + t] - mean[f]) * rstd[f] + bet[f];
    if (A.dropout && A.training) drop_row<H1>(row, uint64_t(A.first_index + b0 + t), 1, A.drop_seed, A.drop_epoch);
    dense_fwd<H1, H2>(row, W, bias, acc);
#pragma unroll
    for (int j = 0; j < pad4(H2); ++j) {
      acc[j] = j < H2 ? act_f<ACT>(acc[j]) : 0.f;
      if (j < H2) A.h2[int64_t(j) * A.B + b0 + t] = acc[j];
    }
  } else {
#pragma unroll
    for (int j = 0; j < pad4(H2); ++j) acc[j] = 0.f;
  }
  if (A.training) {
#pragma unroll
    for (int j = 0; j < pad4(H2); ++j) Hs[t * HP + j] = acc[j];
    __syncthreads();
    col_sums<H2>(Hs, HP, nullptr, 0, A.acc + AC::s2, A.acc + AC::q2);
  }
}

// ------------------------------------------------------------------------------------------------
// C: BN2, dropout2, layer 3, MF dot, head, loss; backward of head and layer 3; BN2-output gradient
// ------------------------------------------------------------------------------------------------
template <int E, int H1, int H2, int H3, int ACT>
__global__ void __launch_bounds__(kTile) neumf_head(const NeumfArgs A) {
  using L = Layout<E, H1, H2, H3>; using AC = Acc<H1, H2>;
  constexpr int XP = pad4(H2) + 4, ZP = pad4(H3) + 4, MP = 2 * E + 4;
  float* X = smem_f;                         // [kTile][XP]  d2 = dropout(bn2(h2)); later dy2
  float* W = X + kTile * XP;                 // [H2][pad4(H3)]
  float* bias = W + H2 * pad4(H3);           // [pad4(H3)]
  float* w4 = bias + pad4(H3);               // [H3 + 2]: W4 (H3+1), b4
  float* Z = w4 + pad4(H3 + 2);              // [kTile][ZP]  dz3
  float* M = Z + kTile * ZP;                 // [kTile][MP]  uMF | iMF rows
  float* Xh = M + kTile * MP;                // [kTile][XP]  xhat2 (for the dy*xhat sums)
  float* mean = Xh + kTile * XP; float* rstd = mean + H2; float* gam = rstd + H2; float* bet = gam + H2;
  float* hz = bet + H2;                      // [kTile][H3+2]: z = [h3, mf] * dlogit and dlogit (head grads)
  int32_t* ids = reinterpret_cast<int32_t*>(hz + kTile * (H3 + 2));
  __shared__ double red[32];
  const int64_t b0 = int64_t(blockIdx.x) * kTile;
  const int valid = int((A.B - b0) < int64_t(kTile) ? (A.B - b0) : int64_t(kTile));
  const int t = threadIdx.x;
  if (t < valid) { ids[t] = __ldg(A.u + b0 + t); ids[kTile + t] = __ldg(A.i + b0 + t); }
  stage_weight<H2, H3>(W, A.dense.w + L::W3);
  for (int j = t; j < pad4(H3); j += kTile) bias[j] = j < H3 ? A.dense.w[L::b3 + j] : 0.f;
  for (int j = t; j < H3 + 2; j += kTile) w4[j] = A.dense.w[L::W4 + j];
  bn_prepare<H2>(mean, rstd, A.acc + AC::s2, A.acc + AC::q2, A.bn_moving + 2 * H1, A.bn_moving + 2 * H1 + H2, A.B, A.training);
  for (int f = t; f < H2; f += kTile) { gam[f] = A.dense.w[L::g2 + f]; bet[f] = A.dense.w[L::be2 + f]; }
  __syncthreads();
  stage_rows<E>(M, MP, 0, A.uMF.w, ids, valid);
  stage_rows<E>(M, MP, E, A.iMF.w, ids + kTile, valid);
  __syncthreads();

  float dz[pad4(H3)];
  float loss_local = 0.f, dlogit = 0.f;
  float* row = X + t * XP;
  if (t < valid) {
#pragma unroll 4
    for (int f = 0; f < H2; ++f) {
      const float xh = (A.h2[int64_t(f) * A.B + b0 + t] - mean[f]) * rstd[f];
      Xh[t * XP + f] = xh;
      row[f] = gam[f] * xh + bet[f];
    }
    if (A.dropout && A.training) drop_row<H2>(row, uint64_t(A.first_index + b0 + t), 2, A.drop_seed, A.drop_epoch);
    float h3[pad4(H3)];
    dense_fwd<H2, H3>(row, W, bias, h3);
    float logit = w4[H3 + 1];
#pragma unroll
    for (int j = 0; j < H3; ++j) { h3[j] = act_f<ACT>(h3[j]); logit = fmaf(h3[j], w4[j], logit); }
    float mf = 0.f;
    const float* mr = M + t * MP;
#pragma unroll 8
    for (int f = 0; f < E; ++f) mf = fmaf(mr[f], mr[E + f], mf);
    logit = fmaf(mf, w4[H3], logit);
    const float o = 1.0f / (1.0f + expf(-logit));
    A.out[b0 + t] = o;
    const float yv = __ldg(A.y + b0 + t);
    const float invB = 1.0f / float(A.global_B);
    if (A.loss_kind == 0) {
      const float e = o - yv;
      loss_local = e * e;
      dlogit = 2.f * e * o * (1.f - o) * invB;
    } else {
      // binary cross-entropy from logits: max(z,0) - z*y + log(1 + exp(-|z|))
      loss_local = fmaxf(logit, 0.f) - logit * yv + log1pf(expf(-fabsf(logit)));
      dlogit = (o - yv) * invB;
    }
    if (A.training) {
      // head gradients staged for the block reduction: z_j * dlogit, then dlogit (bias)
#pragma unroll
      for (int j = 0; j < H3; ++j) hz[t * (H3 + 2) + j] = h3[j] * dlogit;
      hz[t * (H3 + 2) + H3] = mf * dlogit;
      hz[t * (H3 + 2) + H3 + 1] = dlogit;
#pragma unroll
      for (int j = 0; j < pad4(H3); ++j)
        dz[j] = j < H3 ? dlogit * w4[j] * act_grad<ACT>(h3[j]) : 0.f;
    }
  } else {
#pragma unroll
    for (int j = 0; j < pad4(H3); ++j) dz[j] = 0.f;
    if (A.training) {
      for (int f = 0; f < H2; ++f) { row[f] = 0.f; Xh[t * XP + f] = 0.f; }
      for (int j = 0; j < H3 + 2; ++j) hz[t * (H3 + 2) + j] = 0.f;
    }
  }
  // loss: block partial -> double accumulator (finalised by the last kernel of the step)
  const double lsum = block_sum_double(double(loss_local), red);
  if (t == 0) atomicAdd(A.acc + AC::loss, lsum);
  if (!A.training) return;

#pragma unroll
  for (int j = 0; j < pad4(H3); ++j) Z[t * ZP + j] = dz[j];
  __syncthreads();
  // weight gradients of layer 3 and the head
  wgrad_block<H2, H3>(X, XP, Z, ZP, A.dense.g + L::W3, A.dense.g + L::b3);
  for (int j = t; j < H3 + 2; j += kTile) {
    float s = 0.f;
    for (int r = 0; r < kTile; ++r) s += hz[r * (H3 + 2) + j];
    atomicAdd(A.dense.g + L::W4 + j, s);                  // W4[0..H3] then b4 (contiguous in the layout)
  }
  __syncthreads();
  // MF embedding gradients and the gradient w.r.t. BN2's output
  if (t < valid) {
    const float dmf = dlogit * w4[H3];
    const float* mr = M + t * MP;
    float* gu = A.uMF.g + int64_t(ids[t]) * E;
    float* gi = A.iMF.g + int64_t(ids[kTile + t]) * E;
    if constexpr (E % 4 == 0) {
#pragma unroll 4
      for (int c = 0; c < E; c += 4) {
        red_add_f4(gu + c, make_float4(dmf * mr[E + c], dmf * mr[E + c + 1], dmf * mr[E + c + 2], dmf * mr[E + c + 3]));
        red_add_f4(gi + c, make_float4(dmf * mr[c], dmf * mr[c + 1], dmf * mr[c + 2], dmf * mr[c + 3]));
      }
    } else {
      for (int c = 0; c < E; ++c) { atomicAdd(gu + c, dmf * mr[E + c]); atomicAdd(gi + c, dmf * mr[c]); }
    }
    float m16[16];
#pragma unroll 1
    for (int k = 0; k < H2; ++k) {
      if (A.dropout && (k & 15) == 0) drop16(uint64_t(A.first_index + b0 + t), k >> 4, 2, A.drop_seed, A.drop_epoch, m16);
      float d = dense_bwd_one<H2, H3>(k, dz, W);
      if (A.dropout) {
        float mk = m16[0];
#pragma unroll
        for (int q = 1; q < 16; ++q) mk = ((k & 15) == q) ? m16[q] : mk;
        d *= mk;
      }
      row[k] = d;                                           // dy2 (gradient w.r.t. BN2 output), in place
      A.dy2[int64_t(k) * A.B + b0 + t] = d;
    }
  }
  __syncthreads();
  col_sums<H2>(X, XP, Xh, XP, A.acc + AC::d2, A.acc + AC::e2);
}

// ------------------------------------------------------------------------------------------------
// D: BN2 backward, layer 2 backward, gradient w.r.t. BN1 output
// ------------------------------------------------------------------------------------------------
template <int E, int H1, int H2, int H3, int ACT>
__global__ void __launch_bounds__(kTile) neumf_bwd2(const NeumfArgs A) {
  using L = Layout<E, H1, H2, H3>; using AC = Acc<H1, H2>;
  constexpr int XP = pad4(H1) + 4, ZP = pad4(H2) + 4;
  float* X = smem_f;                         // [kTile][XP]  d1 (layer-2 input); later dy1
  float* W = X + kTile * XP;                 // [H1][pad4(H2)]
  float* Z = W + H1 * pad4(H2);              // [kTile][ZP]  dz2
  float* Xh = Z + kTile * ZP;                // [kTile][XP]  xhat1
  float* mean1 = Xh + kTile * XP; float* rstd1 = mean1 + H1; float* gam1 = rstd1 + H1; float* bet1 = gam1 + H1;
  float* mean2 = bet1 + H1; float* rstd2 = mean2 + H2; float* gam2 = rstd2 + H2;
  float* sdy = gam2 + H2; float* sdyx = sdy + H2;      // batch means of dy2 and dy2*xhat2
  const int64_t b0 = int64_t(blockIdx.x) * kTile;
  const int valid = int((A.B - b0) < int64_t(kTile) ? (A.B - b0) : int64_t(kTile));
  const int t = threadIdx.x;
  stage_weight<H1, H2>(W, A.dense.w + L::W2);
  bn_prepare<H1>(mean1, rstd1, A.acc + AC::s1, A.acc + AC::q1, nullptr, nullptr, A.B, true);
  bn_prepare<H2>(mean2, rstd2, A.acc + AC::s2, A.acc + AC::q2, nullptr, nullptr, A.B, true);
  for (int f = t; f < H1; f += kTile) { gam1[f] = A.dense.w[L::g1 + f]; bet1[f] = A.dense.w[L::be1 + f]; }
  for (int f = t; f < H2; f += kTile) {
    gam2[f] = A.dense.w[L::g2 + f];
    sdy[f] = float(A.acc[AC::d2 + f] / double(A.B));
    sdyx[f] = float(A.acc[AC::e2 + f] / double(A.B));
    if (blockIdx.x == 0) {                               // BN2 parameter gradients: d beta = sum dy, d gamma = sum dy*xhat
      A.dense.g[L::be2 + f] += float(A.acc[AC::d2 + f]);
      A.dense.g[L::g2 + f] += float(A.acc[AC::e2 + f]);
    }
  }
  __syncthreads();
  float dz[pad4(H2)];
  float* row = X + t * XP;
  if (t < valid) {
#pragma unroll 4
    for (int f = 0; f < H1; ++f) {
      const float xh = (A.h1[int64_t(f) * A.B + b0 + t] - mean1[f]) * rstd1[f];
      Xh[t * XP + f] = xh;
      row[f] = gam1[f] * xh + bet1[f];
    }
    if (A.dropout) drop_row<H1>(row, uint64_t(A.first_index + b0 + t), 1, A.drop_seed, A.drop_epoch);
#pragma unroll
    for (int j = 0; j < pad4(H2); ++j) {
      if (j < H2) {
        const float h = A.h2[int64_t(j) * A.B + b0 + t];
        const float xh = (h - mean2[j]) * rstd2[j];
        const float dy = A.dy2[int64_t(j) * A.B + b0 + t];
        const float dh = gam2[j] * rstd2[j] * (dy - sdy[j] - xh * sdyx[j]);
        dz[j] = dh * act_grad<ACT>(h);
      } else dz[j] = 0.f;
    }
  } else {
#pragma unroll
    for (int j = 0; j < pad4(H2); ++j) dz[j] = 0.f;
    for (int f = 0; f < H1; ++f) { row[f] = 0.f; Xh[t * XP + f] = 0.f; }
  }
#pragma unroll
  for (int j = 0; j < pad4(H2); ++j) Z[t * ZP + j] = dz[j];
  __syncthreads();
  wgrad_block<H1, H2>(X, XP, Z, ZP, A.dense.g + L::W2, A.dense.g + L::b2);
  __syncthreads();
  if (t < valid) {
    float m16[16];
#pragma unroll 1
    for (int k = 0; k < H1; ++k) {
      if (A.dropout && (k & 15) == 0) drop16(uint64_t(A.first_index + b0 + t), k >> 4, 1, A.drop_seed, A.drop_epoch, m16);
      float d = dense_bwd_one<H1, H2>(k, dz, W);
      if (A.dropout) {
        float mk = m16[0];
#pragma unroll
        for (int q = 1; q < 16; ++q) mk = ((k & 15) == q) ? m16[q] : mk;
        d *= mk;
      }
      row[k] = d;
      A.dy1[int64_t(k) * A.B + b0 + t] = d;
    }
  }
  __syncthreads();
  col_sums<H1>(X, XP, Xh, XP, A.acc + AC::d1, A.acc + AC::e1);
}

// ------------------------------------------------------------------------------------------------
// E: BN1 backward, layer 1 backward, MLP embedding gradients, BN moving statistics, loss output
// ------------------------------------------------------------------------------------------------
template <int E, int H1, int H2, int H3, int ACT>
__global__ void __launch_bounds__(kTile) neumf_bwd1(const NeumfArgs A, unsigned int* ticket) {
  using L = Layout<E, H1, H2, H3>; using AC = Acc<H1, H2>;
  constexpr int XP = 2 * E + 4, ZP = pad4(H1) + 4;
  float* X = smem_f;                         // [kTile][XP]  d0 (layer-1 input)
  float* W = X + kTile * XP;                 // [2E][pad4(H1)]
  float* Z = W + 2 * E * pad4(H1);           // [kTile][ZP]  dz1
  float* mean1 = Z + kTile * ZP; float* rstd1 = mean1 + H1; float* gam1 = rstd1 + H1;
  float* sdy = gam1 + H1; float* sdyx = sdy + H1;
  int32_t* ids = reinterpret_cast<int32_t*>(sdyx + H1);
  const int64_t b0 = int64_t(blockIdx.x) * kTile;
  const int valid = int((A.B - b0) < int64_t(kTile) ? (A.B - b0) : int64_t(kTile));
  const int t = threadIdx.x;
  if (t < valid) { ids[t] = __ldg(A.u + b0 + t); ids[kTile + t] = __ldg(A.i + b0 + t); }
  stage_weight<2 * E, H1>(W, A.dense.w + L::W1);
  bn_prepare<H1>(mean1, rstd1, A.acc + AC::s1, A.acc + AC::q1, nullptr, nullptr, A.B, true);
  for (int f = t; f < H1; f += kTile) {
    gam1[f] = A.dense.w[L::g1 + f];
    sdy[f] = float(A.acc[AC::d1 + f] / double(A.B));
    sdyx[f] = float(A.acc[AC::e1 + f] / double(A.B));
    if (blockIdx.x == 0) {
      A.dense.g[L::be1 + f] += float(A.acc[AC::d1 + f]);
      A.dense.g[L::g1 + f] += float(A.acc[AC::e1 + f]);
    }
  }
  __syncthreads();
  stage_rows<E>(X, XP, 0, A.uMLP.w, ids, valid);
  stage_rows<E>(X, XP, E, A.iMLP.w, ids + kTile, valid);
  __syncthreads();
  float dz[pad4(H1)];
  float* row = X + t * XP;
  if (t < valid) {
    if (A.dropout) drop_row<2 * E>(row, uint64_t(A.first_index + b0 + t), 0, A.drop_seed, A.drop_epoch);
#pragma unroll
    for (int j = 0; j < pad4(H1); ++j) {
      if (j < H1) {
        const float h = A.h1[int64_t(j) * A.B + b0 + t];
        const float xh = (h - mean1[j]) * rstd1[j];
        const float dy = A.dy1[int64_t(j) * A.B + b0 + t];
        const float dh = gam1[j] * rstd1[j] * (dy - sdy[j] - xh * sdyx[j]);
        dz[j] = dh * act_grad<ACT>(h);
      } else dz[j] = 0.f;
    }
  } else {
#pragma unroll
    for (int j = 0; j < pad4(H1); ++j) dz[j] = 0.f;
    for (int f = 0; f < 2 * E; ++f) row[f] = 0.f;
  }
#pragma unroll
  for (int j = 0; j < pad4(H1); ++j) Z[t * ZP + j] = dz[j];
  __syncthreads();
  wgrad_block<2 * E, H1>(X, XP, Z, ZP, A.dense.g + L::W1, A.dense.g + L::b1);
  if (t < valid) {
    float* gu = A.uMLP.g + int64_t(ids[t]) * E;
    float* gi = A.iMLP.g + int64_t(ids[kTile + t]) * E;
    float m16[16];
#pragma unroll 1
    for (int k0 = 0; k0 < 2 * E; k0 += 4) {
      if (A.dropout && (k0 & 15) == 0) drop16(uint64_t(A.first_index + b0 + t), k0 >> 4, 0, A.drop_seed, A.drop_epoch, m16);
      float d[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        d[q] = (k0 + q < 2 * E) ? dense_bwd_one<2 * E, H1>(k0 + q, dz, W) : 0.f;
      }
      if (A.dropout) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float mk = m16[0];
#pragma unroll
          for (int r = 1; r < 16; ++r) mk = (((k0 + q) & 15) == r) ? m16[r] : mk;
          d[q] *= mk;
        }
      }
      if constexpr (E % 4 == 0) {
        float* dst = (k0 < E) ? gu + k0 : gi + (k0 - E);
        red_add_f4(dst, make_float4(d[0], d[1], d[2], d[3]));
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int k = k0 + q;
          if (k < 2 * E) atomicAdd(k < E ? gu + k : gi + (k - E), d[q]);
        }
      }
    }
  }
  // last CTA: BN moving statistics, loss output, accumulator reset
  __syncthreads();
  __shared__ bool last;
  if (t == 0) {
    __threadfence();
    last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (last) {
    __threadfence();
    for (int f = t; f < H1; f += kTile) {
      const double m = A.acc[AC::s1 + f] / double(A.B);
      const double v = fmax(A.acc[AC::q1 + f] / double(A.B) - m * m, 0.0);
      A.bn_moving[f] = A.bn_moving[f] * kBnMomentum + float(m) * (1.f - kBnMomentum);
      A.bn_moving[H1 + f] = A.bn_moving[H1 + f] * kBnMomentum + float(v) * (1.f - kBnMomentum);
    }
    for (int f = t; f < H2; f += kTile) {
      const double m = A.acc[AC::s2 + f] / double(A.B);
      const double v = fmax(A.acc[AC::q2 + f] / double(A.B) - m * m, 0.0);
      A.bn_moving[2 * H1 + f] = A.bn_moving[2 * H1 + f] * kBnMomentum + float(m) * (1.f - kBnMomentum);
      A.bn_moving[2 * H1 + H2 + f] = A.bn_moving[2 * H1 + H2 + f] * kBnMomentum + float(v) * (1.f - kBnMomentum);
    }
    if (t == 0 && A.loss_out) A.loss_out[0] = float(A.acc[AC::loss] / double(A.B));
    __syncthreads();
    for (int j = t; j < AC::total; j += kTile) A.acc[j] = 0.0;
    if (t == 0) *ticket = 0u;
  }
}

// inference epilogue: publish the loss (if labels were given) and reset the accumulators
template <int H1, int H2>
__global__ void neumf_finish_eval(double* acc, int64_t B, float* loss_out) {
  using AC = Acc<H1, H2>;
  if (threadIdx.x == 0 && loss_out) loss_out[0] = float(acc[AC::loss] / double(B));
  __syncthreads();
  for (int j = threadIdx.x; j < AC::total; j += blockDim.x) acc[j] = 0.0;
}

template <int E, int H1, int H2, int H3, int ACT>
int run_neumf(brk_ctx* ctx, const NeumfArgs& A, cudaStream_t st) {
  const int grid = int((A.B + kTile - 1) / kTile);
  auto bytes = [](size_t floats) { return floats * sizeof(float); };
  const size_t smA = bytes(size_t(kTile) * (2 * E + 4) + 2 * E * pad4(H1) + pad4(H1) + size_t(kTile) * (pad4(H1) + 4)) + 2 * kTile * 4;
  const size_t smB = bytes(size_t(kTile) * (pad4(H1) + 4) + H1 * pad4(H2) + pad4(H2) + size_t(kTile) * (pad4(H2) + 4) + 4 * H1);
  const size_t smC = bytes(size_t(kTile) * (pad4(H2) + 4) * 2 + H2 * pad4(H3) + pad4(H3) + pad4(H3 + 2) +
                           size_t(kTile) * (pad4(H3) + 4) + size_t(kTile) * (2 * E + 4) + 4 * H2 + size_t(kTile) * (H3 + 2)) + 2 * kTile * 4;
  const size_t smD = bytes(size_t(kTile) * (pad4(H1) + 4) * 2 + H1 * pad4(H2) + size_t(kTile) * (pad4(H2) + 4) + 4 * H1 + 5 * H2);
  const size_t smE = bytes(size_t(kTile) * (2 * E + 4) + 2 * E * pad4(H1) + size_t(kTile) * (pad4(H1) + 4) + 5 * H1) + 2 * kTile * 4;
  // the shared-memory opt-in is per device: set it for the current one on every call
  BRK_CUDA(cudaFuncSetAttribute(neumf_fwd1<E, H1, H2, H3, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smA)));
  BRK_CUDA(cudaFuncSetAttribute(neumf_fwd2<E, H1, H2, H3, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smB)));
  BRK_CUDA(cudaFuncSetAttribute(neumf_head<E, H1, H2, H3, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smC)));
  BRK_CUDA(cudaFuncSetAttribute(neumf_bwd2<E, H1, H2, H3, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smD)));
  BRK_CUDA(cudaFuncSetAttribute(neumf_bwd1<E, H1, H2, H3, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smE)));
  neumf_fwd1<E, H1, H2, H3, ACT><<<grid, kTile, smA, st>>>(A);
  neumf_fwd2<E, H1, H2, H3, ACT><<<grid, kTile, smB, st>>>(A);
  neumf_head<E, H1, H2, H3, ACT><<<grid, kTile, smC, st>>>(A);
  if (A.training) {
    neumf_bwd2<E, H1, H2, H3, ACT><<<grid, kTile, smD, st>>>(A);
    neumf_bwd1<E, H1, H2, H3, ACT><<<grid, kTile, smE, st>>>(A, ctx->tickets + 3);
  } else {
    neumf_finish_eval<H1, H2><<<1, 128, 0, st>>>(A.acc, A.B, A.loss_out);
  }
  BRK_LAUNCH_CHECK();
  return 0;
}

}  // namespace

// second-generation kernels (neumf2.cu); returns 1 when the spec is not one of theirs
int brk_neumf_step_v2(brk_ctx* ctx, const brk_neumf_model* m, const brk_neumf_shards* sh, const int32_t* u,
                      const int32_t* i, const float* y, int64_t batch, int64_t global_batch, int64_t first_index,
                      int32_t training, uint32_t dropout_seed, uint32_t dropout_epoch, const brk_neumf_workspace* ws,
                      float* out, float* loss_out, cudaStream_t st, int* rc_out);

int brk_neumf_step_tc(brk_ctx* ctx, const brk_neumf_model* m, const brk_neumf_shards* sh, const int32_t* u,
                      const int32_t* i, const float* y, int64_t batch, int64_t global_batch, int64_t first_index,
                      int32_t training, uint32_t dropout_seed, uint32_t dropout_epoch, const brk_neumf_workspace* ws,
                      float* out, float* loss_out, cudaStream_t st, int* rc_out);

int brk_neumf_step_fused(brk_ctx* ctx, const brk_neumf_model* m, const brk_neumf_shards* sh, const int32_t* u,
                         const int32_t* i, const float* y, int64_t batch, int64_t global_batch, int64_t first_index,
                         int32_t training, uint32_t dropout_seed, uint32_t dropout_epoch, const brk_neumf_workspace* ws,
                         float* out, float* loss_out, cudaStream_t st, int* rc_out, int* handled,
                         const brk_adam_hyper* adam_h, int64_t* adam_state);

int brk_neumf_step_generic(brk_ctx* ctx, const brk_neumf_model* m, const int32_t* u, const int32_t* i, const float* y,
                           int64_t B, int64_t global_batch, int64_t first_index, int32_t training, uint32_t seed, uint32_t epoch,
                           const brk_neumf_workspace* ws, float* out, float* loss_out, cudaStream_t st);

extern "C" int64_t brk_neumf_dense_floats_ex(int32_t E, int32_t H1, int32_t H2, int32_t H3, int32_t head_mf) {
  return int64_t(2) * E * H1 + 3 * H1 + int64_t(H1) * H2 + 3 * H2 + int64_t(H2) * H3 + H3 + (H3 + head_mf) + 1;
}
extern "C" int64_t brk_neumf_dense_floats(int32_t E, int32_t H1, int32_t H2, int32_t H3) {
  return brk_neumf_dense_floats_ex(E, H1, H2, H3, 1);
}
// the He et al. variant fields of brk_neumf_model (ABI 2): anything but the reference class graph
static inline bool brk_neumf_is_variant(const brk_neumf_model* m) {
  return (m->EMF > 0 && m->EMF != m->E) || m->mf_mode != 0 || m->no_batch_norm != 0;
}
extern "C" int64_t brk_neumf_acc_doubles(int32_t H1, int32_t H2) { return 4 * int64_t(H1) + 4 * int64_t(H2) + 1; }

extern "C" int brk_neumf_step(brk_ctx* ctx, const brk_neumf_model* m, const int32_t* u, const int32_t* i,
                              const float* y, int64_t batch, int64_t global_batch, int64_t first_index, int32_t training,
                              uint32_t dropout_seed, uint32_t dropout_epoch, const brk_neumf_workspace* ws,
                              float* out, float* loss_out, void* stream) {
  BRK_REQUIRE(ctx && m && u && i && ws && out, BRK_E_ARG, "brk_neumf_step: null argument");
  BRK_REQUIRE(y || !training, BRK_E_ARG, "brk_neumf_step: labels are required for training");
  BRK_REQUIRE(batch > 0, BRK_E_ARG, "brk_neumf_step: batch=%lld", (long long)batch);
  BRK_REQUIRE(m->uMLP.w && m->iMLP.w && m->uMF.w && m->iMF.w && m->dense.w && m->bn_moving, BRK_E_ARG,
              "brk_neumf_step: model tables missing");
  BRK_REQUIRE(!training || (m->uMLP.g && m->iMLP.g && m->uMF.g && m->iMF.g && m->dense.g), BRK_E_ARG,
              "brk_neumf_step: gradient accumulators missing");
  BRK_REQUIRE(ws->h1 && ws->h2 && ws->dy1 && ws->dy2 && ws->acc, BRK_E_ARG, "brk_neumf_step: workspace missing");
  if (m->tensor_cores || brk_neumf_is_variant(m)) {
    int rc2 = 0, handled = 0;
    brk_neumf_step_fused(ctx, m, nullptr, u, i, y, batch, global_batch, first_index, training, dropout_seed, dropout_epoch,
                         ws, out, loss_out, (cudaStream_t)stream, &rc2, &handled, nullptr, nullptr);
    if (handled) return rc2;
    if (brk_neumf_is_variant(m))                             // any other width of the variant: the any-width kernels
      return brk_neumf_step_generic(ctx, m, u, i, y, batch, global_batch, first_index, training, dropout_seed, dropout_epoch, ws,
                                    out, loss_out, (cudaStream_t)stream);
    if (brk_neumf_step_tc(ctx, m, nullptr, u, i, y, batch, global_batch, first_index, training, dropout_seed,
                          dropout_epoch, ws, out, loss_out, (cudaStream_t)stream, &rc2) == 0)
      return rc2;
    brk_set_error("brk_neumf_step: no tensor-core instance for E=%d H=(%d,%d,%d); built: (64;64,32,16) (32;32,16,8)",
                  m->E, m->H1, m->H2, m->H3);
    return BRK_E_ARG;
  }
  int rc2 = 0;
  if (brk_neumf_step_v2(ctx, m, nullptr, u, i, y, batch, global_batch, first_index, training, dropout_seed, dropout_epoch,
                        ws, out, loss_out, (cudaStream_t)stream, &rc2) == 0)
    return rc2;
  NeumfArgs A;
  A.uMLP = m->uMLP; A.iMLP = m->iMLP; A.uMF = m->uMF; A.iMF = m->iMF; A.dense = m->dense;
  A.u = u; A.i = i; A.y = y ? y : out; A.B = batch; A.first_index = first_index; A.global_B = global_batch > 0 ? global_batch : batch;
  A.h1 = ws->h1; A.h2 = ws->h2; A.dy1 = ws->dy1; A.dy2 = ws->dy2; A.out = out; A.acc = ws->acc;
  A.bn_moving = m->bn_moving; A.loss_out = y ? loss_out : nullptr;
  A.drop_seed = dropout_seed; A.drop_epoch = dropout_epoch;
  A.dropout = (m->dropout != 0 && training) ? 1 : 0;
  A.loss_kind = m->loss; A.training = training;
  cudaStream_t st = (cudaStream_t)stream;
  if (m->E == 10 && m->H1 == 100 && m->H2 == 50 && m->H3 == 10)    // script spec trainers/NFC_plain.py:109-152
    return m->act == 0 ? run_neumf<10, 100, 50, 10, 0>(ctx, A, st) : run_neumf<10, 100, 50, 10, 1>(ctx, A, st);
  // numFactor is a free attribute of the reference model (RModel.py:35): every other width runs on the any-width kernels
  return brk_neumf_step_generic(ctx, m, u, i, y, batch, global_batch, first_index, training, dropout_seed, dropout_epoch, ws, out,
                                y ? loss_out : nullptr, st);
}

// Row-sharded tables over NVLink peer memory (BASELINE.json configs[3]; SURVEY.md section 8e): the four
// tables' rows live on rank (row % world) at local row (row / world); `m` describes THIS rank's shards (for
// the optimizer), `sh` every rank's shard pointers.  The gathers read peer rows directly and the gradient
// scatter-adds are REDs into the owner's accumulator, so there is no separate exchange step.
extern "C" int brk_neumf_step_sharded(brk_ctx* ctx, const brk_neumf_model* m, const brk_neumf_shards* sh,
                                      const int32_t* u, const int32_t* i, const float* y, int64_t batch,
                                      int64_t global_batch, int64_t first_index, int32_t training, uint32_t dropout_seed,
                                      uint32_t dropout_epoch, const brk_neumf_workspace* ws, float* out, float* loss_out,
                                      void* stream) {
  BRK_REQUIRE(ctx && m && sh && u && i && ws && out, BRK_E_ARG, "brk_neumf_step_sharded: null argument");
  BRK_REQUIRE(y || !training, BRK_E_ARG, "brk_neumf_step_sharded: labels are required for training");
  BRK_REQUIRE(batch > 0, BRK_E_ARG, "brk_neumf_step_sharded: batch=%lld", (long long)batch);
  BRK_REQUIRE(m->dense.w && m->bn_moving && (!training || m->dense.g), BRK_E_ARG, "brk_neumf_step_sharded: dense block missing");
  BRK_REQUIRE(ws->h1 && ws->h2 && ws->dy1 && ws->dy2 && ws->acc, BRK_E_ARG, "brk_neumf_step_sharded: workspace missing");
  const brk_shards* all[4] = {&sh->uMLP, &sh->iMLP, &sh->uMF, &sh->iMF};
  for (int k = 0; k < 4; ++k) {
    BRK_REQUIRE(all[k]->world >= 1 && all[k]->world <= BRK_MAX_PEERS && all[k]->world == all[0]->world, BRK_E_ARG,
                "brk_neumf_step_sharded: world=%d (max %d, equal for all tables)", all[k]->world, BRK_MAX_PEERS);
    for (int p = 0; p < all[k]->world; ++p)
      BRK_REQUIRE(all[k]->w[p] && (!training || all[k]->g[p]) && brk_aligned16(all[k]->w[p]) && brk_aligned16(all[k]->g[p]),
                  BRK_E_ARG, "brk_neumf_step_sharded: shard %d of table %d missing or not 16-byte aligned", p, k);
  }
  int rc2 = 0;
  BRK_REQUIRE(!brk_neumf_is_variant(m), BRK_E_ARG, "brk_neumf_step_sharded: the reference class graph only");
  if (m->tensor_cores) {
    int handled = 0;
    brk_neumf_step_fused(ctx, m, sh, u, i, y, batch, global_batch, first_index, training, dropout_seed, dropout_epoch, ws, out,
                         loss_out, (cudaStream_t)stream, &rc2, &handled, nullptr, nullptr);
    if (handled) return rc2;
    if (brk_neumf_step_tc(ctx, m, sh, u, i, y, batch, global_batch, first_index, training, dropout_seed, dropout_epoch, ws,
                          out, loss_out, (cudaStream_t)stream, &rc2) == 0)
      return rc2;
    brk_set_error("brk_neumf_step_sharded: no tensor-core instance for E=%d H=(%d,%d,%d)", m->E, m->H1, m->H2, m->H3);
    return BRK_E_ARG;
  }
  if (brk_neumf_step_v2(ctx, m, sh, u, i, y, batch, global_batch, first_index, training, dropout_seed, dropout_epoch, ws,
                        out, loss_out, (cudaStream_t)stream, &rc2) == 0)
    return rc2;
  brk_set_error("brk_neumf_step_sharded: no sharded kernel instance for E=%d H=(%d,%d,%d); built: (32;32,16,8) "
                "(64;64,32,16) (16;16,8,4) (8;8,4,2)", m->E, m->H1, m->H2, m->H3);
  return BRK_E_ARG;
}
