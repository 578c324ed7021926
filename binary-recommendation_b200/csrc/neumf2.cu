// NeuMF forward/backward, second generation (see neumf.cu for the model, the phase split at the
// BatchNorm dependencies and the parameter layout -- both files implement the same five phases).
//
// What changed: the first version mapped one THREAD to one sample and left ~4 warps per SM with
// serial 64-deep FMA chains against broadcast weight loads.  Here a CTA of 128 threads owns a tile of
// 64 samples and every layer is a register-tiled block GEMM out of shared memory:
//   * every activation / gradient tile lives in shared memory feature-major  T[f][s]  (pitch 68), the
//     same orientation as the HBM intermediates, so loads and stores are coalesced float4 both ways;
//   * forward      Y[s][j]  = sum_k X[k][s] W[k][j]      outer-product form over k   (RM x RN per thread)
//   * weight grad  dW[k][j] = sum_s X[k][s] dZ[j][s]     inner-product form, float4 along the samples
//   * input grad   dX[s][k] = sum_j dZs[s][j] W[k][j]    inner-product form, float4 along j -- the Keras
//     [in][out] weight layout serves all three products, no transposed weight copy;
//   * thread-per-sample work only where it is natural: row gathers, Philox dropout masks, loss.
// Supported specs: 2E, H1, H2, H3 powers of two (E >= 8, H3 >= 2); anything else takes neumf.cu.
#include "neumf_common.cuh"

namespace v2 {

constexpr int TS = 64;                // samples per CTA
constexpr int PT = TS + 4;            // tile pitch (floats): keeps float4 alignment, staggers banks
constexpr int NT = 128;               // threads per CTA
// per-thread tile shape for a [TS x OUT] output on NT threads: RM x RN = OUT / 2 elements
template <int OUT> struct Tile {
  static constexpr int RN = OUT >= 64 ? 8 : OUT >= 16 ? 4 : OUT >= 8 ? 2 : OUT >= 4 ? 2 : 1;
  static constexpr int RM = (OUT / 2) / RN;
  static_assert(RM * RN * 2 == OUT && (TS / RM) * (OUT / RN) == NT, "tile shape");
};

template <int N> __device__ __forceinline__ void ldv(const float* p, float (&v)[N]) {
  if constexpr (N == 8) {
    const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else if constexpr (N == 4) {
    const float4 a = *reinterpret_cast<const float4*>(p);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
  } else if constexpr (N == 2) {
    const float2 a = *reinterpret_cast<const float2*>(p);
    v[0] = a.x; v[1] = a.y;
  } else {
    v[0] = p[0];
  }
}

// acc[i][j] += sum_k A[k][m0+i] * Bw[k][n0+j]        A: [K][PT] tile, Bw: [K][ldb] weights
template <int K, int RM, int RN>
__device__ __forceinline__ void gemm_outer(const float* A, const float* Bw, int ldb, int m0, int n0, float (&acc)[RM][RN]) {
#pragma unroll 4
  for (int k = 0; k < K; ++k) {
    float a[RM], b[RN];
    ldv<RM>(A + k * PT + m0, a);
    ldv<RN>(Bw + k * ldb + n0, b);
#pragma unroll
    for (int i = 0; i < RM; ++i)
#pragma unroll
      for (int j = 0; j < RN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
  }
}
// acc[i][j] = sum_r A[(m0+i)*lda + r] * Bm[(n0+j)*ldb + r], r in [0,R), float4 along r
template <int R, int RM, int RN>
__device__ __forceinline__ void gemm_inner(const float* A, int lda, const float* Bm, int ldb, int m0, int n0,
                                           float (&acc)[RM][RN]) {
#pragma unroll
  for (int i = 0; i < RM; ++i)
#pragma unroll
    for (int j = 0; j < RN; ++j) acc[i][j] = 0.f;
#pragma unroll 2
  for (int r = 0; r < R; r += 4) {
    float4 a[RM], b[RN];
#pragma unroll
    for (int i = 0; i < RM; ++i) a[i] = *reinterpret_cast<const float4*>(A + (m0 + i) * lda + r);
#pragma unroll
    for (int j = 0; j < RN; ++j) b[j] = *reinterpret_cast<const float4*>(Bm + (n0 + j) * ldb + r);
#pragma unroll
    for (int i = 0; i < RM; ++i)
#pragma unroll
      for (int j = 0; j < RN; ++j) {
        acc[i][j] = fmaf(a[i].x, b[j].x, acc[i][j]); acc[i][j] = fmaf(a[i].y, b[j].y, acc[i][j]);
        acc[i][j] = fmaf(a[i].z, b[j].z, acc[i][j]); acc[i][j] = fmaf(a[i].w, b[j].w, acc[i][j]);
      }
  }
}

// Dropout in place on column s of a feature-major tile (thread-per-sample).
template <int N>
__device__ __forceinline__ void drop_col(float* T, int s, uint64_t idx, int layer, uint32_t seed, uint32_t epoch) {
#pragma unroll 1
  for (int c = 0; c < (N + 15) / 16; ++c) {
    float m[16];
    drop16(idx, c, layer, seed, epoch, m);
#pragma unroll
    for (int j = 0; j < 16; ++j) if (c * 16 + j < N) T[(c * 16 + j) * PT + s] *= m[j];
  }
}

// Thread-per-row gather of embedding rows into a feature-major tile: thread (s = t % TS) reads its row as
// float4 and writes T[col0 + 4c + q][s]; lanes hold consecutive samples -> conflict-free stores.
template <int E>
__device__ __forceinline__ void gather_col(float* T, int col0, const float* __restrict__ rowp, int s, bool valid) {
#pragma unroll 4
  for (int c = 0; c < E / 4; ++c) {
    const float4 v = valid ? __ldg(reinterpret_cast<const float4*>(rowp) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    T[(col0 + 4 * c + 0) * PT + s] = v.x; T[(col0 + 4 * c + 1) * PT + s] = v.y;
    T[(col0 + 4 * c + 2) * PT + s] = v.z; T[(col0 + 4 * c + 3) * PT + s] = v.w;
  }
}

template <int N>
__device__ __forceinline__ void copy_to_smem(float* dst, const float* __restrict__ src) {
  const bool al = (reinterpret_cast<uintptr_t>(src) & 15) == 0;      // parameter offsets need not be 16-byte aligned
  for (int i = threadIdx.x * 4; i < N; i += NT * 4) {
    if (al && i + 3 < N) *reinterpret_cast<float4*>(dst + i) = __ldg(reinterpret_cast<const float4*>(src + i));
    else for (int q = i; q < N && q < i + 4; ++q) dst[q] = __ldg(src + q);
  }
}

// Load a feature-major [H][TS] tile of an HBM intermediate (rows of B samples) into shared memory.
template <int H>
__device__ __forceinline__ void load_tile(float* T, const float* __restrict__ src, int64_t B, int64_t b0, int valid) {
  for (int idx = threadIdx.x; idx < H * (TS / 4); idx += NT) {
    const int f = idx / (TS / 4), s4 = (idx % (TS / 4)) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    const float* p = src + int64_t(f) * B + b0 + s4;
    if (s4 + 3 < valid && ((reinterpret_cast<uintptr_t>(p) & 15) == 0)) v = __ldg(reinterpret_cast<const float4*>(p));
    else {
      if (s4 + 0 < valid) v.x = __ldg(p + 0);
      if (s4 + 1 < valid) v.y = __ldg(p + 1);
      if (s4 + 2 < valid) v.z = __ldg(p + 2);
      if (s4 + 3 < valid) v.w = __ldg(p + 3);
    }
    *reinterpret_cast<float4*>(T + f * PT + s4) = v;
  }
}
template <int H>
__device__ __forceinline__ void store_tile(const float* T, float* __restrict__ dst, int64_t B, int64_t b0, int valid) {
  for (int idx = threadIdx.x; idx < H * (TS / 4); idx += NT) {
    const int f = idx / (TS / 4), s4 = (idx % (TS / 4)) * 4;
    const float4 v = *reinterpret_cast<const float4*>(T + f * PT + s4);
    float* p = dst + int64_t(f) * B + b0 + s4;
    if (s4 + 3 < valid && ((reinterpret_cast<uintptr_t>(p) & 15) == 0)) *reinterpret_cast<float4*>(p) = v;
    else {
      if (s4 + 0 < valid) p[0] = v.x;
      if (s4 + 1 < valid) p[1] = v.y;
      if (s4 + 2 < valid) p[2] = v.z;
      if (s4 + 3 < valid) p[3] = v.w;
    }
  }
}

// Per-feature sums over the tile's samples (double), one atomic pair per feature per CTA.
template <int H>
__device__ __forceinline__ void row_sums(const float* A, const float* Bm, double* sumA, double* sumAB) {
  for (int f = threadIdx.x; f < H; f += NT) {
    double s = 0.0, q = 0.0;
    for (int r = 0; r < TS; r += 4) {
      const float4 a = *reinterpret_cast<const float4*>(A + f * PT + r);
      const float4 b = Bm ? *reinterpret_cast<const float4*>(Bm + f * PT + r) : a;
      s += double(a.x) + double(a.y) + double(a.z) + double(a.w);
      q += double(a.x) * double(b.x) + double(a.y) * double(b.y) + double(a.z) * double(b.z) + double(a.w) * double(b.w);
    }
    atomicAdd(sumA + f, s);
    atomicAdd(sumAB + f, q);
  }
}
template <int H>
__device__ __forceinline__ void bn_prepare(float* mean, float* rstd, const double* sum, const double* sq,
                                           const float* mov_mean, const float* mov_var, int64_t B, bool training) {
  for (int f = threadIdx.x; f < H; f += NT) {
    float mu, var;
    if (training) {
      const double m = sum[f] / double(B);
      mu = float(m); var = float(fmax(sq[f] / double(B) - m * m, 0.0));
    } else { mu = mov_mean[f]; var = mov_var[f]; }
    mean[f] = mu; rstd[f] = 1.0f / sqrtf(var + kBnEps);
  }
}

// Y tile = act(X W + b) for one layer: X [IN][PT] in smem, W [IN][OUT] in smem, result to Ys [OUT][PT].
template <int IN, int OUT, int ACT>
__device__ __forceinline__ void layer_fwd(const float* Xs, const float* Ws, int ldb, const float* bs, float* Ys, int valid) {
  using T = Tile<OUT>;
  constexpr int NG = OUT / T::RN;
  const int ng = threadIdx.x % NG, mg = threadIdx.x / NG;
  const int m0 = mg * T::RM, n0 = ng * T::RN;
  float acc[T::RM][T::RN];
#pragma unroll
  for (int i = 0; i < T::RM; ++i)
#pragma unroll
    for (int j = 0; j < T::RN; ++j) acc[i][j] = bs[n0 + j];
  gemm_outer<IN, T::RM, T::RN>(Xs, Ws, ldb, m0, n0, acc);
#pragma unroll
  for (int j = 0; j < T::RN; ++j)
#pragma unroll
    for (int i = 0; i < T::RM; ++i) Ys[(n0 + j) * PT + m0 + i] = (m0 + i < valid) ? act_f<ACT>(acc[i][j]) : 0.f;
}

// dW[k][j] += sum_s X[k][s] dZ[j][s]; db[j] += sum_s dZ[j][s]   (X: [IN][PT], dZ: [OUT][PT])
template <int IN, int OUT>
__device__ __forceinline__ void layer_wgrad(const float* Xs, const float* dZs, float* __restrict__ gW, float* __restrict__ gb) {
  constexpr int RM = IN >= 4 ? 4 : IN, RN = OUT >= 4 ? 4 : OUT;
  constexpr int TJ = OUT / RN, NTILES = (IN / RM) * TJ;
  for (int t = threadIdx.x; t < NTILES; t += NT) {
    const int k0 = (t / TJ) * RM, j0 = (t % TJ) * RN;
    float acc[RM][RN];
    gemm_inner<TS, RM, RN>(Xs, PT, dZs, PT, k0, j0, acc);
#pragma unroll
    for (int i = 0; i < RM; ++i)
#pragma unroll
      for (int j = 0; j < RN; ++j) atomicAdd(gW + (k0 + i) * OUT + j0 + j, acc[i][j]);
  }
  for (int j = threadIdx.x; j < OUT; j += NT) {
    float s = 0.f;
    for (int r = 0; r < TS; r += 4) {
      const float4 a = *reinterpret_cast<const float4*>(dZs + j * PT + r);
      s += (a.x + a.y) + (a.z + a.w);
    }
    atomicAdd(gb + j, s);
  }
}

template <int OUT> __host__ __device__ constexpr int zpitch() { return (OUT >= 4 ? OUT : 4) + 4; }   // sample-major dz pitch

// dX[k][s] = sum_j dZt[s][j] W[k][j]   (dZt: sample-major [TS][zpitch], W: [IN][OUT]) -> DX [IN][PT]
template <int IN, int OUT>
__device__ __forceinline__ void layer_dgrad(const float* dZt, const float* Ws, float* DX) {
  constexpr int ZP = zpitch<OUT>();
  constexpr int RM = 4, RN = IN >= 4 ? 4 : IN;                      // 4 samples x 4 inputs per tile
  constexpr int TK = IN / RN, NTILES = (TS / RM) * TK;
  constexpr int R = OUT >= 4 ? OUT : 4;                              // OUT == 2: rows padded with zeros to 4
  for (int t = threadIdx.x; t < NTILES; t += NT) {
    const int s0 = (t / TK) * RM, k0 = (t % TK) * RN;
    float acc[RM][RN];
    gemm_inner<R, RM, RN>(dZt, ZP, Ws, OUT >= 4 ? OUT : 4, s0, k0, acc);
#pragma unroll
    for (int j = 0; j < RN; ++j)
#pragma unroll
      for (int i = 0; i < RM; ++i) DX[(k0 + j) * PT + s0 + i] = acc[i][j];
  }
}

extern __shared__ __align__(16) float sm[];

// weights of an [IN][OUT] layer into smem; when OUT < 4 rows are padded to 4 floats (for the float4 dgrad)
template <int IN, int OUT>
__device__ __forceinline__ void stage_w(float* dst, const float* __restrict__ src) {
  if constexpr (OUT >= 4) copy_to_smem<IN * OUT>(dst, src);
  else for (int i = threadIdx.x; i < IN * 4; i += NT) dst[i] = (i % 4) < OUT ? __ldg(src + (i / 4) * OUT + (i % 4)) : 0.f;
}
template <int OUT> constexpr int wld() { return OUT >= 4 ? OUT : 4; }

// ------------------------------------------------------------------------------------------------
template <int E, int H1, int H2, int H3, int ACT>
__global__ void __launch_bounds__(NT) fwd1(const Args A) {
  using L = Layout<E, H1, H2, H3>; using AC = Acc<H1, H2>;
  float* Xs = sm;                          // [2E][PT]
  float* Ws = Xs + 2 * E * PT;             // [2E][H1]
  float* bs = Ws + 2 * E * H1;             // [H1]
  float* Ys = bs + H1;                     // [H1][PT]
  const int64_t b0 = int64_t(blockIdx.x) * TS;
  const int valid = int((A.B - b0) < int64_t(TS) ? (A.B - b0) : int64_t(TS));
  const int t = threadIdx.x, s = t % TS;
  copy_to_smem<2 * E * H1>(Ws, A.dense.w + L::W1);
  copy_to_smem<H1>(bs, A.dense.w + L::b1);
  const bool ok = s < valid;
  if (t < TS) gather_col<E>(Xs, 0, locate<E>(A.uMLP, ok ? int64_t(__ldg(A.u + b0 + s)) : 0).w, s, ok);
  else        gather_col<E>(Xs, E, locate<E>(A.iMLP, ok ? int64_t(__ldg(A.i + b0 + s)) : 0).w, s, ok);
  __syncthreads();
  if (A.dropout && t < TS && ok) drop_col<2 * E>(Xs, s, uint64_t(A.first_index + b0 + s), 0, A.drop_seed, A.drop_epoch);
  if (A.dropout) __syncthreads();
  layer_fwd<2 * E, H1, ACT>(Xs, Ws, H1, bs, Ys, valid);
  __syncthreads();
  store_tile<H1>(Ys, A.h1, A.B, b0, valid);
  if (A.training) row_sums<H1>(Ys, nullptr, A.acc + AC::s1, A.acc + AC::q1);
}

template <int E, int H1, int H2, int H3, int ACT>
__global__ void __launch_bounds__(NT) fwd2(const Args A) {
  using L = Layout<E, H1, H2, H3>; using AC = Acc<H1, H2>;
  float* Xs = sm;                          // [H1][PT]
  float* Ws = Xs + H1 * PT;                // [H1][H2]
  float* bs = Ws + H1 * H2;                // [H2]
  float* Ys = bs + H2;                     // [H2][PT]
  float* mean = Ys + H2 * PT; float* rstd = mean + H1; float* gam = rstd + H1; float* bet = gam + H1;
  const int64_t b0 = int64_t(blockIdx.x) * TS;
  const int valid = int((A.B - b0) < int64_t(TS) ? (A.B - b0) : int64_t(TS));
  const int t = threadIdx.x;
  copy_to_smem<H1 * H2>(Ws, A.dense.w + L::W2);
  copy_to_smem<H2>(bs, A.dense.w + L::b2);
  copy_to_smem<H1>(gam, A.dense.w + L::g1);
  copy_to_smem<H1>(bet, A.dense.w + L::be1);
  bn_prepare<H1>(mean, rstd, A.acc + AC::s1, A.acc + AC::q1, A.bn_moving, A.bn_moving + H1, A.B, A.training);
  load_tile<H1>(Xs, A.h1, A.B, b0, valid);
  __syncthreads();
  for (int idx = t; idx < H1 * TS; idx += NT) {
    const int f = idx / TS, s = idx % TS;
    Xs[f * PT + s] = s < valid ? gam[f] * (Xs[f * PT + s] - mean[f]) * rstd[f] + bet[f] : 0.f;
  }
  __syncthreads();
  if (A.dropout && t < valid) drop_col<H1>(Xs, t, uint64_t(A.first_index + b0 + t), 1, A.drop_seed, A.drop_epoch);
  if (A.dropout) __syncthreads();
  layer_fwd<H1, H2, ACT>(Xs, Ws, H2, bs, Ys, valid);
  __syncthreads();
  store_tile<H2>(Ys, A.h2, A.B, b0, valid);
  if (A.training) row_sums<H2>(Ys, nullptr, A.acc + AC::s2, A.acc + AC::q2);
}

template <int E, int H1, int H2, int H3, int ACT>
__global__ void __launch_bounds__(NT) head(const Args A) {
  using L = Layout<E, H1, H2, H3>; using AC = Acc<H1, H2>;
  constexpr int ZP = zpitch<H3>();
  float* Xs = sm;                          // [H2][PT]  d2 = dropout(bn2(h2)); later dy2
  float* Xh = Xs + H2 * PT;                // [H2][PT]  xhat2
  float* Ws = Xh + H2 * PT;                // [H2][wld(H3)]
  float* bs = Ws + H2 * wld<H3>();         // [H3]
  float* w4 = bs + ((H3 + 3) & ~3);        // [H3 + 2]
  float* Ys = w4 + ((H3 + 2 + 3) & ~3);    // [H3][PT]   h3, later dz3 (feature-major)
  float* Zt = Ys + H3 * PT;                // [TS][ZP]   dz3 sample-major
  float* dl = Zt + TS * ZP;                // [TS] dlogit, then [TS] mf
  float* mfs = dl + TS;
  float* mean = mfs + TS; float* rstd = mean + H2; float* gam = rstd + H2; float* bet = gam + H2;
  __shared__ double red[32];
  const int64_t b0 = int64_t(blockIdx.x) * TS;
  const int valid = int((A.B - b0) < int64_t(TS) ? (A.B - b0) : int64_t(TS));
  const int t = threadIdx.x;
  stage_w<H2, H3>(Ws, A.dense.w + L::W3);
  copy_to_smem<H3>(bs, A.dense.w + L::b3);
  copy_to_smem<H3 + 2>(w4, A.dense.w + L::W4);
  copy_to_smem<H2>(gam, A.dense.w + L::g2);
  copy_to_smem<H2>(bet, A.dense.w + L::be2);
  bn_prepare<H2>(mean, rstd, A.acc + AC::s2, A.acc + AC::q2, A.bn_moving + 2 * H1, A.bn_moving + 2 * H1 + H2, A.B, A.training);
  load_tile<H2>(Xs, A.h2, A.B, b0, valid);
  // MF dot product: thread-per-sample straight from the tables (threads TS..2TS-1; rows stay in L1 for the backward)
  RowRef ru, ri;
  ru.w = ri.w = nullptr; ru.g = ri.g = nullptr; ru.t = ri.t = nullptr; ru.lrow = ri.lrow = 0;
  if (t >= TS && t - TS < valid) {
    ru = locate<E>(A.uMF, __ldg(A.u + b0 + t - TS)); ri = locate<E>(A.iMF, __ldg(A.i + b0 + t - TS));
    float mf = 0.f;
#pragma unroll 4
    for (int c = 0; c < E / 4; ++c) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(ru.w) + c);
      const float4 b = __ldg(reinterpret_cast<const float4*>(ri.w) + c);
      mf = fmaf(a.x, b.x, mf); mf = fmaf(a.y, b.y, mf); mf = fmaf(a.z, b.z, mf); mf = fmaf(a.w, b.w, mf);
    }
    mfs[t - TS] = mf;
  }
  __syncthreads();
  for (int idx = t; idx < H2 * TS; idx += NT) {
    const int f = idx / TS, s = idx % TS;
    const float xh = s < valid ? (Xs[f * PT + s] - mean[f]) * rstd[f] : 0.f;
    Xh[f * PT + s] = xh;
    Xs[f * PT + s] = s < valid ? gam[f] * xh + bet[f] : 0.f;
  }
  __syncthreads();
  if (A.dropout && t < valid) drop_col<H2>(Xs, t, uint64_t(A.first_index + b0 + t), 2, A.drop_seed, A.drop_epoch);
  if (A.dropout) __syncthreads();
  layer_fwd<H2, H3, ACT>(Xs, Ws, wld<H3>(), bs, Ys, valid);
  __syncthreads();
  // logit, prediction, loss, dlogit: threads TS..2TS-1 (they hold the MF rows' ids)
  float loss_local = 0.f;
  if (t >= TS) {
    const int s = t - TS;
    float dlogit = 0.f;
    if (s < valid) {
      float logit = w4[H3 + 1];
#pragma unroll
      for (int j = 0; j < H3; ++j) logit = fmaf(Ys[j * PT + s], w4[j], logit);
      logit = fmaf(mfs[s], w4[H3], logit);
      const float o = 1.0f / (1.0f + expf(-logit));
      A.out[b0 + s] = o;
      const float yv = __ldg(A.y + b0 + s);
      const float invB = 1.0f / float(A.global_B);
      if (A.loss_kind == 0) { const float e = o - yv; loss_local = e * e; dlogit = 2.f * e * o * (1.f - o) * invB; }
      else { loss_local = fmaxf(logit, 0.f) - logit * yv + log1pf(expf(-fabsf(logit))); dlogit = (o - yv) * invB; }
    }
    dl[s] = dlogit;
  }
  const double lsum = block_sum_double(double(loss_local), red);
  if (t == 0) atomicAdd(A.acc + AC::loss, lsum);
  if (!A.training) return;
  __syncthreads();
  // head weight gradients: dW4[j] = sum_s z[j][s] dl[s] (z = [h3, mf]), db4 = sum_s dl[s]
  for (int j = t; j < H3 + 2; j += NT) {
    float sacc = 0.f;
    for (int s = 0; s < TS; ++s) sacc = fmaf(j < H3 ? Ys[j * PT + s] : (j == H3 ? mfs[s] : 1.f), dl[s], sacc);
    atomicAdd(A.dense.g + L::W4 + j, sacc);
  }
  __syncthreads();
  // dz3 = dl * w4[j] * act'(h3) in both orientations
  for (int idx = t; idx < H3 * TS; idx += NT) {
    const int j = idx / TS, s = idx % TS;
    const float dz = dl[s] * w4[j] * act_grad<ACT>(Ys[j * PT + s]);
    Ys[j * PT + s] = dz;
    Zt[s * ZP + j] = dz;
  }
  if constexpr (H3 < 4) {
    constexpr int PADC = 4 - H3;
    for (int idx = t; idx < TS * PADC; idx += NT) Zt[(idx / PADC) * ZP + H3 + idx % PADC] = 0.f;
  }
  __syncthreads();
  layer_wgrad<H2, H3>(Xs, Ys, A.dense.g + L::W3, A.dense.g + L::b3);
  // MF embedding gradients (thread-per-sample, rows re-read through L1)
  if (t >= TS && t - TS < valid) {
    const float dmf = dl[t - TS] * w4[H3];
    float* gu = ru.g; float* gi = ri.g;
#pragma unroll 4
    for (int c = 0; c < E / 4; ++c) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(ru.w) + c);
      const float4 b = __ldg(reinterpret_cast<const float4*>(ri.w) + c);
      red_add_f4(gu + 4 * c, make_float4(dmf * b.x, dmf * b.y, dmf * b.z, dmf * b.w));
      red_add_f4(gi + 4 * c, make_float4(dmf * a.x, dmf * a.y, dmf * a.z, dmf * a.w));
    }
    mark_row(ru); mark_row(ri);
  }
  __syncthreads();                                          // wgrad has consumed Xs
  layer_dgrad<H2, H3>(Zt, Ws, Xs);                          // Xs <- dd2 [H2][PT]
  __syncthreads();
  if (A.dropout && t < valid) drop_col<H2>(Xs, t, uint64_t(A.first_index + b0 + t), 2, A.drop_seed, A.drop_epoch);
  __syncthreads();
  store_tile<H2>(Xs, A.dy2, A.B, b0, valid);
  row_sums<H2>(Xs, Xh, A.acc + AC::d2, A.acc + AC::e2);
}

// Shared body of the two BN-backward phases: given the layer's input tile Xs (post-BN, post-dropout),
// its output h (HBM), the gradient dy w.r.t. the following BN output (HBM) and that BN's statistics,
// build dz in both orientations.
template <int H, int ACT>
__device__ __forceinline__ void bn_backward_dz(float* Zf, float* Zt, const float* __restrict__ h, const float* __restrict__ dy,
                                               const float* mean, const float* rstd, const float* gam, const float* sdy,
                                               const float* sdyx, int64_t B, int64_t b0, int valid) {
  constexpr int ZP = zpitch<H>();
  for (int idx = threadIdx.x; idx < H * TS; idx += NT) {
    const int j = idx / TS, s = idx % TS;
    float dz = 0.f;
    if (s < valid) {
      const float hv = __ldg(h + int64_t(j) * B + b0 + s);
      const float xh = (hv - mean[j]) * rstd[j];
      const float dh = gam[j] * rstd[j] * (__ldg(dy + int64_t(j) * B + b0 + s) - sdy[j] - xh * sdyx[j]);
      dz = dh * act_grad<ACT>(hv);
    }
    Zf[j * PT + s] = dz;
    Zt[s * ZP + j] = dz;
  }
}

template <int E, int H1, int H2, int H3, int ACT>
__global__ void __launch_bounds__(NT) bwd2(const Args A) {
  using L = Layout<E, H1, H2, H3>; using AC = Acc<H1, H2>;
  constexpr int ZP = zpitch<H2>();
  float* Xs = sm;                          // [H1][PT]  d1, later dy1
  float* Xh = Xs + H1 * PT;                // [H1][PT]  xhat1
  float* Ws = Xh + H1 * PT;                // [H1][H2]
  float* Zf = Ws + H1 * H2;                // [H2][PT]
  float* Zt = Zf + H2 * PT;                // [TS][ZP]
  float* mean1 = Zt + TS * ZP; float* rstd1 = mean1 + H1; float* gam1 = rstd1 + H1; float* bet1 = gam1 + H1;
  float* mean2 = bet1 + H1; float* rstd2 = mean2 + H2; float* gam2 = rstd2 + H2; float* sdy = gam2 + H2; float* sdyx = sdy + H2;
  const int64_t b0 = int64_t(blockIdx.x) * TS;
  const int valid = int((A.B - b0) < int64_t(TS) ? (A.B - b0) : int64_t(TS));
  const int t = threadIdx.x;
  copy_to_smem<H1 * H2>(Ws, A.dense.w + L::W2);
  copy_to_smem<H1>(gam1, A.dense.w + L::g1);
  copy_to_smem<H1>(bet1, A.dense.w + L::be1);
  copy_to_smem<H2>(gam2, A.dense.w + L::g2);
  bn_prepare<H1>(mean1, rstd1, A.acc + AC::s1, A.acc + AC::q1, nullptr, nullptr, A.B, true);
  bn_prepare<H2>(mean2, rstd2, A.acc + AC::s2, A.acc + AC::q2, nullptr, nullptr, A.B, true);
  for (int f = t; f < H2; f += NT) {
    sdy[f] = float(A.acc[AC::d2 + f] / double(A.B));
    sdyx[f] = float(A.acc[AC::e2 + f] / double(A.B));
    if (blockIdx.x == 0) {                                  // BN2 parameter gradients
      A.dense.g[L::be2 + f] += float(A.acc[AC::d2 + f]);
      A.dense.g[L::g2 + f] += float(A.acc[AC::e2 + f]);
    }
  }
  load_tile<H1>(Xs, A.h1, A.B, b0, valid);
  __syncthreads();
  for (int idx = t; idx < H1 * TS; idx += NT) {
    const int f = idx / TS, s = idx % TS;
    const float xh = s < valid ? (Xs[f * PT + s] - mean1[f]) * rstd1[f] : 0.f;
    Xh[f * PT + s] = xh;
    Xs[f * PT + s] = s < valid ? gam1[f] * xh + bet1[f] : 0.f;
  }
  bn_backward_dz<H2, ACT>(Zf, Zt, A.h2, A.dy2, mean2, rstd2, gam2, sdy, sdyx, A.B, b0, valid);
  __syncthreads();
  if (A.dropout && t < valid) drop_col<H1>(Xs, t, uint64_t(A.first_index + b0 + t), 1, A.drop_seed, A.drop_epoch);
  if (A.dropout) __syncthreads();
  layer_wgrad<H1, H2>(Xs, Zf, A.dense.g + L::W2, A.dense.g + L::b2);
  __syncthreads();
  layer_dgrad<H1, H2>(Zt, Ws, Xs);                          // Xs <- dd1
  __syncthreads();
  if (A.dropout && t < valid) drop_col<H1>(Xs, t, uint64_t(A.first_index + b0 + t), 1, A.drop_seed, A.drop_epoch);
  __syncthreads();
  store_tile<H1>(Xs, A.dy1, A.B, b0, valid);
  row_sums<H1>(Xs, Xh, A.acc + AC::d1, A.acc + AC::e1);
}

template <int E, int H1, int H2, int H3, int ACT>
__global__ void __launch_bounds__(NT) bwd1(const Args A, unsigned int* ticket) {
  using L = Layout<E, H1, H2, H3>; using AC = Acc<H1, H2>;
  constexpr int ZP = zpitch<H1>();
  float* Xs = sm;                          // [2E][PT]  d0, later dx0
  float* Ws = Xs + 2 * E * PT;             // [2E][H1]
  float* Zf = Ws + 2 * E * H1;             // [H1][PT]
  float* Zt = Zf + H1 * PT;                // [TS][ZP]
  float* mean1 = Zt + TS * ZP; float* rstd1 = mean1 + H1; float* gam1 = rstd1 + H1; float* sdy = gam1 + H1; float* sdyx = sdy + H1;
  const int64_t b0 = int64_t(blockIdx.x) * TS;
  const int valid = int((A.B - b0) < int64_t(TS) ? (A.B - b0) : int64_t(TS));
  const int t = threadIdx.x, s = t % TS;
  copy_to_smem<2 * E * H1>(Ws, A.dense.w + L::W1);
  copy_to_smem<H1>(gam1, A.dense.w + L::g1);
  bn_prepare<H1>(mean1, rstd1, A.acc + AC::s1, A.acc + AC::q1, nullptr, nullptr, A.B, true);
  for (int f = t; f < H1; f += NT) {
    sdy[f] = float(A.acc[AC::d1 + f] / double(A.B));
    sdyx[f] = float(A.acc[AC::e1 + f] / double(A.B));
    if (blockIdx.x == 0) {
      A.dense.g[L::be1 + f] += float(A.acc[AC::d1 + f]);
      A.dense.g[L::g1 + f] += float(A.acc[AC::e1 + f]);
    }
  }
  const bool ok = s < valid;
  const RowRef rr = locate<E>(t < TS ? A.uMLP : A.iMLP, ok ? int64_t(__ldg((t < TS ? A.u : A.i) + b0 + s)) : 0);
  gather_col<E>(Xs, t < TS ? 0 : E, rr.w, s, ok);
  __syncthreads();
  bn_backward_dz<H1, ACT>(Zf, Zt, A.h1, A.dy1, mean1, rstd1, gam1, sdy, sdyx, A.B, b0, valid);
  if (A.dropout && t < TS && ok) drop_col<2 * E>(Xs, s, uint64_t(A.first_index + b0 + s), 0, A.drop_seed, A.drop_epoch);
  __syncthreads();
  layer_wgrad<2 * E, H1>(Xs, Zf, A.dense.g + L::W1, A.dense.g + L::b1);
  __syncthreads();
  layer_dgrad<2 * E, H1>(Zt, Ws, Xs);                        // Xs <- dx0 [2E][PT]
  __syncthreads();
  if (A.dropout && t < TS && ok) drop_col<2 * E>(Xs, s, uint64_t(A.first_index + b0 + s), 0, A.drop_seed, A.drop_epoch);
  __syncthreads();
  // MLP embedding gradients: threads 0..63 scatter the user half, 64..127 the item half (16-byte REDs)
  if (ok) {
    float* g = rr.g;
    const int c0 = t < TS ? 0 : E;
#pragma unroll 4
    for (int c = 0; c < E; c += 4)
      red_add_f4(g + c, make_float4(Xs[(c0 + c) * PT + s], Xs[(c0 + c + 1) * PT + s], Xs[(c0 + c + 2) * PT + s],
                                    Xs[(c0 + c + 3) * PT + s]));
    mark_row(rr);
  }
  // last CTA: BN moving statistics, loss output, accumulator reset
  __syncthreads();
  __shared__ bool last;
  if (t == 0) { __threadfence(); last = atomicAdd(ticket, 1u) == gridDim.x - 1; }
  __syncthreads();
  if (last) {
    __threadfence();
    for (int f = t; f < H1; f += NT) {
      const double m = A.acc[AC::s1 + f] / double(A.B);
      const double v = fmax(A.acc[AC::q1 + f] / double(A.B) - m * m, 0.0);
      A.bn_moving[f] = A.bn_moving[f] * kBnMomentum + float(m) * (1.f - kBnMomentum);
      A.bn_moving[H1 + f] = A.bn_moving[H1 + f] * kBnMomentum + float(v) * (1.f - kBnMomentum);
    }
    for (int f = t; f < H2; f += NT) {
      const double m = A.acc[AC::s2 + f] / double(A.B);
      const double v = fmax(A.acc[AC::q2 + f] / double(A.B) - m * m, 0.0);
      A.bn_moving[2 * H1 + f] = A.bn_moving[2 * H1 + f] * kBnMomentum + float(m) * (1.f - kBnMomentum);
      A.bn_moving[2 * H1 + H2 + f] = A.bn_moving[2 * H1 + H2 + f] * kBnMomentum + float(v) * (1.f - kBnMomentum);
    }
    if (t == 0 && A.loss_out) A.loss_out[0] = float(A.acc[AC::loss] / double(A.B));
    __syncthreads();
    for (int j = t; j < AC::total; j += NT) A.acc[j] = 0.0;
    if (t == 0) *ticket = 0u;
  }
}

template <int H1, int H2>
__global__ void finish_eval(double* acc, int64_t B, float* loss_out) {
  using AC = Acc<H1, H2>;
  if (threadIdx.x == 0 && loss_out) loss_out[0] = float(acc[AC::loss] / double(B));
  __syncthreads();
  for (int j = threadIdx.x; j < AC::total; j += blockDim.x) acc[j] = 0.0;
}

template <int E, int H1, int H2, int H3, int ACT>
int run(brk_ctx* ctx, const Args& A, cudaStream_t st) {
  const int grid = int((A.B + TS - 1) / TS);
  auto by = [](size_t floats) { return floats * sizeof(float); };
  const size_t smA = by(size_t(2 * E) * PT + 2 * E * H1 + H1 + size_t(H1) * PT);
  const size_t smB = by(size_t(H1) * PT + H1 * H2 + H2 + size_t(H2) * PT + 4 * H1);
  const size_t smC = by(size_t(2 * H2) * PT + H2 * wld<H3>() + ((H3 + 3) & ~3) + ((H3 + 5) & ~3) + size_t(H3) * PT +
                        size_t(TS) * v2::zpitch<H3>() + 2 * TS + 4 * H2);
  const size_t smD = by(size_t(2 * H1) * PT + H1 * H2 + size_t(H2) * PT + size_t(TS) * v2::zpitch<H2>() + 4 * H1 + 5 * H2);
  const size_t smE = by(size_t(2 * E) * PT + 2 * E * H1 + size_t(H1) * PT + size_t(TS) * v2::zpitch<H1>() + 5 * H1);
  // the shared-memory opt-in is per device: set it for the current one on every call
  BRK_CUDA(cudaFuncSetAttribute(fwd1<E, H1, H2, H3, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smA)));
  BRK_CUDA(cudaFuncSetAttribute(fwd2<E, H1, H2, H3, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smB)));
  BRK_CUDA(cudaFuncSetAttribute(head<E, H1, H2, H3, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smC)));
  BRK_CUDA(cudaFuncSetAttribute(bwd2<E, H1, H2, H3, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smD)));
  BRK_CUDA(cudaFuncSetAttribute(bwd1<E, H1, H2, H3, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smE)));
  fwd1<E, H1, H2, H3, ACT><<<grid, NT, smA, st>>>(A);
  fwd2<E, H1, H2, H3, ACT><<<grid, NT, smB, st>>>(A);
  head<E, H1, H2, H3, ACT><<<grid, NT, smC, st>>>(A);
  if (A.training) {
    bwd2<E, H1, H2, H3, ACT><<<grid, NT, smD, st>>>(A);
    bwd1<E, H1, H2, H3, ACT><<<grid, NT, smE, st>>>(A, ctx->tickets + 4);
  } else {
    finish_eval<H1, H2><<<1, 128, 0, st>>>(A.acc, A.B, A.loss_out);
  }
  BRK_LAUNCH_CHECK();
  return 0;
}

}  // namespace v2

// Returns 0 when the spec was handled, 1 when it is not a v2 spec (caller falls through to neumf.cu).
static void tab_ref(v2::TabRef& T, const brk_table& local, const brk_shards* sh) {
  for (int p = 0; p < BRK_MAX_PEERS; ++p) { T.w[p] = nullptr; T.g[p] = nullptr; T.t[p] = nullptr; }
  if (sh && sh->world > 1) {
    T.world = sh->world;
    for (int p = 0; p < sh->world; ++p) { T.w[p] = sh->w[p]; T.g[p] = sh->g[p]; T.t[p] = sh->touched[p]; }
  } else {
    T.world = 1; T.w[0] = local.w; T.g[0] = local.g; T.t[0] = local.touched;
  }
}

void brk_neumf_fill_args(v2::Args& A, const brk_neumf_model* m, const brk_neumf_shards* sh, const int32_t* u,
                         const int32_t* i, const float* y, int64_t batch, int64_t global_batch, int64_t first_index,
                         int32_t training, uint32_t dropout_seed, uint32_t dropout_epoch, const brk_neumf_workspace* ws,
                         float* out, float* loss_out) {
  tab_ref(A.uMLP, m->uMLP, sh ? &sh->uMLP : nullptr); tab_ref(A.iMLP, m->iMLP, sh ? &sh->iMLP : nullptr);
  tab_ref(A.uMF, m->uMF, sh ? &sh->uMF : nullptr); tab_ref(A.iMF, m->iMF, sh ? &sh->iMF : nullptr);
  A.dense = m->dense;
  A.u = u; A.i = i; A.y = y ? y : out; A.B = batch; A.first_index = first_index;
  A.global_B = global_batch > 0 ? global_batch : batch;
  A.h1 = ws->h1; A.h2 = ws->h2; A.dy1 = ws->dy1; A.dy2 = ws->dy2; A.out = out; A.acc = ws->acc;
  A.bn_moving = m->bn_moving; A.loss_out = y ? loss_out : nullptr;
  A.drop_seed = dropout_seed; A.drop_epoch = dropout_epoch;
  A.dropout = (m->dropout != 0 && training) ? 1 : 0;
  A.loss_kind = m->loss; A.training = training;
}

int brk_neumf_step_v2(brk_ctx* ctx, const brk_neumf_model* m, const brk_neumf_shards* sh, const int32_t* u,
                      const int32_t* i, const float* y, int64_t batch, int64_t global_batch, int64_t first_index,
                      int32_t training, uint32_t dropout_seed, uint32_t dropout_epoch, const brk_neumf_workspace* ws,
                      float* out, float* loss_out, cudaStream_t st, int* rc_out) {
  v2::Args A;
  brk_neumf_fill_args(A, m, sh, u, i, y, batch, global_batch, first_index, training, dropout_seed, dropout_epoch, ws, out, loss_out);
#define BRK_V2_CASE(E_, A_, B_, C_)                                                                      \
  if (m->E == E_ && m->H1 == A_ && m->H2 == B_ && m->H3 == C_) {                                          \
    *rc_out = m->act == 0 ? v2::run<E_, A_, B_, C_, 0>(ctx, A, st) : v2::run<E_, A_, B_, C_, 1>(ctx, A, st); \
    return 0;                                                                                             \
  }
  BRK_V2_CASE(32, 32, 16, 8)
  BRK_V2_CASE(64, 64, 32, 16)
  BRK_V2_CASE(16, 16, 8, 4)
  BRK_V2_CASE(8, 8, 4, 2)
#undef BRK_V2_CASE
  return 1;
}
