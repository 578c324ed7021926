// NeuMF on the 5th-generation tensor cores (tcgen05, TF32 operands, fp32 accumulation in TMEM).
//
// Every activation / gradient tile of 128 samples is staged in shared memory sample-major (rows of 32 floats
// = 128 B, one region of ROWS*128 B per block of 32 columns), in one of the two swizzles the tensor core reads
// fp32 (TF32) operands through:
//   "KM" K-major, SWIZZLE_128B        : 8-row groups of 1024 B, 16-byte chunk index ^ (row & 7)
//   "MN" MN-major, SWIZZLE_128B_BASE32B: 4-row groups of  512 B, 32-byte chunk index ^ (row & 3)
// and the three products of a layer are
//   forward      Y[s][j]  = sum_k X[s][k] Wt[j][k]     A = X  (KM),  B = W^T image (KM)
//   input grad   dX[s][k] = sum_j dZ[s][j] W[k][j]     A = dZ (KM),  B = W image, Keras [in][out] (KM)
//   weight grad  dW[k][j] = sum_s X[s][k] dZ[s][j]     A = X  (MN: rows are the reduction index), B = dZ (MN)
// so no tile is ever transposed: the sample-major rows are simply written with the swizzle of the view(s)
// that will read them.  One elected thread issues the MMAs (M = 128 samples or features, N = layer
// width, K = 8 per instruction); the accumulators are read back with tcgen05.ld, one TMEM lane (= one sample,
// or one weight row) per thread.
//
// This file starts with the building blocks and a self-test entry (brk_tc_selftest) that checks each
// descriptor form against a host product; the NeuMF phases are built from the same helpers.
#include "neumf_common.cuh"
#include "tc.cuh"
#include "tc_tiles.cuh"

namespace ntc {

// ---- self-test ---------------------------------------------------------------------------------------------
// Stages Ag [a_rows x a_cols] and Bg [b_rows x b_cols] (row-major fp32, cols multiples of 32, rows multiples of
// 8) into swizzled tiles, runs one product and dumps TMEM lanes 0..127 x N columns to out [128 x N].
template <int M, int N, int A_MN, int B_MN>
__global__ void __launch_bounds__(kThreads) selftest_kernel(const float* __restrict__ Ag, int a_rows, int a_cols,
                                                            const float* __restrict__ Bg, int b_rows, int b_cols,
                                                            int K, float* __restrict__ out) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* As = smem;
  uint8_t* Bs = As + size_t(a_rows) * a_cols * 4;
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_slot;
  const int t = threadIdx.x;
  auto stage = [&](uint8_t* dst, const float* src, int rows, int cols, int mn) {
    for (int idx = t; idx < rows * (cols / 4); idx += kThreads) {
      const int r = idx / (cols / 4), c4 = idx % (cols / 4);
      const float4 v = *reinterpret_cast<const float4*>(src + size_t(r) * cols + c4 * 4);
      *reinterpret_cast<float4*>(dst + (mn ? mn_off16(rows, r, c4) : km_off16(rows, r, c4))) = v;
    }
  };
  stage(As, Ag, a_rows, a_cols, A_MN);
  stage(Bs, Bg, b_rows, b_cols, B_MN);
  if (t == 0) { tc::mbar_init(tc::smem_u32(&bar), 1); tc::fence_barrier_init(); }
  if (t < 32) tc::tmem_alloc<256>(tc::smem_u32(&tmem_slot));
  tc::fence_proxy_async_smem();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = tmem_slot;
  if (t == 0) {
    issue_gemm<M, N, A_MN, B_MN>(tmem, tc::smem_u32(As), a_rows, tc::smem_u32(Bs), b_rows, K, false);
    tc::mma_commit(tc::smem_u32(&bar));
  }
  tc::mbar_wait(tc::smem_u32(&bar), 0);
  tc::fence_after_sync();
  const int warp = t >> 5;
  for (int c0 = 0; c0 < N; c0 += 32) {
    uint32_t r[32];
    tc::tmem_ld_32x32_issue(tmem + (uint32_t(warp * 32) << 16) + uint32_t(c0), r);
    tc::tmem_ld_wait(r);
    for (int j = 0; j < 32 && c0 + j < N; ++j) out[size_t(t) * N + c0 + j] = __uint_as_float(r[j]);
  }
  tc::fence_before_sync();
  __syncthreads();
  if (t < 32) tc::tmem_dealloc<256>(tmem);
}


// =====================================================================================================
// NeuMF phases (same five-phase split at the BatchNorm dependencies as neumf.cu / neumf2.cu, same HBM
// intermediates h1, h2, dy1, dy2 in feature-major [H][B] order, same accumulators and parameter layout).
// =====================================================================================================
using v2::Acc; using v2::Args; using v2::Layout; using v2::RowRef; using v2::TabRef;
using v2::act_f; using v2::act_grad; using v2::drop16_bits; using v2::locate; using v2::mark_row;
using v2::kBnEps; using v2::kBnMomentum; using v2::kDropScale;

constexpr int TS = 128;          // samples per tile = TMEM lanes
constexpr int NT = 256;          // threads per CTA: warp w reads TMEM lane quadrant (w & 3), column half (w >> 2)
constexpr int SP = TS + 1;       // pitch of the feature-major fp32 staging tiles: odd -> conflict-free along s and along f

// Weight images: the Dense kernels pre-arranged (once per step, prep_images) as the swizzled K-major B
// operands the phases copy straight into shared memory.
template <int E, int H1, int H2, int H3>
struct Img {
  static constexpr int K0 = 2 * E;
  static constexpr int N3 = H3 < 16 ? 16 : H3;                    // layer-3 width padded to the MMA's minimum N
  static constexpr int W1t = 0;                                   // [H1 rows][K0]   forward 1:  B[n=j][k]
  static constexpr int W2t = W1t + H1 * pad32(K0);                // [H2 rows][H1]   forward 2
  static constexpr int W3t = W2t + H2 * pad32(H1);                // [N3 rows][H2]   forward 3
  static constexpr int W1 = W3t + N3 * pad32(H2);                 // [K0 rows][H1]   input grad 1: B[n=k][kred=j]
  static constexpr int W2 = W1 + K0 * pad32(H1);                  // [H1 rows][H2]   input grad 2
  static constexpr int total = W2 + H1 * pad32(H2);
};

template <int E, int H1, int H2, int H3>
__global__ void prep_images(const float* __restrict__ w, float* __restrict__ img) {
  using L = Layout<E, H1, H2, H3>; using I = Img<E, H1, H2, H3>;
  constexpr int K0 = I::K0;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < I::total; idx += gridDim.x * blockDim.x) {
    int base, rows, cols, r, c; float v = 0.f;
    if (idx < I::W2t)      { base = I::W1t; rows = H1;    cols = pad32(K0); r = (idx - base) / cols; c = (idx - base) % cols; if (c < K0) v = w[L::W1 + c * H1 + r]; }
    else if (idx < I::W3t) { base = I::W2t; rows = H2;    cols = pad32(H1); r = (idx - base) / cols; c = (idx - base) % cols; if (c < H1) v = w[L::W2 + c * H2 + r]; }
    else if (idx < I::W1)  { base = I::W3t; rows = I::N3; cols = pad32(H2); r = (idx - base) / cols; c = (idx - base) % cols; if (c < H2 && r < H3) v = w[L::W3 + c * H3 + r]; }
    else if (idx < I::W2)  { base = I::W1;  rows = K0;    cols = pad32(H1); r = (idx - base) / cols; c = (idx - base) % cols; if (c < H1) v = w[L::W1 + r * H1 + c]; }
    else                   { base = I::W2;  rows = H1;    cols = pad32(H2); r = (idx - base) / cols; c = (idx - base) % cols; if (c < H2) v = w[L::W2 + r * H2 + c]; }
    img[base + km_off16(rows, r, c >> 2) / 4 + (c & 3)] = v;
  }
}

__device__ __forceinline__ void copy16(uint8_t* dst, const float* __restrict__ src, int n_floats) {
  for (int i = threadIdx.x * 4; i < n_floats; i += NT * 4)
    *reinterpret_cast<float4*>(dst + size_t(i) * 4) = __ldg(reinterpret_cast<const float4*>(src + i));
}
template <int N>
__device__ __forceinline__ void copy_small(float* dst, const float* __restrict__ src) {
  for (int i = threadIdx.x; i < N; i += NT) dst[i] = __ldg(src + i);
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
// per-feature sums over the tile's samples of a staged feature-major tile: all threads take a slice of the
// samples (float partials over <= 32 samples), combined with double atomics
template <int H>
__device__ __forceinline__ void row_sums(const float* A, const float* Bm, double* sumA, double* sumAB) {
  constexpr int PARTS = NT / H, LEN = TS / PARTS;
  static_assert(PARTS * H == NT && LEN * PARTS == TS, "row_sums split");
  const int f = threadIdx.x % H, part = threadIdx.x / H;
  float s = 0.f, q = 0.f;
#pragma unroll 8
  for (int i = 0; i < LEN; ++i) {
    const int r = part * LEN + ((i + f) & (LEN - 1));          // rotate: lanes of a warp hit distinct banks
    const float a = A[f * SP + r], b = Bm ? Bm[f * SP + r] : a;
    s += a; q = fmaf(a, b, q);
  }
  __shared__ float rs_part[2][NT];
  rs_part[0][threadIdx.x] = s; rs_part[1][threadIdx.x] = q;
  __syncthreads();
  if (threadIdx.x < H) {                                       // one atomic pair per feature per CTA
    double ds = 0.0, dq = 0.0;
#pragma unroll
    for (int p = 0; p < PARTS; ++p) { ds += double(rs_part[0][p * H + f]); dq += double(rs_part[1][p * H + f]); }
    atomicAdd(sumA + f, ds);
    atomicAdd(sumAB + f, dq);
  }
}
template <int H>
__device__ __forceinline__ void store_tile(const float* T, float* __restrict__ dst, int64_t B, int64_t b0, int valid) {
  for (int idx = threadIdx.x; idx < H * TS; idx += NT) {
    const int f = idx / TS, s = idx % TS;
    if (s < valid) dst[int64_t(f) * B + b0 + s] = T[f * SP + s];
  }
}
// TMEM -> registers: 32 consecutive columns of this thread's lane
__device__ __forceinline__ void tmem_load32(uint32_t tmem, int warp, int col, float (&v)[32]) {
  uint32_t r[32];
  tc::tmem_ld_32x32_issue(tmem + (uint32_t((warp & 3) * 32) << 16) + uint32_t(col), r);
  tc::tmem_ld_wait(r);
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
}

struct Ctl {                       // per-CTA control block in static shared memory
  uint64_t bar;
  uint32_t tmem;
};
template <int COLS>
__device__ __forceinline__ uint32_t tc_begin(Ctl& c) {
  if (threadIdx.x == 0) { tc::mbar_init(tc::smem_u32(&c.bar), 1); tc::fence_barrier_init(); }
  if (threadIdx.x < 32) tc::tmem_alloc<COLS>(tc::smem_u32(&c.tmem));
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  return c.tmem;
}
template <int COLS>
__device__ __forceinline__ void tc_end(uint32_t tmem) {
  tc::fence_before_sync();
  __syncthreads();
  if (threadIdx.x < 32) tc::tmem_dealloc<COLS>(tmem);
}
// operands written with st.shared -> visible to the tensor core; then one thread issues
#define NTC_OPERANDS_READY() do { tc::fence_proxy_async_smem(); __syncthreads(); tc::fence_after_sync(); } while (0)

// BRK_NTC_TRACE (hex address of a device buffer of >= 320 uint64): %globaltimer stamps of block 0 / thread 0 of
// tc_head (words 0..63), tc_bwd2 (64..127), tc_bwd1 (128..191), tc_fwd1 (192..223), tc_fwd2 (224..255) --
// profiles/neumf_tc_trace.py.  A null pointer (the default) costs one predicated-off branch per stamp.
__device__ unsigned long long* g_trace = nullptr;
struct Stamper {
  unsigned long long* p; unsigned long long* end;
  __device__ __forceinline__ Stamper(int base, int n) {
    unsigned long long* g = (blockIdx.x == 0 && threadIdx.x == 0) ? g_trace : nullptr;
    p = g ? g + base : nullptr; end = g ? g + base + n : nullptr;
  }
  __device__ __forceinline__ void operator()() {
    if (p != nullptr && p < end) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
      *p++ = t;
    }
  }
};

extern __shared__ __align__(1024) uint8_t ntc_smem_raw[];
__device__ __forceinline__ uint8_t* smem_base() {
  return reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ntc_smem_raw) + 1023) & ~uintptr_t(1023));
}

// zero columns [H, pad32(H)) of a 128-row tile (both swizzles share the 16-byte granularity)
template <int H>
__device__ __forceinline__ void zero_pad_cols(uint8_t* T, bool mn) {
  constexpr int PC = (pad32(H) - H) / 4;
  if constexpr (PC > 0) {
    for (int idx = threadIdx.x; idx < TS * PC; idx += NT) {
      const int s = idx / PC, c4 = H / 4 + idx % PC;
      *reinterpret_cast<float4*>(T + (mn ? mn_off16(TS, s, c4) : km_off16(TS, s, c4))) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
}

// Tile ids into shared memory (one coalesced load per table), so that the row gathers do not chain on them.
__device__ __forceinline__ void load_tile_ids(int32_t* ids_s, const Args& A, int64_t b0, int valid) {
  const int t = threadIdx.x;
  if (t < 2 * TS) {
    const int r = t & (TS - 1);
    ids_s[t] = r < valid ? __ldg((t < TS ? A.u : A.i) + b0 + r) : 0;
  }
}
// Gather x0 = [uMLP[u], iMLP[i]] for a tile: E/4 lanes per row, 16 bytes each (coalesced rows); every load of the
// thread is issued before the first use.  MN = 0: K-major swizzle, 1: MN-major swizzle.
template <int E>
__device__ __forceinline__ void gather_x0_issue(float4 (&v)[2 * (TS / (NT / (E / 4)))], const Args& A, const int32_t* ids_s, int valid) {
  constexpr int LPR = E / 4, RPP = NT / LPR, NP = TS / RPP;
  const int t = threadIdx.x, c4 = t % LPR, rr = t / LPR;
#pragma unroll
  for (int tab = 0; tab < 2; ++tab)
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      const int r = p * RPP + rr;
      v[tab * NP + p] = r < valid ? __ldg(reinterpret_cast<const float4*>(locate<E>(tab == 0 ? A.uMLP : A.iMLP, ids_s[tab * TS + r]).w) + c4)
                                  : make_float4(0.f, 0.f, 0.f, 0.f);
    }
}
template <int E, int MN>
__device__ __forceinline__ void gather_x0_store(uint8_t* Xs, const float4 (&v)[2 * (TS / (NT / (E / 4)))], const Args& A,
                                                const uint32_t* masks) {
  constexpr int LPR = E / 4, RPP = NT / LPR, NP = TS / RPP, MW = 2 * E / 32;
  const int t = threadIdx.x, c4 = t % LPR, rr = t / LPR;
#pragma unroll
  for (int tab = 0; tab < 2; ++tab)
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      const int r = p * RPP + rr;
      float4 x = v[tab * NP + p];
      if (A.dropout) {
        const int f = tab * E + 4 * c4;
        const uint32_t m = masks[r * MW + (f >> 5)] >> (f & 31);
        x.x = (m & 1u) ? x.x * kDropScale : 0.f; x.y = (m & 2u) ? x.y * kDropScale : 0.f;
        x.z = (m & 4u) ? x.z * kDropScale : 0.f; x.w = (m & 8u) ? x.w * kDropScale : 0.f;
      }
      *reinterpret_cast<float4*>(Xs + (MN ? mn_off16(TS, r, tab * LPR + c4) : km_off16(TS, r, tab * LPR + c4))) = x;
    }
}
template <int E, int MN>
__device__ __forceinline__ void gather_x0(uint8_t* Xs, const Args& A, const int32_t* ids_s, const uint32_t* masks, int valid) {
  float4 v[2 * (TS / (NT / (E / 4)))];
  gather_x0_issue<E>(v, A, ids_s, valid);
  gather_x0_store<E, MN>(Xs, v, A, masks);
}

// ---- phase 1: x0 = dropout([uMLP[u], iMLP[i]]); h1 = act(x0 W1 + b1); batch sums of h1 -----------------
template <int E, int H1, int H2, int H3, int ACT>
__global__ void __launch_bounds__(NT) tc_fwd1(const Args A, const float* __restrict__ img) {
  using L = Layout<E, H1, H2, H3>; using AC = Acc<H1, H2>; using I = Img<E, H1, H2, H3>;
  constexpr int K0 = 2 * E, MW = K0 / 32;
  uint8_t* sm = smem_base();
  uint8_t* As = sm;                                        // [K0/32][128 rows][128 B]   x0, K-major view
  uint8_t* Ws = As + TS * K0 * 4;                          // W1^T image
  float* bs = reinterpret_cast<float*>(Ws + H1 * pad32(K0) * 4);   // [H1]
  uint32_t* masks = reinterpret_cast<uint32_t*>(bs + H1);  // [128][MW] keep bits of layer 0
  float* Ys = reinterpret_cast<float*>(As);                // staging [H1][SP], aliases x0 once the MMA has read it
  __shared__ Ctl ctl;
  __shared__ int32_t ids_s[2 * TS];
  const int64_t b0 = int64_t(blockIdx.x) * TS;
  const int valid = int((A.B - b0) < int64_t(TS) ? (A.B - b0) : int64_t(TS));
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  load_tile_ids(ids_s, A, b0, valid);
  const uint32_t tmem = tc_begin<64>(ctl);
  copy16(Ws, img + I::W1t, H1 * pad32(K0));
  copy_small<H1>(bs, A.dense.w + L::b1);
  if (A.dropout) {
    const int s = t & (TS - 1), hf = t >> 7;
    for (int c = hf * (K0 / 32); c < (hf + 1) * (K0 / 32); ++c) {     // K0/16 calls per sample, half per thread
      const uint32_t bits = s < valid ? drop16_bits(uint64_t(A.first_index + b0 + s), c, 0, A.drop_seed, A.drop_epoch) : 0u;
      reinterpret_cast<uint16_t*>(masks + s * MW)[c] = uint16_t(bits);
    }
    __syncthreads();
  }
  gather_x0<E, 0>(As, A, ids_s, masks, valid);
  NTC_OPERANDS_READY();
  if (t == 0) {
    issue_gemm<128, H1, 0, 0>(tmem, tc::smem_u32(As), TS, tc::smem_u32(Ws), H1, K0, false);
    tc::mma_commit(tc::smem_u32(&ctl.bar));
  }
  tc::mbar_wait(tc::smem_u32(&ctl.bar), 0);
  tc::fence_after_sync();
  {                                                        // epilogue: bias + activation, staged feature-major
    constexpr int HC = H1 / 2;                             // columns per warp half
    const int s = (warp & 3) * 32 + lane, c0 = (warp >> 2) * HC;
    for (int cc = 0; cc < HC; cc += 32) {
      float v[32];
      tmem_load32(tmem, warp, c0 + cc, v);
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (cc + j < HC) Ys[(c0 + cc + j) * SP + s] = s < valid ? act_f<ACT>(v[j] + bs[c0 + cc + j]) : 0.f;
    }
  }
  __syncthreads();
  store_tile<H1>(Ys, A.h1, A.B, b0, valid);
  if (A.training) row_sums<H1>(Ys, nullptr, A.acc + AC::s1, A.acc + AC::q1);
  tc_end<64>(tmem);
}

// A tile from a feature-major HBM intermediate: thread-per-sample scalar loads (coalesced along the samples),
// BatchNorm + dropout applied on the fly, rows written in the K-major swizzle.  Also returns nothing else:
// the epilogues recompute what they need.
template <int H, int LAYER>
__device__ __forceinline__ void stage_bn_tile(uint8_t* At, const float* __restrict__ h, const Args& A, int64_t b0, int valid,
                                              const float* mean, const float* rstd, const float* gam, const float* bet,
                                              float* Xh /* optional feature-major xhat staging */) {
  const int t = threadIdx.x, s = t & (TS - 1), hf = t >> 7;
  constexpr int HH = H / 2;                               // features per thread half (multiple of 8 for H >= 16)
  const bool ok = s < valid;
  uint32_t bits[(HH + 15) / 16];
#pragma unroll
  for (int c = 0; c < (HH + 15) / 16; ++c)
    bits[c] = (A.dropout && ok) ? drop16_bits(uint64_t(A.first_index + b0 + s), (hf * HH) / 16 + c, LAYER, A.drop_seed, A.drop_epoch)
                                : 0xFFFFu;
  // when HH is 8 the half's bits are the upper or lower byte of one 16-feature call
  const int bit0 = (hf * HH) & 15;
  float hv[HH];
#pragma unroll
  for (int fl = 0; fl < HH; ++fl) hv[fl] = ok ? __ldg(h + int64_t(hf * HH + fl) * A.B + b0 + s) : 0.f;   // all loads in flight
#pragma unroll
  for (int f4 = 0; f4 < HH / 4; ++f4) {
    float v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int fl = f4 * 4 + q, f = hf * HH + fl;
      const float xh = (hv[fl] - mean[f]) * rstd[f];
      if (Xh) Xh[f * SP + s] = ok ? xh : 0.f;
      float y = gam[f] * xh + bet[f];
      if (A.dropout) y = ((bits[(bit0 + fl) >> 4] >> ((bit0 + fl) & 15)) & 1u) ? y * kDropScale : 0.f;
      v[q] = ok ? y : 0.f;
    }
    *reinterpret_cast<float4*>(At + km_off16(TS, s, (hf * HH) / 4 + f4)) = make_float4(v[0], v[1], v[2], v[3]);
  }
}

// ---- phase 2: d1 = dropout(bn1(h1)); h2 = act(d1 W2 + b2); batch sums of h2 -----------------------------
template <int E, int H1, int H2, int H3, int ACT>
__global__ void __launch_bounds__(NT) tc_fwd2(const Args A, const float* __restrict__ img) {
  using L = Layout<E, H1, H2, H3>; using AC = Acc<H1, H2>; using I = Img<E, H1, H2, H3>;
  uint8_t* sm = smem_base();
  uint8_t* As = sm;                                        // [pad32(H1)/32][128][128 B]
  uint8_t* Ws = As + TS * pad32(H1) * 4;                   // W2^T image
  float* bs = reinterpret_cast<float*>(Ws + H2 * pad32(H1) * 4);
  float* mean = bs + H2; float* rstd = mean + H1; float* gam = rstd + H1; float* bet = gam + H1;
  float* Ys = reinterpret_cast<float*>(As);                // staging [H2][SP]
  __shared__ Ctl ctl;
  const int64_t b0 = int64_t(blockIdx.x) * TS;
  const int valid = int((A.B - b0) < int64_t(TS) ? (A.B - b0) : int64_t(TS));
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const uint32_t tmem = tc_begin<64>(ctl);
  copy16(Ws, img + I::W2t, H2 * pad32(H1));
  copy_small<H2>(bs, A.dense.w + L::b2);
  copy_small<H1>(gam, A.dense.w + L::g1);
  copy_small<H1>(bet, A.dense.w + L::be1);
  bn_prepare<H1>(mean, rstd, A.acc + AC::s1, A.acc + AC::q1, A.bn_moving, A.bn_moving + H1, A.B, A.training);
  __syncthreads();
  stage_bn_tile<H1, 1>(As, A.h1, A, b0, valid, mean, rstd, gam, bet, nullptr);
  NTC_OPERANDS_READY();
  if (t == 0) {
    issue_gemm<128, H2, 0, 0>(tmem, tc::smem_u32(As), TS, tc::smem_u32(Ws), H2, H1, false);
    tc::mma_commit(tc::smem_u32(&ctl.bar));
  }
  tc::mbar_wait(tc::smem_u32(&ctl.bar), 0);
  tc::fence_after_sync();
  {
    constexpr int HC = H2 / 2;
    const int s = (warp & 3) * 32 + lane, c0 = (warp >> 2) * HC;
    float v[32];
    tmem_load32(tmem, warp, c0, v);
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (j < HC) Ys[(c0 + j) * SP + s] = s < valid ? act_f<ACT>(v[j] + bs[c0 + j]) : 0.f;
  }
  __syncthreads();
  store_tile<H2>(Ys, A.h2, A.B, b0, valid);
  if (A.training) row_sums<H2>(Ys, nullptr, A.acc + AC::s2, A.acc + AC::q2);
  tc_end<64>(tmem);
}

// ---- phase 3: d2 = dropout(bn2(h2)); h3 = act(d2 W3 + b3); MF dot; logit, prediction, loss; then (training)
//      head / layer-3 gradients and dd2 = d loss / d d2 with its BatchNorm-backward sums -----------------------
template <int E, int H1, int H2, int H3, int ACT>
__global__ void __launch_bounds__(NT, 2) tc_head(const Args A, const float* __restrict__ img, int n_tiles) {
  using L = Layout<E, H1, H2, H3>; using AC = Acc<H1, H2>; using I = Img<E, H1, H2, H3>;
  constexpr int N3 = I::N3, LPR = E / 4, RPP = NT / LPR, ZP = H3 + 1;
  uint8_t* sm = smem_base();
  uint8_t* As = sm;                                        // d2, K-major view: [128][32 floats] (H2 <= 32)
  uint8_t* Ws = As + TS * pad32(H2) * 4;                   // W3^T image [N3][pad32(H2)]
  float* W3s = reinterpret_cast<float*>(Ws + N3 * pad32(H2) * 4);   // W3 plain [H2][H3] (input grad, SIMT)
  float* bs = W3s + H2 * H3;                               // [H3]
  float* w4 = bs + ((H3 + 3) & ~3);                        // [H3 + 2]
  float* Xh = w4 + ((H3 + 2 + 3) & ~3);                    // [H2][SP] xhat2
  float* Ds = Xh + H2 * SP;                                // [H2][SP] dd2 staging
  float* Ys = Ds + H2 * SP;                                // [H3][SP] h3
  float* Zt = Ys + H3 * SP;                                // [128][ZP] dz3 sample-major
  float* dl = Zt + TS * ZP;                                // [128]
  float* mfs = dl + TS;                                    // [128]
  float* mean = mfs + TS; float* rstd = mean + H2; float* gam = rstd + H2; float* bet = gam + H2;
  __shared__ Ctl ctl;
  __shared__ double red[32];
  __shared__ int32_t ids_s[2 * TS];
  // Persistent over tiles: the head / layer-3 weight gradients of all of this CTA's tiles are summed here and leave
  // with ONE atomic per entry per CTA.  (One CTA per tile with its own atomics put 512 tiles' worth of adds on the same
  // ~550 words at configs[3] sizes: 85 us for this kernel, most of it the serialised atomics.)
  __shared__ float aW3[H2 * H3], ab3[H3], aW4[H3 + 2];
  const int t = threadIdx.x, warp = t >> 5;
  Stamper stamp(0, 64);
  stamp();
  for (int j = t; j < H2 * H3; j += NT) aW3[j] = 0.f;
  if (t < H3) ab3[t] = 0.f;
  if (t < H3 + 2) aW4[t] = 0.f;
  const uint32_t tmem = tc_begin<32>(ctl);
  copy16(Ws, img + I::W3t, N3 * pad32(H2));
  copy_small<H2 * H3>(W3s, A.dense.w + L::W3);
  copy_small<H3>(bs, A.dense.w + L::b3);
  copy_small<H3 + 2>(w4, A.dense.w + L::W4);
  copy_small<H2>(gam, A.dense.w + L::g2);
  copy_small<H2>(bet, A.dense.w + L::be2);
  bn_prepare<H2>(mean, rstd, A.acc + AC::s2, A.acc + AC::q2, A.bn_moving + 2 * H1, A.bn_moving + 2 * H1 + H2, A.B, A.training);
  zero_pad_cols<H2>(As, false);                            // unused K columns of the tile
  uint32_t phase = 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
  const int64_t b0 = int64_t(tile) * TS;
  const int valid = int((A.B - b0) < int64_t(TS) ? (A.B - b0) : int64_t(TS));
  stamp();
  load_tile_ids(ids_s, A, b0, valid);
  __syncthreads();
  stamp();
  stage_bn_tile<H2, 2>(As, A.h2, A, b0, valid, mean, rstd, gam, bet, Xh);
  NTC_OPERANDS_READY();
  stamp();
  if (t == 0) {
    issue_gemm<128, N3, 0, 0>(tmem, tc::smem_u32(As), TS, tc::smem_u32(Ws), N3, H2, false);
    tc::mma_commit(tc::smem_u32(&ctl.bar));
  }
  // MF dot product while the tensor core works: LPR lanes per row pair; the row chunks stay in registers for
  // the gradient REDs further down
  constexpr int NP = TS / RPP;
  float4 mu[NP], mi[NP];
  const int mc4 = t % LPR, mrr = t / LPR;
#pragma unroll
  for (int p = 0; p < NP; ++p) {
    const int r = p * RPP + mrr;
    mu[p] = mi[p] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < valid) {
      mu[p] = __ldg(reinterpret_cast<const float4*>(locate<E>(A.uMF, ids_s[r]).w) + mc4);
      mi[p] = __ldg(reinterpret_cast<const float4*>(locate<E>(A.iMF, ids_s[TS + r]).w) + mc4);
    }
  }
#pragma unroll
  for (int p = 0; p < NP; ++p) {
    float part = fmaf(mu[p].x, mi[p].x, fmaf(mu[p].y, mi[p].y, fmaf(mu[p].z, mi[p].z, mu[p].w * mi[p].w)));
    part = group_sum<LPR>(part);
    if (mc4 == 0) mfs[p * RPP + mrr] = part;
  }
  tc::mbar_wait(tc::smem_u32(&ctl.bar), phase);
  phase ^= 1u;
  tc::fence_after_sync();
  __syncthreads();                                         // mfs visible
  stamp();
  float loss_local = 0.f;
  if (t < TS) {                                            // one thread per sample: warps 0..3 = the four lane quadrants
    const int s = t;
    float v[32];
    tmem_load32(tmem, warp, 0, v);
    float dlogit = 0.f;
    float h3[H3];
    if (s < valid) {
      float logit = w4[H3 + 1];
#pragma unroll
      for (int j = 0; j < H3; ++j) { h3[j] = act_f<ACT>(v[j] + bs[j]); logit = fmaf(h3[j], w4[j], logit); }
      logit = fmaf(mfs[s], w4[H3], logit);
      const float o = 1.0f / (1.0f + expf(-logit));
      A.out[b0 + s] = o;
      const float yv = __ldg(A.y + b0 + s);
      const float invB = 1.0f / float(A.global_B);
      if (A.loss_kind == 0) { const float e = o - yv; loss_local = e * e; dlogit = 2.f * e * o * (1.f - o) * invB; }
      else { loss_local = fmaxf(logit, 0.f) - logit * yv + log1pf(expf(-fabsf(logit))); dlogit = (o - yv) * invB; }
    } else {
#pragma unroll
      for (int j = 0; j < H3; ++j) h3[j] = 0.f;
    }
    dl[s] = dlogit;
#pragma unroll
    for (int j = 0; j < H3; ++j) {
      Ys[j * SP + s] = h3[j];
      Zt[s * ZP + j] = dlogit * w4[j] * act_grad<ACT>(h3[j]);
    }
  }
  const double lsum = block_sum_double(double(loss_local), red);
  if (t == 0) atomicAdd(A.acc + AC::loss, lsum);
  stamp();
  if (A.training) {
    __syncthreads();
    // head weights: dW4[j] = sum_s z[j][s] dl[s] (z = [h3, mf]), db4 = sum_s dl[s]: one warp per output, lanes over samples
    for (int j = warp; j < H3 + 2; j += NT / 32) {
      float sacc = 0.f;
#pragma unroll
      for (int q = 0; q < TS / 32; ++q) {
        const int s = q * 32 + (t & 31);
        sacc = fmaf(j < H3 ? Ys[j * SP + s] : (j == H3 ? mfs[s] : 1.f), dl[s], sacc);
      }
      sacc = warp_sum(sacc);
      if ((t & 31) == 0) aW4[j] += sacc;
    }
    // layer-3 weights: dW3[k][j] = sum_s d2[s][k] dz3[s][j]; db3[j] = sum_s dz3[s][j]   (small: CUDA cores).
    // thread = (k, group of JG outputs j); d2 is read from the swizzled K-major tile, 8 rows per address step
    {
      constexpr int JG = (H2 * H3) / NT > 0 ? (H2 * H3) / NT : 1;      // outputs j per thread
      constexpr int NTH = (H2 * H3) / JG;                              // threads used
      if (t < NTH) {
        const int k = t % H2, j0 = (t / H2) * JG;
        float acc[JG];
#pragma unroll
        for (int q = 0; q < JG; ++q) acc[q] = 0.f;
        const uint8_t* base = As + (k & 3) * 4;
        for (int s8 = 0; s8 < TS / 8; ++s8) {
#pragma unroll
          for (int r = 0; r < 8; ++r) {
            const float a = *reinterpret_cast<const float*>(base + s8 * 1024 + r * 128 + (((k >> 2) ^ r) << 4));
            const float* z = Zt + (s8 * 8 + r) * ZP + j0;
#pragma unroll
            for (int q = 0; q < JG; ++q) acc[q] = fmaf(a, z[q], acc[q]);
          }
        }
#pragma unroll
        for (int q = 0; q < JG; ++q) aW3[k * H3 + j0 + q] += acc[q];
      }
      for (int j = warp; j < H3; j += NT / 32) {                       // db3: one warp per j
        float sacc = 0.f;
#pragma unroll
        for (int q = 0; q < TS / 32; ++q) sacc += Zt[(q * 32 + (t & 31)) * ZP + j];
        sacc = warp_sum(sacc);
        if ((t & 31) == 0) ab3[j] += sacc;
      }
    }
    // dd2[s][k] = dropout-mask * sum_j dz3[s][j] W3[k][j]: thread (sample, half of the k range)
    {
      const int s = t & (TS - 1), hf = t >> 7;
      constexpr int HH = H2 / 2;
      float z[H3];
#pragma unroll
      for (int j = 0; j < H3; ++j) z[j] = Zt[s * ZP + j];
      uint32_t bits = 0xFFFFFFFFu;
      if (A.dropout && s < valid) {
        bits = 0;
        for (int c = 0; c < (HH + 15) / 16; ++c)
          bits |= drop16_bits(uint64_t(A.first_index + b0 + s), (hf * HH) / 16 + c, 2, A.drop_seed, A.drop_epoch) << (16 * c);
        bits >>= (hf * HH) & 15;
      }
#pragma unroll 4
      for (int kl = 0; kl < HH; ++kl) {
        const int k = hf * HH + kl;
        float d = 0.f;
        if constexpr ((H3 & 3) == 0) {                       // W3 row k as float4 broadcasts: a quarter of the LDS instructions
#pragma unroll
          for (int j = 0; j < H3; j += 4) {
            const float4 w = *reinterpret_cast<const float4*>(W3s + k * H3 + j);
            d = fmaf(z[j], w.x, d); d = fmaf(z[j + 1], w.y, d); d = fmaf(z[j + 2], w.z, d); d = fmaf(z[j + 3], w.w, d);
          }
        } else
#pragma unroll
        for (int j = 0; j < H3; ++j) d = fmaf(z[j], W3s[k * H3 + j], d);
        if (A.dropout) d = ((bits >> kl) & 1u) ? d * kDropScale : 0.f;
        Ds[k * SP + s] = s < valid ? d : 0.f;
      }
    }
    stamp();
    // MF embedding gradients: LPR lanes per row pair, 16-byte REDs into the owners' accumulators
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      const int r = p * RPP + mrr;
      if (r < valid) {
        const RowRef ru = locate<E>(A.uMF, ids_s[r]), ri = locate<E>(A.iMF, ids_s[TS + r]);
        const float dmf = dl[r] * w4[H3];
        red_add_f4(ru.g + 4 * mc4, make_float4(dmf * mi[p].x, dmf * mi[p].y, dmf * mi[p].z, dmf * mi[p].w));
        red_add_f4(ri.g + 4 * mc4, make_float4(dmf * mu[p].x, dmf * mu[p].y, dmf * mu[p].z, dmf * mu[p].w));
        if (mc4 == 0) { mark_row(ru); mark_row(ri); }
      }
    }
    __syncthreads();
    stamp();
    store_tile<H2>(Ds, A.dy2, A.B, b0, valid);
    row_sums<H2>(Ds, Xh, A.acc + AC::d2, A.acc + AC::e2);
  }
  tc::fence_before_sync();
  __syncthreads();                                         // tiles, ids and TMEM may be overwritten by the next iteration
  }
  stamp();
  if (A.training) {                                        // one atomic per entry per CTA
    for (int j = t; j < H2 * H3; j += NT) atomicAdd(A.dense.g + L::W3 + j, aW3[j]);
    if (t < H3) atomicAdd(A.dense.g + L::b3 + t, ab3[t]);
    if (t < H3 + 2) atomicAdd(A.dense.g + L::W4 + t, aW4[t]);
  }
  tc_end<32>(tmem);
}

// dz of a BatchNorm-followed layer for this thread's (sample, feature half): written in both operand
// swizzles (K-major for the input-gradient product, MN-major for the weight-gradient product)
template <int H>
__device__ __forceinline__ void dz_issue(float (&hv)[H / 2], float (&dv)[H / 2], const float* __restrict__ h, const float* __restrict__ dy,
                                         int64_t B, int64_t b0, int valid) {
  const int t = threadIdx.x, s = t & (TS - 1), hf = t >> 7;
  constexpr int HH = H / 2;
  const bool ok = s < valid;
#pragma unroll
  for (int fl = 0; fl < HH; ++fl) {                       // all loads in flight before the first use
    hv[fl] = ok ? __ldg(h + int64_t(hf * HH + fl) * B + b0 + s) : 0.f;
    dv[fl] = ok ? __ldg(dy + int64_t(hf * HH + fl) * B + b0 + s) : 0.f;
  }
}
template <int H, int ACT>
__device__ __forceinline__ void dz_store(uint8_t* Zk, uint8_t* Zm, const float (&hv)[H / 2], const float (&dv)[H / 2], const float* mean,
                                         const float* rstd, const float* gam, const float* sdy, const float* sdyx, int valid) {
  const int t = threadIdx.x, s = t & (TS - 1), hf = t >> 7;
  constexpr int HH = H / 2;
  const bool ok = s < valid;
#pragma unroll
  for (int f4 = 0; f4 < HH / 4; ++f4) {
    float v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int fl = f4 * 4 + q, j = hf * HH + fl;
      const float xh = (hv[fl] - mean[j]) * rstd[j];
      const float dh = gam[j] * rstd[j] * (dv[fl] - sdy[j] - xh * sdyx[j]);
      v[q] = ok ? dh * act_grad<ACT>(hv[fl]) : 0.f;
    }
    const float4 v4 = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(Zk + km_off16(TS, s, (hf * HH) / 4 + f4)) = v4;
    *reinterpret_cast<float4*>(Zm + mn_off16(TS, s, (hf * HH) / 4 + f4)) = v4;
  }
}
template <int H, int ACT>
__device__ __forceinline__ void stage_dz_tiles(uint8_t* Zk, uint8_t* Zm, const float* __restrict__ h, const float* __restrict__ dy,
                                               const float* mean, const float* rstd, const float* gam, const float* sdy,
                                               const float* sdyx, int64_t B, int64_t b0, int valid) {
  float hv[H / 2], dv[H / 2];
  dz_issue<H>(hv, dv, h, dy, B, b0, valid);
  dz_store<H, ACT>(Zk, Zm, hv, dv, mean, rstd, gam, sdy, sdyx, valid);
}

// ---- phase 4 (backward through layer 2 and BatchNorm 1), persistent over tiles ------------------------------
//   dz2 = bn2-backward(dy2) * act'(h2);  dW2 += d1^T dz2 (accumulated in TMEM across this CTA's tiles);
//   dd1 = dropout-mask * dz2 W2^T -> dy1 with its BatchNorm-backward sums
template <int E, int H1, int H2, int H3, int ACT>
__global__ void __launch_bounds__(NT, 2) tc_bwd2(const Args A, const float* __restrict__ img, int n_tiles) {
  using L = Layout<E, H1, H2, H3>; using AC = Acc<H1, H2>; using I = Img<E, H1, H2, H3>;
  constexpr int MW = H1 >= 64 ? H1 : 64;                   // weight-gradient rows per MMA (M); H1 = 32 reads its column block twice
  constexpr int WCOL = H1;                                 // TMEM: [0, H1) dd1, [WCOL, WCOL + H2) dW2
  constexpr int TCOLS = 128;
  uint8_t* sm = smem_base();
  uint8_t* Xm = sm;                                        // d1, MN view [pad32(H1)/32][128][128 B]
  uint8_t* Zk = Xm + TS * pad32(H1) * 4;                   // dz2, K-major view  [128][pad32(H2)]
  uint8_t* Zm = Zk + TS * pad32(H2) * 4;                   // dz2, MN view
  uint8_t* Ws = Zm + TS * pad32(H2) * 4;                   // W2 image [H1 rows][pad32(H2)]
  float* Ds = reinterpret_cast<float*>(Ws + H1 * pad32(H2) * 4);   // [H1][SP] staging (dd1, then dd1 * xhat1)
  float* mean1 = Ds + H1 * SP; float* rstd1 = mean1 + H1; float* gam1 = rstd1 + H1; float* bet1 = gam1 + H1;
  float* mean2 = bet1 + H1; float* rstd2 = mean2 + H2; float* gam2 = rstd2 + H2; float* sdy = gam2 + H2; float* sdyx = sdy + H2;
  __shared__ Ctl ctl;
  __shared__ float rs_part[NT];
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const uint32_t tmem = tc_begin<TCOLS>(ctl);
  copy16(Ws, img + I::W2, H1 * pad32(H2));
  copy_small<H1>(gam1, A.dense.w + L::g1);
  copy_small<H1>(bet1, A.dense.w + L::be1);
  copy_small<H2>(gam2, A.dense.w + L::g2);
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
  zero_pad_cols<H2>(Zk, false);
  zero_pad_cols<H2>(Zm, true);
  __syncthreads();
  uint32_t phase = 0;
  int it = 0;
  float db_acc = 0.f;                                      // this thread's bias-gradient feature, summed over the CTA's tiles
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
    const int64_t b0 = int64_t(tile) * TS;
    const int valid = int((A.B - b0) < int64_t(TS) ? (A.B - b0) : int64_t(TS));
    const int s = t & (TS - 1), hf = t >> 7;
    const bool ok = s < valid;
    // both memory phases of the tile are issued back to back (h2 / dy2 columns, then h1 columns): one DRAM round trip, not two
    float hv2[H2 / 2], dv2[H2 / 2];
    dz_issue<H2>(hv2, dv2, A.h2, A.dy2, A.B, b0, valid);
    constexpr int HH = H1 / 2;
    float hv1[HH];                                          // kept for the epilogue's dd1 * xhat1 (same thread = same sample, same half)
    // d1 = dropout(bn1(h1)) in the MN swizzle (weight-gradient A operand)
    {
      uint32_t bits[(HH + 15) / 16];
#pragma unroll
      for (int c = 0; c < (HH + 15) / 16; ++c)
        bits[c] = (A.dropout && ok) ? drop16_bits(uint64_t(A.first_index + b0 + s), (hf * HH) / 16 + c, 1, A.drop_seed, A.drop_epoch) : 0xFFFFu;
      const int bit0 = (hf * HH) & 15;
#pragma unroll
      for (int fl = 0; fl < HH; ++fl) hv1[fl] = ok ? __ldg(A.h1 + int64_t(hf * HH + fl) * A.B + b0 + s) : 0.f;
#pragma unroll
      for (int f4 = 0; f4 < HH / 4; ++f4) {
        float v[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int fl = f4 * 4 + q, f = hf * HH + fl;
          const float hv = hv1[fl];
          float y = gam1[f] * (hv - mean1[f]) * rstd1[f] + bet1[f];
          if (A.dropout) y = ((bits[(bit0 + fl) >> 4] >> ((bit0 + fl) & 15)) & 1u) ? y * kDropScale : 0.f;
          v[q] = ok ? y : 0.f;
        }
        *reinterpret_cast<float4*>(Xm + mn_off16(TS, s, (hf * HH) / 4 + f4)) = make_float4(v[0], v[1], v[2], v[3]);
      }
    }
    dz_store<H2, ACT>(Zk, Zm, hv2, dv2, mean2, rstd2, gam2, sdy, sdyx, valid);
    NTC_OPERANDS_READY();
    if (t == 0) {
      issue_gemm<128, H1, 0, 0>(tmem, tc::smem_u32(Zk), TS, tc::smem_u32(Ws), H1, H2, false);              // dd1
      // dW2 (+)= d1^T dz2; for H1 < 64 the second 32-column block of the M = 64 operand aliases the first
      constexpr uint32_t idesc = tc::idesc_tf32_f32(MW, H2, 1, 1);
      for (int ks = 0; ks < TS / 8; ++ks) {
        const uint64_t ad = tc::smem_desc_sw128_base32(tc::smem_u32(Xm) + uint32_t(ks) * 1024u, H1 >= 64 ? TS * 128u : 0u, 512);
        const uint64_t bd = tc::smem_desc_sw128_base32(tc::smem_u32(Zm) + uint32_t(ks) * 1024u, TS * 128u, 512);
        tc::mma_tf32_ss(tmem + WCOL, ad, bd, idesc, (ks != 0 || it != 0) ? 1u : 0u);
      }
      tc::mma_commit(tc::smem_u32(&ctl.bar));
    }
    // db2[j] += sum_s dz2[s][j] on the CUDA cores while the tensor core works
    if (t < H2) {
      float sacc = 0.f;
      for (int r = 0; r < TS; ++r) sacc += *reinterpret_cast<const float*>(Zk + km_off16(TS, r, t >> 2) + (t & 3) * 4);
      db_acc += sacc;                                       // one atomic per feature per CTA, after the last tile
    }
    tc::mbar_wait(tc::smem_u32(&ctl.bar), phase);
    phase ^= 1u;
    tc::fence_after_sync();
    // epilogue: dd1 -> dropout mask -> dy1 (HBM) and the sums  sum dd1, sum dd1 * xhat1
    constexpr int HC = H1 / 2;
    const int es = (warp & 3) * 32 + lane, c0 = (warp >> 2) * HC;
    uint32_t ebits[(HC + 15) / 16];
#pragma unroll
    for (int c = 0; c < (HC + 15) / 16; ++c)
      ebits[c] = (A.dropout && es < valid) ? drop16_bits(uint64_t(A.first_index + b0 + es), c0 / 16 + c, 1, A.drop_seed, A.drop_epoch) : 0xFFFFu;
    const int ebit0 = c0 & 15;
    float dd[HC];
    for (int cc = 0; cc < HC; cc += 32) {
      float v[32];
      tmem_load32(tmem, warp, c0 + cc, v);
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (cc + j < HC) {
          float d = v[j];
          if (A.dropout) d = ((ebits[(ebit0 + cc + j) >> 4] >> ((ebit0 + cc + j) & 15)) & 1u) ? d * kDropScale : 0.f;
          d = es < valid ? d : 0.f;
          dd[cc + j] = d;
          Ds[(c0 + cc + j) * SP + es] = d;
        }
    }
    tc::fence_before_sync();
    __syncthreads();
    store_tile<H1>(Ds, A.dy1, A.B, b0, valid);
    double* sum_d = A.acc + AC::d1; double* sum_e = A.acc + AC::e1;
    {
      constexpr int PARTS = NT / H1, LEN = TS / PARTS;
      const int f = t % H1, part = t / H1;
      float sd = 0.f;
#pragma unroll 8
      for (int i = 0; i < LEN; ++i) sd += Ds[f * SP + part * LEN + ((i + f) & (LEN - 1))];
      rs_part[t] = sd;
      __syncthreads();
      if (t < H1) {
        double d = 0.0;
#pragma unroll
        for (int p = 0; p < PARTS; ++p) d += double(rs_part[p * H1 + t]);
        atomicAdd(sum_d + t, d);
      }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < HC; ++j) {                          // second pass through the same staging tile: dd1 * xhat1
      const int f = c0 + j;
      Ds[f * SP + es] = dd[j] * (hv1[j] - mean1[f]) * rstd1[f];      // es == s, c0 == hf * HH: the h1 values loaded for d1
    }
    __syncthreads();
    {
      constexpr int PARTS = NT / H1, LEN = TS / PARTS;
      const int f = t % H1, part = t / H1;
      float se = 0.f;
#pragma unroll 8
      for (int i = 0; i < LEN; ++i) se += Ds[f * SP + part * LEN + ((i + f) & (LEN - 1))];
      rs_part[t] = se;
      __syncthreads();
      if (t < H1) {
        double d = 0.0;
#pragma unroll
        for (int p = 0; p < PARTS; ++p) d += double(rs_part[p * H1 + t]);
        atomicAdd(sum_e + t, d);
      }
    }
    __syncthreads();
  }
  // flush this CTA's weight-gradient accumulator: TMEM lane = row k of dW2, columns = j
  if (it > 0 && warp < 4) {
    tc::fence_after_sync();
    float v[32];
    tmem_load32(tmem, warp, WCOL, v);
    const int k = row_of_lane<MW>(warp * 32 + lane);
    if (k >= 0 && k < H1)                                  // 16-byte REDs: a quarter of the L2 atomic operations
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        if (j < H2) red_add_f4(A.dense.g + L::W2 + k * H2 + j, make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
  }
  if (it > 0 && t < H2) atomicAdd(A.dense.g + L::b2 + t, db_acc);
  tc_end<TCOLS>(tmem);
}

// ---- phase 5 (backward through layer 1 into the embedding rows), persistent over tiles -----------------------
//   dz1 = bn1-backward(dy1) * act'(h1);  dW1 += x0^T dz1 (TMEM-resident);  dx0 = dropout-mask * dz1 W1^T ->
//   16-byte REDs into the user / item MLP rows (the owners' accumulators when the tables are sharded)
template <int E, int H1, int H2, int H3, int ACT>
__global__ void __launch_bounds__(NT) tc_bwd1(const Args A, const float* __restrict__ img, int n_tiles, unsigned int* ticket) {
  using L = Layout<E, H1, H2, H3>; using AC = Acc<H1, H2>; using I = Img<E, H1, H2, H3>;
  constexpr int K0 = 2 * E, MWORDS = K0 / 32;
  constexpr int WCOL = K0;                                 // TMEM: [0, K0) dx0, [WCOL, WCOL + H1) dW1
  constexpr int TCOLS = 256;
  uint8_t* sm = smem_base();
  uint8_t* Xm = sm;                                        // x0 (after dropout), MN view [K0/32][128][128 B]
  uint8_t* Zk = Xm + TS * K0 * 4;                          // dz1, K-major view [128][H1]
  uint8_t* Zm = Zk + TS * pad32(H1) * 4;                   // dz1, MN view
  uint8_t* Ws = Zm + TS * pad32(H1) * 4;                   // W1 image [K0 rows][pad32(H1)]
  uint32_t* masks = reinterpret_cast<uint32_t*>(Ws + K0 * pad32(H1) * 4);   // [128][MWORDS]
  float* mean1 = reinterpret_cast<float*>(masks + TS * MWORDS); float* rstd1 = mean1 + H1; float* gam1 = rstd1 + H1;
  float* sdy = gam1 + H1; float* sdyx = sdy + H1;
  __shared__ Ctl ctl;
  __shared__ int32_t ids_s[2][2 * TS];
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  Stamper stamp(128, 64);
  stamp();
  const uint32_t tmem = tc_begin<TCOLS>(ctl);
  copy16(Ws, img + I::W1, K0 * pad32(H1));
  copy_small<H1>(gam1, A.dense.w + L::g1);
  bn_prepare<H1>(mean1, rstd1, A.acc + AC::s1, A.acc + AC::q1, nullptr, nullptr, A.B, true);
  for (int f = t; f < H1; f += NT) {
    sdy[f] = float(A.acc[AC::d1 + f] / double(A.B));
    sdyx[f] = float(A.acc[AC::e1 + f] / double(A.B));
    if (blockIdx.x == 0) {                                  // BN1 parameter gradients
      A.dense.g[L::be1 + f] += float(A.acc[AC::d1 + f]);
      A.dense.g[L::g1 + f] += float(A.acc[AC::e1 + f]);
    }
  }
  __syncthreads();
  uint32_t phase = 0;
  int it = 0;
  float db_acc = 0.f;                                      // this thread's bias-gradient feature, summed over the CTA's tiles
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
    const int64_t b0 = int64_t(tile) * TS;
    const int valid = int((A.B - b0) < int64_t(TS) ? (A.B - b0) : int64_t(TS));
    stamp();
    // three independent memory phases, issued back to back so their DRAM latencies overlap: the h1 / dy1 columns of
    // the tile (no dependence on the ids), the ids (prefetched into the other half of ids_s during the previous tile),
    // the embedding rows; the dropout bits are drawn while the first loads fly
    float hv[H1 / 2], dv[H1 / 2];
    dz_issue<H1>(hv, dv, A.h1, A.dy1, A.B, b0, valid);
    const int32_t* ids_c = ids_s[it & 1];
    if (it == 0) load_tile_ids(ids_s[0], A, b0, valid);
    if (A.dropout) {
      const int s = t & (TS - 1), hf = t >> 7;
      for (int c = hf * (K0 / 32); c < (hf + 1) * (K0 / 32); ++c) {
        const uint32_t bits = s < valid ? drop16_bits(uint64_t(A.first_index + b0 + s), c, 0, A.drop_seed, A.drop_epoch) : 0u;
        reinterpret_cast<uint16_t*>(masks + s * MWORDS)[c] = uint16_t(bits);
      }
    }
    __syncthreads();
    stamp();
    float4 xv[2 * (TS / (NT / (E / 4)))];
    gather_x0_issue<E>(xv, A, ids_c, valid);
    {                                                       // next tile's ids
      const int64_t nb0 = int64_t(tile + gridDim.x) * TS;
      if (tile + int(gridDim.x) < n_tiles) {
        const int nvalid = int((A.B - nb0) < int64_t(TS) ? (A.B - nb0) : int64_t(TS));
        load_tile_ids(ids_s[(it + 1) & 1], A, nb0, nvalid);
      }
    }
    dz_store<H1, ACT>(Zk, Zm, hv, dv, mean1, rstd1, gam1, sdy, sdyx, valid);
    stamp();
    gather_x0_store<E, 1>(Xm, xv, A, masks);
    NTC_OPERANDS_READY();
    stamp();
    if (t == 0) {
      issue_gemm<128, K0, 0, 0>(tmem, tc::smem_u32(Zk), TS, tc::smem_u32(Ws), K0, H1, false);             // dx0
      constexpr uint32_t idesc = tc::idesc_tf32_f32(K0, H1, 1, 1);
      for (int ks = 0; ks < TS / 8; ++ks) {                                                                 // dW1 (+)= x0^T dz1
        const uint64_t ad = tc::smem_desc_sw128_base32(tc::smem_u32(Xm) + uint32_t(ks) * 1024u, TS * 128u, 512);
        const uint64_t bd = tc::smem_desc_sw128_base32(tc::smem_u32(Zm) + uint32_t(ks) * 1024u, TS * 128u, 512);
        tc::mma_tf32_ss(tmem + WCOL, ad, bd, idesc, (ks != 0 || it != 0) ? 1u : 0u);
      }
      tc::mma_commit(tc::smem_u32(&ctl.bar));
    }
    if (t < H1) {                                           // db1 on the CUDA cores meanwhile
      float sacc = 0.f;
      for (int r = 0; r < TS; ++r) sacc += *reinterpret_cast<const float*>(Zk + km_off16(TS, r, t >> 2) + (t & 3) * 4);
      db_acc += sacc;                                       // one atomic per feature per CTA, after the last tile
    }
    tc::mbar_wait(tc::smem_u32(&ctl.bar), phase);
    phase ^= 1u;
    tc::fence_after_sync();
    stamp();
    // epilogue: warps 0..3 read the user half of dx0 out of TMEM, warps 4..7 the item half (lane = sample) and park it,
    // masked, in the x0 tile (free once the products have completed; 16-byte chunk ^ (sample & 7): conflict-free both
    // ways).  The REDs then go out ROW-contiguous, 16 lanes per 256-byte row: with lane = sample every RED instruction
    // touched 32 different lines and the epilogue was half of the tile's time (profiles/r02_neumf_tc_trace.txt).
    {
      const int s = (warp & 3) * 32 + lane, tab = warp >> 2;
      const bool ok = s < valid;
      for (int cc = 0; cc < E; cc += 32) {
        float v[32];
        tmem_load32(tmem, warp, tab * E + cc, v);
        const int f0 = tab * E + cc;
        const uint32_t m = !ok ? 0u : (A.dropout ? masks[s * MWORDS + (f0 >> 5)] : 0xFFFFFFFFu);
        const float sc = A.dropout ? kDropScale : 1.f;
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          float4 g4;
          g4.x = ((m >> (j + 0)) & 1u) ? v[j + 0] * sc : 0.f; g4.y = ((m >> (j + 1)) & 1u) ? v[j + 1] * sc : 0.f;
          g4.z = ((m >> (j + 2)) & 1u) ? v[j + 2] * sc : 0.f; g4.w = ((m >> (j + 3)) & 1u) ? v[j + 3] * sc : 0.f;
          if (cc + j < E) *reinterpret_cast<float4*>(Xm + s * (K0 * 4) + ((((f0 + j) >> 2) ^ (s & 7)) << 4)) = g4;
        }
      }
    }
    __syncthreads();
    {
      constexpr int LPR = E / 4, RPP = NT / LPR, NPASS = 2 * TS / RPP;
      const int c4 = t % LPR, q = t / LPR;
#pragma unroll 4
      for (int p = 0; p < NPASS; ++p) {
        const int pr = p * RPP + q, s = pr & (TS - 1), tab = pr / TS;
        if (s < valid) {
          const RowRef rr = locate<E>(tab == 0 ? A.uMLP : A.iMLP, ids_c[tab * TS + s]);
          const float4 g4 = *reinterpret_cast<const float4*>(Xm + s * (K0 * 4) + (((tab * LPR + c4) ^ (s & 7)) << 4));
          red_add_f4(rr.g + 4 * c4, g4);
          if (c4 == 0) mark_row(rr);
        }
      }
    }
    stamp();
    tc::fence_before_sync();
    __syncthreads();                                        // tiles and masks may be overwritten by the next iteration
  }
  stamp();
  if (it > 0) {                                             // flush dW1: lane = row k, this warp's column half
    tc::fence_after_sync();
    constexpr int HC = H1 / 2;
    const int k = row_of_lane<K0>(( warp & 3) * 32 + lane), c0 = (warp >> 2) * HC;
    float v[32];
    tmem_load32(tmem, warp, WCOL + c0, v);
    if (k >= 0)                                             // 16-byte REDs: a quarter of the L2 atomic operations
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        if (j < HC) red_add_f4(A.dense.g + L::W1 + k * H1 + c0 + j, make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
    if (t < H1) atomicAdd(A.dense.g + L::b1 + t, db_acc);
  }
  // last CTA: BN moving statistics, loss output, accumulator reset
  __syncthreads();
  __shared__ bool last;
  if (t == 0) { __threadfence(); last = atomicAdd(ticket, 1u) == gridDim.x - 1; }
  __syncthreads();
  stamp();
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
  tc_end<TCOLS>(tmem);
}

template <int H1, int H2>
__global__ void tc_finish_eval(double* acc, int64_t B, float* loss_out) {
  using AC = Acc<H1, H2>;
  if (threadIdx.x == 0 && loss_out) loss_out[0] = float(acc[AC::loss] / double(B));
  __syncthreads();
  for (int j = threadIdx.x; j < AC::total; j += blockDim.x) acc[j] = 0.0;
}

template <int E, int H1, int H2, int H3, int ACT>
int run(brk_ctx* ctx, const Args& A, cudaStream_t st) {
  using I = Img<E, H1, H2, H3>;
  constexpr int K0 = 2 * E, N3 = I::N3;
  if (ctx->neumf_img_floats < size_t(I::total)) {
    if (ctx->neumf_img) BRK_CUDA(cudaFree(ctx->neumf_img));
    ctx->neumf_img = nullptr; ctx->neumf_img_floats = 0;
    BRK_CUDA(cudaMalloc(&ctx->neumf_img, size_t(I::total) * sizeof(float)));
    ctx->neumf_img_floats = size_t(I::total);
  }
  float* img = ctx->neumf_img;
  const int n_tiles = int((A.B + TS - 1) / TS);
  auto by = [](size_t floats) { return floats * sizeof(float) + 1024; };
  const size_t smA = by(size_t(TS) * K0 + H1 * pad32(K0) + H1 + TS * (K0 / 32));
  const size_t smB = by(size_t(TS) * pad32(H1) + H2 * pad32(H1) + H2 + 4 * H1);
  const size_t smC = by(size_t(TS) * pad32(H2) + N3 * pad32(H2) + H2 * H3 + ((H3 + 3) & ~3) + ((H3 + 5) & ~3) + 2 * size_t(H2) * SP +
                        size_t(H3) * SP + size_t(TS) * (H3 + 1) + 2 * TS + 4 * H2);
  const size_t smD = by(size_t(TS) * pad32(H1) + 2 * size_t(TS) * pad32(H2) + H1 * pad32(H2) + size_t(H1) * SP + 4 * H1 + 5 * H2);
  const size_t smE = by(size_t(TS) * K0 + 2 * size_t(TS) * pad32(H1) + K0 * pad32(H1) + TS * (K0 / 32) + 5 * H1);
  // the shared-memory opt-in is per device: set it for the current one on every call; the occupancy caps below are
  // properties of the kernels, computed once
  BRK_CUDA(cudaFuncSetAttribute(tc_fwd1<E, H1, H2, H3, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smA)));
  BRK_CUDA(cudaFuncSetAttribute(tc_fwd2<E, H1, H2, H3, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smB)));
  BRK_CUDA(cudaFuncSetAttribute(tc_head<E, H1, H2, H3, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smC)));
  BRK_CUDA(cudaFuncSetAttribute(tc_bwd2<E, H1, H2, H3, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smD)));
  BRK_CUDA(cudaFuncSetAttribute(tc_bwd1<E, H1, H2, H3, ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smE)));
  static bool occ_done = false;
  static int occ_d = 0, occ_e = 0, occ_c = 0;
  if (!occ_done) {
    // persistent grids: CTAs per SM by shared memory (227 KB), registers (2 x 256 threads) and TMEM (512 columns:
    // bwd2 allocates 128, bwd1 256 per CTA)
    occ_d = int((227 * 1024) / (smD + 1024)); if (occ_d > 2) occ_d = 2;
    occ_e = int((227 * 1024) / (smE + 1024)); if (occ_e > 2) occ_e = 2;
    {
      // tc_head: CTAs per SM from its own resource use.  (cudaOccupancyMaxActiveBlocksPerMultiprocessor answers 1 for
      // this kernel at 128 registers x 256 threads + 80 KB although two CTAs do run side by side -- in-kernel stamps,
      // profiles/r02_neumf_tc_trace.txt -- and the persistent tile loop is correct for any grid.)
      cudaFuncAttributes fa;
      BRK_CUDA(cudaFuncGetAttributes(&fa, tc_head<E, H1, H2, H3, ACT>));
      const int by_smem = int((227 * 1024) / (smC + fa.sharedSizeBytes + 1024));
      const int by_regs = 65536 / (((fa.numRegs + 7) & ~7) * NT);
      occ_c = by_smem < by_regs ? by_smem : by_regs;
      if (occ_c > 4) occ_c = 4;
      if (occ_c < 1) occ_c = 1;
    }
    BRK_REQUIRE(occ_d > 0 && occ_e > 0 && occ_c > 0, BRK_E_STATE, "brk_neumf_step: tensor-core kernels do not fit");
    occ_done = true;
  }
  {
    static unsigned long long* trace_set = nullptr;
    const char* tr = getenv("BRK_NTC_TRACE");
    unsigned long long* want = tr ? reinterpret_cast<unsigned long long*>(strtoull(tr, nullptr, 16)) : nullptr;
    if (want != trace_set) { BRK_CUDA(cudaMemcpyToSymbolAsync(g_trace, &want, sizeof(want), 0, cudaMemcpyHostToDevice, st)); trace_set = want; }
  }
  prep_images<E, H1, H2, H3><<<(I::total + 255) / 256, 256, 0, st>>>(A.dense.w, img);
  tc_fwd1<E, H1, H2, H3, ACT><<<n_tiles, NT, smA, st>>>(A, img);
  tc_fwd2<E, H1, H2, H3, ACT><<<n_tiles, NT, smB, st>>>(A, img);
  {
    const int gc = n_tiles < occ_c * ctx->sm_count ? n_tiles : occ_c * ctx->sm_count;
    tc_head<E, H1, H2, H3, ACT><<<gc, NT, smC, st>>>(A, img, n_tiles);
  }
  if (A.training) {
    const int gd = n_tiles < occ_d * ctx->sm_count ? n_tiles : occ_d * ctx->sm_count;
    const int ge = n_tiles < occ_e * ctx->sm_count ? n_tiles : occ_e * ctx->sm_count;
    tc_bwd2<E, H1, H2, H3, ACT><<<gd, NT, smD, st>>>(A, img, n_tiles);
    tc_bwd1<E, H1, H2, H3, ACT><<<ge, NT, smE, st>>>(A, img, n_tiles, ctx->tickets + 5);
  } else {
    tc_finish_eval<H1, H2><<<1, 128, 0, st>>>(A.acc, A.B, A.loss_out);
  }
  BRK_LAUNCH_CHECK();
  return 0;
}

}  // namespace ntc

// mode = a_mn | (b_mn << 1); M in {64, 128}; N in {16, 32, 64, 128}.  Test hook (tests/test_gpu_tc.py).
extern "C" int brk_tc_selftest(brk_ctx* ctx, int32_t M, int32_t N, int32_t K, int32_t mode, const float* A, int32_t a_rows,
                               int32_t a_cols, const float* B, int32_t b_rows, int32_t b_cols, float* out, void* stream) {
  BRK_REQUIRE(ctx && A && B && out, BRK_E_ARG, "brk_tc_selftest: null argument");
  BRK_REQUIRE(a_cols % 32 == 0 && b_cols % 32 == 0 && a_rows % 8 == 0 && b_rows % 8 == 0 && K % 8 == 0, BRK_E_ARG,
              "brk_tc_selftest: shapes");
  const size_t smem = size_t(a_rows) * a_cols * 4 + size_t(b_rows) * b_cols * 4 + 2048;
  cudaStream_t st = (cudaStream_t)stream;
#define BRK_TC_CASE(M_, N_, AM_, BM_)                                                                         \
  if (M == M_ && N == N_ && mode == (AM_ | (BM_ << 1))) {                                                     \
    BRK_CUDA(cudaFuncSetAttribute(ntc::selftest_kernel<M_, N_, AM_, BM_>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem))); \
    ntc::selftest_kernel<M_, N_, AM_, BM_><<<1, ntc::kThreads, smem, st>>>(A, a_rows, a_cols, B, b_rows, b_cols, K, out); \
    BRK_LAUNCH_CHECK();                                                                                       \
    return 0;                                                                                                 \
  }
  BRK_TC_CASE(128, 64, 0, 0) BRK_TC_CASE(128, 32, 0, 0) BRK_TC_CASE(128, 16, 0, 0) BRK_TC_CASE(128, 128, 0, 0)
  BRK_TC_CASE(128, 64, 1, 1) BRK_TC_CASE(128, 32, 1, 1) BRK_TC_CASE(64, 32, 1, 1) BRK_TC_CASE(64, 16, 1, 1)
  BRK_TC_CASE(64, 32, 0, 0) BRK_TC_CASE(128, 64, 1, 0) BRK_TC_CASE(128, 64, 0, 1)
#undef BRK_TC_CASE
  brk_set_error("brk_tc_selftest: no instance for M=%d N=%d mode=%d", M, N, mode);
  return BRK_E_ARG;
}

// Tensor-core NeuMF step (TF32 operands): returns 0 when the spec was handled, 1 when it is not one of the
// built instances.  Called by brk_neumf_step / brk_neumf_step_sharded when the model asks for it.
void brk_neumf_fill_args(v2::Args& A, const brk_neumf_model* m, const brk_neumf_shards* sh, const int32_t* u,
                         const int32_t* i, const float* y, int64_t batch, int64_t global_batch, int64_t first_index,
                         int32_t training, uint32_t dropout_seed, uint32_t dropout_epoch, const brk_neumf_workspace* ws,
                         float* out, float* loss_out);

int brk_neumf_step_tc(brk_ctx* ctx, const brk_neumf_model* m, const brk_neumf_shards* sh, const int32_t* u,
                      const int32_t* i, const float* y, int64_t batch, int64_t global_batch, int64_t first_index,
                      int32_t training, uint32_t dropout_seed, uint32_t dropout_epoch, const brk_neumf_workspace* ws,
                      float* out, float* loss_out, cudaStream_t st, int* rc_out) {
  v2::Args A;
  brk_neumf_fill_args(A, m, sh, u, i, y, batch, global_batch, first_index, training, dropout_seed, dropout_epoch, ws, out, loss_out);
#define BRK_TC_SPEC(E_, A_, B_, C_)                                                                        \
  if (m->E == E_ && m->H1 == A_ && m->H2 == B_ && m->H3 == C_) {                                            \
    *rc_out = m->act == 0 ? ntc::run<E_, A_, B_, C_, 0>(ctx, A, st) : ntc::run<E_, A_, B_, C_, 1>(ctx, A, st); \
    return 0;                                                                                               \
  }
  BRK_TC_SPEC(64, 64, 32, 16)
  BRK_TC_SPEC(32, 32, 16, 8)
#undef BRK_TC_SPEC
  return 1;
}
