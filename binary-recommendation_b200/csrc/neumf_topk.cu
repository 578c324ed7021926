// Full-catalog NeuMF top-K in one launch: the model's inference score of every (user, item) pair, fused with the
// per-user selection of score_topk_kernel (topk.cu), so that no score reaches HBM.
//
// NeuMF's first layer factors over the concatenated input x0 = [uMLP[u], iMLP[i]]:
//   x0 W1 + b1 = uMLP[u] W1[0:E] + (iMLP[i] W1[E:2E] + b1) = A_u + B_i,
// so the caller computes A [U, H1] once per query and B [I, H1] once per index (TF32 products, brk_gemm_tf32), and
// this kernel is left with, per pair: z1 = A_u + B_i, y1 = BN1(relu(z1)), the layer-2 product (H1 x H2), BN2, the
// layer-3 product (H2 x H3), the head and the sigmoid.  The two products run on tcgen05 (kind::tf32, fp32
// accumulation in TMEM); everything else is fp32 on the CUDA cores.
//
// CTA = 128 users, one per thread and TMEM lane (4 warps; thread 0 also issues the MMAs).  A thread keeps its user's
// A_u, its MF row (times the head's MF weights for the Hadamard GMF) and its running top-K list in registers (the MF
// row of numFactor 64 in shared memory).  Items stream in
// ascending id, G at a time: each thread writes its row of the G layer-2 A tiles (K-major, SWIZZLE_128B), one thread
// issues the G layer-2 MMAs into G TMEM slots, the threads read z2 back and write the layer-3 A tiles over the
// consumed layer-2 ones, then the G layer-3 MMAs, then z3 -> head -> sigmoid -> compare with the row's k-th best.
// The item rows (B_i, iMF[i]) of the next group are loaded while the current one is computed.  Several CTAs per SM
// overlap one CTA's MMA round trips with another's CUDA-core work.
//
// Selection: strict '>' against the row's k-th best while items arrive in ascending id keeps the lower id on ties;
// candidates are voted on per warp and inserted with topk_insert (topk_select.cuh).  Exclusions (EXCL): one monotone
// cursor per thread into its row's ascending list, advanced only on the candidate path.  blockIdx.y splits the item
// range; the partial lists are merged by brk_topk_merge (score desc, id asc), identical to one unsplit scan.
#include "common.cuh"
#include "tc.cuh"
#include "tc_tiles.cuh"
#include "topk_select.cuh"
#include <limits.h>
#include <math_constants.h>

namespace ntk {

using ntc::issue_gemm;
using ntc::km_off16;
using ntc::pad32;

constexpr int NT = 128;             // threads = users per CTA = TMEM lanes
constexpr int TCOLS = 128;          // TMEM columns per CTA
constexpr int kMaxSplits = 32;
constexpr float kBnEps = 1e-3f;

template <int E_, int EMF_, int H1_, int H2_, int H3_, int BN_, int HAD_>
struct Spec {
  static constexpr int E = E_, EMF = EMF_, H1 = H1_, H2 = H2_, H3 = H3_, BN = BN_, HAD = HAD_;
  static constexpr int N3 = H3 < 16 ? 16 : H3, HM = HAD ? EMF : 1;
  static constexpr int SLOT = H2 + N3;                     // TMEM columns per item: z2, then z3
  static constexpr int G = TCOLS / SLOT;                   // items per group
  // dense parameter block (include/brk_b200.h): W4 has H3 + HM rows
  static constexpr int ob1 = 2 * E * H1, og1 = ob1 + H1, obe1 = og1 + H1;
  static constexpr int oW2 = obe1 + H1, ob2 = oW2 + H1 * H2, og2 = ob2 + H2, obe2 = og2 + H2;
  static constexpr int oW3 = obe2 + H2, ob3 = oW3 + H2 * H3, oW4 = ob3 + H3, ob4 = oW4 + H3 + HM;
  // shared memory (bytes from the 1024-aligned base): G operand tiles (layer 2, then layer 3 in the same place), the
  // two weight images, then floats: s1 t1 [H1], b2 s2 t2 [H2], b3 [H3], w4 [H3 + HM + 1], item rows [2][G][H1 + EMF]
  static constexpr int TILE = NT * (pad32(H1) > pad32(H2) ? pad32(H1) : pad32(H2)) * 4;
  static constexpr int oW2t = G * TILE, oW3t = oW2t + H2 * pad32(H1) * 4, oF = oW3t + N3 * pad32(H2) * 4;
  static constexpr int IROW = H1 + EMF;
  // the user's MF row stays in registers up to 32 floats; wider (the scalar Dot at numFactor 64) it lives in shared
  // memory, [EMF][128] (thread-major: conflict-free), so that A_u and the list keep their registers
  static constexpr bool GSM = EMF > 32;
  static constexpr int nF = 2 * H1 + 3 * H2 + H3 + ((H3 + HM + 1 + 3) & ~3) + 2 * G * IROW;
  static constexpr size_t smem = size_t(oF) + size_t(nF) * 4 + 1024 + NT * G * 4 + (GSM ? NT * EMF * 4 : 0);   // + scratch
  static_assert(H1 % 32 == 0 && H2 % 16 == 0 && H2 <= 32 && H3 % 8 == 0 && EMF % 4 == 0, "widths");
  static_assert(G >= 1 && G <= 8 && (G * IROW) % 4 == 0, "item group");
};

struct Params {
  const float* A;                    // [U, H1] user side
  const int32_t* users;              // [U] rows of uMF
  const float* uMF;                  // [numUser, EMF]
  const float* B;                    // [I, H1] item side (b1 included)
  const float* iMF;                  // [I, EMF] MF rows of the indexed items
  const float* dense;                // the model's dense block
  const float* bn;                   // moving mean1, var1, mean2, var2
  int64_t U, I;
  int32_t k, id_offset;
  int32_t groups_per_split, n_groups;
  float* out_vals;                   // [n_splits, U, k]
  int32_t* out_ids;
  const int64_t* excl_indptr;        // EXCL: [U + 1]
  const int32_t* excl_ids;
};

template <int N>
__device__ __forceinline__ void tmem_ld(uint32_t taddr, float (&v)[N]) {
  static_assert(N == 16 || N == 32, "TMEM read width");
  if constexpr (N == 16) {
    uint32_t r[16];
    tc::tmem_ld_32x32_x16(taddr, r);
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]);
  } else {
    uint32_t r[32];
    tc::tmem_ld_32x32_issue(taddr, r);
    tc::tmem_ld_wait(r);
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
  }
}

// operands written with st.shared -> visible to the tensor core; earlier tcgen05.ld of every thread ordered before
#define NTK_OPERANDS_READY() \
  do { tc::fence_proxy_async_smem(); tc::fence_before_sync(); __syncthreads(); tc::fence_after_sync(); } while (0)

template <class S, int K_CAP, bool EXCL>
__global__ void __launch_bounds__(NT, 2) neumf_topk_kernel(const Params P) {
  constexpr int H1 = S::H1, H2 = S::H2, H3 = S::H3, N3 = S::N3, EMF = S::EMF, HM = S::HM, G = S::G, IROW = S::IROW;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* W2t = sm + S::oW2t;                             // [H2 rows][pad32(H1)] K-major image of W2^T
  uint8_t* W3t = sm + S::oW3t;                             // [N3 rows][pad32(H2)] K-major image of W3^T, rows >= H3 zero
  float* s1 = reinterpret_cast<float*>(sm + S::oF);
  float* t1 = s1 + H1;
  float* b2 = t1 + H1; float* s2 = b2 + H2; float* t2 = s2 + H2;
  float* b3 = t2 + H2;
  float* w4 = b3 + H3;                                      // [H3 + HM] head weights, then b4
  float* items = w4 + ((H3 + HM + 1 + 3) & ~3);             // [2][G][H1 + EMF]: B rows, then iMF rows
  float* scratch = items + 2 * G * IROW;                    // [G][128] scores of a group (candidate path)
  float* gsm = scratch + G * NT;                            // GSM: [EMF][128] MF rows of the CTA's users
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_slot;

  const int t = threadIdx.x, warp = t >> 5;
  const int64_t row = int64_t(blockIdx.x) * NT + t;
  const bool live = row < P.U;
  const int g_begin = blockIdx.y * P.groups_per_split;
  const int g_end = min(P.n_groups, g_begin + P.groups_per_split);
  const float* D = P.dense;

  if (t == 0) { tc::mbar_init(tc::smem_u32(&bar), 1); tc::fence_barrier_init(); }
  if (warp == 0) tc::tmem_alloc<TCOLS>(tc::smem_u32(&tmem_slot));
  // weight images and per-feature constants; BatchNorm folded into scale / shift with the moving statistics
  for (int idx = t; idx < H2 * pad32(H1); idx += NT) {
    const int r = idx / pad32(H1), c = idx % pad32(H1);
    *reinterpret_cast<float*>(W2t + km_off16(H2, r, c >> 2) + (c & 3) * 4) = c < H1 ? D[S::oW2 + c * H2 + r] : 0.f;
  }
  for (int idx = t; idx < N3 * pad32(H2); idx += NT) {
    const int r = idx / pad32(H2), c = idx % pad32(H2);
    *reinterpret_cast<float*>(W3t + km_off16(N3, r, c >> 2) + (c & 3) * 4) = (c < H2 && r < H3) ? D[S::oW3 + c * H3 + r] : 0.f;
  }
  for (int f = t; f < H1; f += NT) {
    float sc = 1.f, sh = 0.f;
    if (S::BN) {
      const float rstd = 1.0f / sqrtf(P.bn[H1 + f] + kBnEps);
      sc = D[S::og1 + f] * rstd; sh = D[S::obe1 + f] - P.bn[f] * sc;
    }
    s1[f] = sc; t1[f] = sh;
  }
  for (int f = t; f < H2; f += NT) {
    float sc = 1.f, sh = 0.f;
    if (S::BN) {
      const float rstd = 1.0f / sqrtf(P.bn[2 * H1 + H2 + f] + kBnEps);
      sc = D[S::og2 + f] * rstd; sh = D[S::obe2 + f] - P.bn[2 * H1 + f] * sc;
    }
    b2[f] = D[S::ob2 + f]; s2[f] = sc; t2[f] = sh;
  }
  for (int f = t; f < H3; f += NT) b3[f] = D[S::ob3 + f];
  for (int f = t; f < H3 + HM + 1; f += NT) w4[f] = D[S::oW4 + f];

  // item rows of group g: G rows of B and of iMF, zero past I; one float4 per thread at most
  constexpr int NV = G * IROW / 4;
  static_assert(NV <= NT, "item group loads");
  auto load_group = [&](int g) -> float4 {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t < NV && g < g_end) {
      const int e = 4 * t;
      const int64_t i0 = int64_t(g) * G;
      if (e < G * H1) {
        const int64_t it = i0 + e / H1;
        if (it < P.I) v = __ldg(reinterpret_cast<const float4*>(P.B + it * H1 + e % H1));
      } else {
        const int e2 = e - G * H1;
        const int64_t it = i0 + e2 / EMF;
        if (it < P.I) v = __ldg(reinterpret_cast<const float4*>(P.iMF + it * EMF + e2 % EMF));
      }
    }
    return v;
  };
  auto store_group = [&](int buf, float4 v) {
    if (t < NV) *reinterpret_cast<float4*>(items + buf * G * IROW + 4 * t) = v;
  };
  store_group(0, load_group(g_begin));

  // this thread's user: A_u, the GMF vector, the list
  float a[H1], gv[S::GSM ? 1 : EMF];
  {
    const int32_t uid = live ? __ldg(P.users + row) : 0;
#pragma unroll
    for (int c4 = 0; c4 < H1 / 4; ++c4) {
      const float4 v = live ? __ldg(reinterpret_cast<const float4*>(P.A + row * H1) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
      a[4 * c4] = v.x; a[4 * c4 + 1] = v.y; a[4 * c4 + 2] = v.z; a[4 * c4 + 3] = v.w;
    }
#pragma unroll
    for (int c4 = 0; c4 < EMF / 4; ++c4) {
      const float4 v = live ? __ldg(reinterpret_cast<const float4*>(P.uMF + int64_t(uid) * EMF) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
      if constexpr (S::GSM) {
        gsm[(4 * c4) * NT + t] = v.x; gsm[(4 * c4 + 1) * NT + t] = v.y; gsm[(4 * c4 + 2) * NT + t] = v.z; gsm[(4 * c4 + 3) * NT + t] = v.w;
      } else {
        gv[4 * c4] = v.x; gv[4 * c4 + 1] = v.y; gv[4 * c4 + 2] = v.z; gv[4 * c4 + 3] = v.w;
      }
    }
  }
  float vals[K_CAP]; int32_t ids[K_CAP];
#pragma unroll
  for (int j = 0; j < K_CAP; ++j) { vals[j] = -CUDART_INF_F; ids[j] = -1; }
  float thr = -CUDART_INF_F;
  // exclusion cursor: the first listed id >= this split's first id; rows >= U get an empty list
  const int32_t* cur = nullptr; int32_t left = 0, next = INT_MAX;
  if constexpr (EXCL) {
    if (live) {
      int64_t pos = P.excl_indptr[row], end = P.excl_indptr[row + 1];
      const int64_t first = int64_t(g_begin) * G + P.id_offset;
      int64_t hi = end;
      while (pos < hi) {
        const int64_t mid = pos + ((hi - pos) >> 1);
        if (P.excl_ids[mid] < first) pos = mid + 1; else hi = mid;
      }
      const int64_t n = end - pos;
      cur = P.excl_ids + pos;
      left = int32_t(n < INT_MAX ? n : INT_MAX);
      next = pos < end ? P.excl_ids[pos] : INT_MAX;
    }
  }

  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  if constexpr (S::HAD) {                                   // Hadamard GMF: uMF[u] times the head's MF weights
#pragma unroll
    for (int f = 0; f < EMF; ++f) gv[f] *= w4[H3 + f];
  }
  const uint32_t tmem = tmem_slot;
  const uint32_t tlane = tmem + (uint32_t(warp * 32) << 16);
  const uint32_t sm_u32 = tc::smem_u32(sm);
  uint32_t phase = 0;

  for (int g = g_begin; g < g_end; ++g) {
    const int buf = (g - g_begin) & 1;
    const float* it_rows = items + buf * G * IROW;
    const float4 pre = load_group(g + 1);                   // next group's rows, in flight during this one
    // ---- layer 1 -> layer-2 A tiles: y1 = BN1(relu(A_u + B_i)) ----
    // (the item loops are not unrolled: one item's temporaries live at a time, next to A_u, the GMF vector and the list)
#pragma unroll 1
    for (int j = 0; j < G; ++j) {
      uint8_t* tile = sm + j * S::TILE;
#pragma unroll
      for (int c4 = 0; c4 < H1 / 4; ++c4) {
        const float4 b = *reinterpret_cast<const float4*>(it_rows + j * H1 + 4 * c4);
        const float4 sc = *reinterpret_cast<const float4*>(s1 + 4 * c4);
        const float4 sh = *reinterpret_cast<const float4*>(t1 + 4 * c4);
        float4 y;
        y.x = fmaf(fmaxf(a[4 * c4] + b.x, 0.f), sc.x, sh.x);
        y.y = fmaf(fmaxf(a[4 * c4 + 1] + b.y, 0.f), sc.y, sh.y);
        y.z = fmaf(fmaxf(a[4 * c4 + 2] + b.z, 0.f), sc.z, sh.z);
        y.w = fmaf(fmaxf(a[4 * c4 + 3] + b.w, 0.f), sc.w, sh.w);
        *reinterpret_cast<float4*>(tile + km_off16(NT, t, c4)) = y;
      }
    }
    NTK_OPERANDS_READY();
    if (t == 0) {
#pragma unroll 1
      for (int j = 0; j < G; ++j)
        issue_gemm<128, H2, 0, 0>(tmem + j * S::SLOT, sm_u32 + j * S::TILE, NT, sm_u32 + S::oW2t, H2, H1, false);
      tc::mma_commit(tc::smem_u32(&bar));
    }
    tc::mbar_wait(tc::smem_u32(&bar), phase); phase ^= 1u;
    tc::fence_after_sync();
    // ---- z2 -> y2 = BN2(relu(z2 + b2)) -> layer-3 A tiles (over the consumed layer-2 tiles) ----
#pragma unroll 1
    for (int j = 0; j < G; ++j) {
      float z[H2];
      tmem_ld<H2>(tlane + j * S::SLOT, z);
      uint8_t* tile = sm + j * S::TILE;
#pragma unroll
      for (int c4 = 0; c4 < H2 / 4; ++c4) {
        float4 y;
        y.x = fmaf(fmaxf(z[4 * c4] + b2[4 * c4], 0.f), s2[4 * c4], t2[4 * c4]);
        y.y = fmaf(fmaxf(z[4 * c4 + 1] + b2[4 * c4 + 1], 0.f), s2[4 * c4 + 1], t2[4 * c4 + 1]);
        y.z = fmaf(fmaxf(z[4 * c4 + 2] + b2[4 * c4 + 2], 0.f), s2[4 * c4 + 2], t2[4 * c4 + 2]);
        y.w = fmaf(fmaxf(z[4 * c4 + 3] + b2[4 * c4 + 3], 0.f), s2[4 * c4 + 3], t2[4 * c4 + 3]);
        *reinterpret_cast<float4*>(tile + km_off16(NT, t, c4)) = y;
      }
    }
    store_group(buf ^ 1, pre);                              // read from the next group on, after the barrier below
    NTK_OPERANDS_READY();
    if (t == 0) {
#pragma unroll 1
      for (int j = 0; j < G; ++j)
        issue_gemm<128, N3, 0, 0>(tmem + j * S::SLOT + H2, sm_u32 + j * S::TILE, NT, sm_u32 + S::oW3t, N3, H2, false);
      tc::mma_commit(tc::smem_u32(&bar));
    }
    tc::mbar_wait(tc::smem_u32(&bar), phase); phase ^= 1u;
    tc::fence_after_sync();
    // ---- z3 -> head -> sigmoid, parked in shared memory; candidates against the row's k-th best ----
    uint32_t cand = 0u;
#pragma unroll 1
    for (int j = 0; j < G; ++j) {
      float z[N3];
      tmem_ld<N3>(tlane + j * S::SLOT + H2, z);
      float logit = w4[H3 + HM];
#pragma unroll
      for (int q = 0; q < H3; ++q) logit = fmaf(fmaxf(z[q] + b3[q], 0.f), w4[q], logit);
      const float* mi = it_rows + G * H1 + j * EMF;
      float mf = 0.f;
#pragma unroll
      for (int f = 0; f < EMF; f += 4) {
        const float4 m4 = *reinterpret_cast<const float4*>(mi + f);
        if constexpr (S::GSM) {
          mf = fmaf(gsm[f * NT + t], m4.x, mf); mf = fmaf(gsm[(f + 1) * NT + t], m4.y, mf);
          mf = fmaf(gsm[(f + 2) * NT + t], m4.z, mf); mf = fmaf(gsm[(f + 3) * NT + t], m4.w, mf);
        } else {
          mf = fmaf(gv[f], m4.x, mf); mf = fmaf(gv[f + 1], m4.y, mf); mf = fmaf(gv[f + 2], m4.z, mf); mf = fmaf(gv[f + 3], m4.w, mf);
        }
      }
      logit = S::HAD ? logit + mf : fmaf(mf, w4[H3], logit);   // Dot: the forward's fmaf(<uMF, iMF>, W4[H3], .)
      const float o = 1.0f / (1.0f + expf(-logit));
      scratch[j * NT + t] = o;
      cand |= (o > thr && int64_t(g) * G + j < P.I) ? (1u << j) : 0u;
    }
    if (__any_sync(0xffffffffu, cand)) {                    // rare once the lists have filled
#pragma unroll 1
      while (cand) {                                        // ascending j = ascending item id
        const int j = __ffs(cand) - 1;
        cand &= cand - 1;
        const float x = scratch[j * NT + t];
        const int32_t id = int32_t(int64_t(g) * G + j) + P.id_offset;
        if (x > thr) {
          if constexpr (EXCL) {
            while (next < id) next = (--left > 0) ? *++cur : INT_MAX;
            if (next == id) continue;
          }
          topk_insert<K_CAP>(vals, ids, x, id);
          thr = vals[K_CAP - 1];
        }
      }
    }
  }

  if (live) {
    float* ov = P.out_vals + (int64_t(blockIdx.y) * P.U + row) * P.k;
    int32_t* oi = P.out_ids + (int64_t(blockIdx.y) * P.U + row) * P.k;
#pragma unroll
    for (int j = 0; j < K_CAP; ++j)
      if (j < P.k) { ov[j] = vals[j]; oi[j] = ids[j]; }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc<TCOLS>(tmem);
}

// Item splits so that a few hundred users still fill every SM: at most kMaxSplits, each a whole number of groups.
// Without the group count (the workspace query does not know the model) it is the largest the launch may use.
int plan_splits(int slots, int64_t U, int n_groups) {
  const int64_t m_tiles = (U + NT - 1) / NT;
  int S = 1;
  if (m_tiles < slots) S = int((slots + m_tiles - 1) / m_tiles);
  if (S > kMaxSplits) S = kMaxSplits;
  if (n_groups > 0 && S > n_groups) S = n_groups;
  return S < 1 ? 1 : S;
}

template <class S, int K_CAP, bool EXCL>
int launch(brk_ctx* ctx, Params P, cudaStream_t st) {
  const int n_groups = int((P.I + S::G - 1) / S::G);
  const int splits = plan_splits(2 * ctx->sm_count, P.U, n_groups);
  P.groups_per_split = (n_groups + splits - 1) / splits;
  P.n_groups = n_groups;
  const int used = (n_groups + P.groups_per_split - 1) / P.groups_per_split;
  BRK_CUDA(cudaFuncSetAttribute(neumf_topk_kernel<S, K_CAP, EXCL>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(S::smem)));
  const dim3 grid(unsigned((P.U + NT - 1) / NT), unsigned(used));
  neumf_topk_kernel<S, K_CAP, EXCL><<<grid, NT, S::smem, st>>>(P);
  BRK_LAUNCH_CHECK();
  return used;
}

template <class S, bool EXCL>
int launch_k(brk_ctx* ctx, const Params& P, cudaStream_t st) {
  if (P.k <= 10) return launch<S, 10, EXCL>(ctx, P, st);
  if (P.k <= 16) return launch<S, 16, EXCL>(ctx, P, st);
  return launch<S, 32, EXCL>(ctx, P, st);
}

}  // namespace ntk

extern "C" int brk_topk_merge(brk_ctx* ctx, const float* part_vals, const int32_t* part_ids, int32_t n_parts, int64_t U,
                              int32_t k, float* out_vals, int32_t* out_ids, void* stream);

extern "C" int64_t brk_neumf_topk_workspace_bytes(brk_ctx* ctx, int64_t U, int64_t I, int32_t k) {
  if (!ctx || U <= 0 || I <= 0 || k <= 0) return 0;
  return int64_t(ntk::plan_splits(2 * ctx->sm_count, U, 0)) * U * k * 8;
}

namespace {

int neumf_score_topk(brk_ctx* ctx, const brk_neumf_model* m, const float* user_side, const int32_t* users, int64_t U,
                     const float* item_side, const float* item_mf, int64_t I, int32_t k, int32_t id_offset,
                     const int64_t* excl_indptr, const int32_t* excl_ids, float* out_vals, int32_t* out_ids,
                     void* workspace, int64_t workspace_bytes, void* stream) {
  BRK_REQUIRE(ctx && m && user_side && users && item_side && item_mf && out_vals && out_ids, BRK_E_ARG,
              "brk_neumf_score_topk: null argument");
  BRK_REQUIRE(m->uMF.w && m->dense.w && m->bn_moving, BRK_E_ARG, "brk_neumf_score_topk: model tables missing");
  BRK_REQUIRE(U > 0 && I > 0 && U < (int64_t(1) << 31) && I < (int64_t(1) << 31), BRK_E_ARG,
              "brk_neumf_score_topk: U=%lld I=%lld", (long long)U, (long long)I);
  BRK_REQUIRE(k >= 1 && k <= 32, BRK_E_ARG, "brk_neumf_score_topk: k=%d (1..32)", k);
  BRK_REQUIRE(id_offset >= 0 && int64_t(id_offset) + I + 8 < int64_t(INT_MAX), BRK_E_ARG,
              "brk_neumf_score_topk: id_offset=%d + I=%lld reaches INT_MAX", id_offset, (long long)I);
  BRK_REQUIRE(brk_aligned16(user_side) && brk_aligned16(item_side) && brk_aligned16(item_mf) && brk_aligned16(m->uMF.w) &&
              brk_aligned16(m->dense.w), BRK_E_ALIGN, "brk_neumf_score_topk: operands must be 16-byte aligned");
  const int emf = m->EMF > 0 ? m->EMF : m->E;
  const int bn = m->no_batch_norm ? 0 : 1;
  const bool excl = excl_indptr != nullptr;
  const int64_t S_max = ntk::plan_splits(2 * ctx->sm_count, U, 0);
  const int64_t need = S_max * U * k * 8;
  BRK_REQUIRE(workspace && workspace_bytes >= need, BRK_E_ARG,
              "brk_neumf_score_topk: workspace of %lld bytes needed, %lld given", (long long)need, (long long)workspace_bytes);
  ntk::Params P;
  P.A = user_side; P.users = users; P.uMF = m->uMF.w; P.B = item_side; P.iMF = item_mf;
  P.dense = m->dense.w; P.bn = m->bn_moving;
  P.U = U; P.I = I; P.k = k; P.id_offset = id_offset;
  P.groups_per_split = 0; P.n_groups = 0;
  float* pv = reinterpret_cast<float*>(workspace);
  int32_t* pi = reinterpret_cast<int32_t*>(pv + S_max * U * k);
  P.out_vals = pv; P.out_ids = pi;
  P.excl_indptr = excl_indptr; P.excl_ids = excl_ids;
  cudaStream_t st = (cudaStream_t)stream;
  int parts = 0;
  bool handled = false;
#define BRK_NTK_SPEC(TC_, E_, EMF_, A_, B_, C_, BN_, HAD_)                                                              \
  if (!handled && (TC_ < 0 || m->tensor_cores == TC_) && m->act == 0 && m->E == E_ && emf == EMF_ && m->H1 == A_ && m->H2 == B_ &&     \
      m->H3 == C_ && bn == BN_ && m->mf_mode == HAD_) {                                                                   \
    using S = ntk::Spec<E_, EMF_, A_, B_, C_, BN_, HAD_>;                                                                \
    parts = excl ? ntk::launch_k<S, true>(ctx, P, st) : ntk::launch_k<S, false>(ctx, P, st);                              \
    handled = true;                                                                                                      \
  }
  BRK_NTK_SPEC(1, 32, 32, 32, 16, 8, 1, 0)       // class graph, numFactor 32, tensor cores
  BRK_NTK_SPEC(1, 64, 64, 64, 32, 16, 1, 0)      // class graph, numFactor 64, tensor cores
  BRK_NTK_SPEC(-1, 32, 8, 32, 16, 8, 0, 1)       // He et al.: EMF 8, Hadamard GMF, no BatchNorm
#undef BRK_NTK_SPEC
  if (!handled) {
    brk_set_error("brk_neumf_score_topk: no instance for E=%d EMF=%d H=(%d,%d,%d) act=%d mf_mode=%d batch_norm=%d "
                  "tensor_cores=%d; built (relu): class graph (32;32,16,8) and (64;64,32,16) with tensor_cores = 1, He et "
                  "al. E=32 EMF=8 (32,16,8) Hadamard without BatchNorm -- other models rank through score_all",
                  m->E, emf, m->H1, m->H2, m->H3, m->act, m->mf_mode, bn, m->tensor_cores);
    return BRK_E_ARG;
  }
  if (parts < 0) return parts;                           // a launch error, already reported
  return brk_topk_merge(ctx, pv, pi, parts, U, k, out_vals, out_ids, stream);
}

}  // namespace

extern "C" int brk_neumf_score_topk(brk_ctx* ctx, const brk_neumf_model* m, const float* user_side, const int32_t* users,
                                    int64_t U, const float* item_side, const float* item_mf, int64_t I, int32_t k,
                                    int32_t id_offset, float* out_vals, int32_t* out_ids, void* workspace,
                                    int64_t workspace_bytes, void* stream) {
  return neumf_score_topk(ctx, m, user_side, users, U, item_side, item_mf, I, k, id_offset, nullptr, nullptr, out_vals,
                          out_ids, workspace, workspace_bytes, stream);
}

extern "C" int brk_neumf_score_topk_excl(brk_ctx* ctx, const brk_neumf_model* m, const float* user_side,
                                         const int32_t* users, int64_t U, const float* item_side, const float* item_mf,
                                         int64_t I, int32_t k, int32_t id_offset, const int64_t* excl_indptr,
                                         const int32_t* excl_ids, float* out_vals, int32_t* out_ids, void* workspace,
                                         int64_t workspace_bytes, void* stream) {
  BRK_REQUIRE(excl_indptr && excl_ids, BRK_E_ARG, "brk_neumf_score_topk_excl: null exclusion list");
  return neumf_score_topk(ctx, m, user_side, users, U, item_side, item_mf, I, k, id_offset, excl_indptr, excl_ids,
                          out_vals, out_ids, workspace, workspace_bytes, stream);
}
