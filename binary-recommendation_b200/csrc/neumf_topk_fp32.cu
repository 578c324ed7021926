// Full-catalog NeuMF top-K for the fp32 models in one launch: the inference score of every (user, item) pair of an
// fp32 NeuMF network of any width up to the caps below, computed on the CUDA cores and fused with the per-user
// selection, so that no score reaches HBM.  The tensor-core instances have their own kernel (neumf_topk.cu).
//
// The first layer factors as in neumf_topk.cu: x0 W1 + b1 = uMLP[u] W1[0:E] + (iMLP[i] W1[E:2E] + b1) = A_u + B_i,
// both halves fp32 products (brk_sgemm) supplied by the caller.  Per pair this kernel computes the rest of the fp32
// forward pass in inference mode, every sum in the order of the any-width forward (neumf_generic.cu):
//   y1 = BN1(act(A_u + B_i));  y2 = BN2(act(y1 W2 + b2));  h3 = act(y2 W3 + b3);
//   logit = h3 W4[0:H3] + MF term + b4;  score = 1 / (1 + expf(-logit)),
// BatchNorm with the moving statistics folded into one scale / shift per feature, the MF term W4[H3] <uMF, iMF> for
// the Dot head and sum_f (uMF[f] iMF[f]) W4[H3 + f] for the Hadamard head.
//
// CTA = 128 users, one per thread.  A_u and the user's MF row sit in shared memory, thread-major (conflict-free); the
// weights, the folded BatchNorm and a chunk of kChunk items (B rows and iMF rows, feature-major) sit in shared memory
// as well.  Every thread walks the chunk's items two at a time, in ascending id: each weight row read from shared
// memory (a broadcast float4) feeds the accumulators of both items, so the layer-2 loop -- H1 x H2 FMAs per pair, the
// bulk of the work -- is bound by FFMA issue rather than by shared-memory bandwidth.  The accumulators need
// compile-time extents: the kernel is instantiated on a width tier (H2 <= 16 / 32 / 64 / 64 with H3 <= 8 / 16 / 16 / 32), the
// activation and the list length, and loops over the real widths at run time, four columns at a time; padded weight
// columns are zero and padded features are never read, so they never enter a real sum.
//
// Selection: strict '>' against the row's k-th best while the items arrive in ascending id keeps the lower id on
// ties; topk_insert (topk_select.cuh).  Exclusions: one monotone cursor per thread into its row's ascending list,
// advanced only on the candidate path.  blockIdx.y splits the item range; the partial lists are merged by
// brk_topk_merge (score desc, id asc), identical to one unsplit scan.  A pair's score depends on A_u, B_i, the two MF
// rows and the dense block alone: the two items of a step run the same instructions, and nothing is reduced across
// pairs.
#include "common.cuh"
#include "topk_select.cuh"
#include <limits.h>
#include <math_constants.h>

namespace ntf {

constexpr int NT = 128;              // threads = users per CTA
constexpr int LDU = NT + 1;          // stride of the thread-major user rows (conflict-free staging stores)
constexpr int kChunk = 32;           // items staged per pass
constexpr int LDI = kChunk + 2;      // stride of the feature-major item rows (8-byte aligned pairs, 2-way staging)
constexpr int kMaxSplits = 32;
constexpr float kBnEps = 1e-3f;
constexpr int kMaxH1 = 128, kMaxH2 = 64, kMaxH3 = 32, kMaxEMF = 128;

template <int ACT> __device__ __forceinline__ float act_f(float x) {
  return ACT == 0 ? fmaxf(x, 0.f) : 1.0f / (1.0f + expf(-x));   // neumf_common.cuh act_f
}

struct Params {
  const float* A;                    // [U, H1] user side
  const int32_t* users;              // [U] rows of uMF
  const float* uMF;                  // [numUser, EMF]
  const float* B;                    // [I, H1] item side (b1 included)
  const float* iMF;                  // [I, EMF] MF rows of the indexed items
  const float* dense;                // the model's dense block
  const float* bn;                   // moving mean1, var1, mean2, var2
  int64_t U, I;
  int32_t H1, H2, H3, EMF, E, had, bn_on;
  int32_t k, id_offset;
  int64_t items_per_split;           // a multiple of kChunk
  float* out_vals;                   // [n_splits, U, k]
  int32_t* out_ids;
  const int64_t* excl_indptr;        // [U + 1], or null
  const int32_t* excl_ids;
};

__host__ __device__ inline int pad4(int x) { return (x + 3) & ~3; }

// Shared-memory layout in floats, every block 16-byte aligned.
struct Smem {
  int au, mu, w2, w3, st1, p2, b3, w4, bc, mc, total;
  __host__ __device__ Smem(int H1, int H2, int H3, int EMF, int HM) {
    int o = 0;
    au = o; o += pad4(H1 * LDU);                 // [H1][LDU]  A_u, thread-major
    mu = o; o += pad4(EMF * LDU);                // [EMF][LDU] uMF[u], thread-major
    w2 = o; o += H1 * pad4(H2);                  // [H1][pad4(H2)] W2, zero columns past H2
    w3 = o; o += H2 * pad4(H3);                  // [H2][pad4(H3)] W3, zero columns past H3
    st1 = o; o += pad4(2 * H1);                  // [H1] (scale, shift) of BN1
    p2 = o; o += 4 * H2;                         // [H2] (b2, scale, shift, 0) of layer 2
    b3 = o; o += pad4(H3);
    w4 = o; o += pad4(H3 + HM + 1);              // head weights, then b4
    bc = o; o += pad4(H1 * LDI);                 // [H1][LDI]  B rows of the chunk, feature-major
    mc = o; o += pad4(EMF * LDI);                // [EMF][LDI] iMF rows of the chunk
    total = o;
  }
};

template <int H2C, int H3C, int ACT, int K_CAP>
__global__ void __launch_bounds__(NT, H2C <= 16 ? 3 : 2) neumf_topk_fp32_kernel(const Params P) {
  extern __shared__ __align__(16) float sm[];
  const int H1 = P.H1, H2 = P.H2, H3 = P.H3, EMF = P.EMF, had = P.had;
  const int HM = had ? EMF : 1;
  const int H2p = pad4(H2), H3p = pad4(H3), nq2 = H2p / 4, nq3 = H3p / 4;
  const Smem L(H1, H2, H3, EMF, HM);
  float* Au = sm + L.au; float* Mu = sm + L.mu;
  float* W2 = sm + L.w2; float* W3 = sm + L.w3;
  float* st1 = sm + L.st1; float* p2 = sm + L.p2; float* b3 = sm + L.b3; float* w4 = sm + L.w4;
  float* Bc = sm + L.bc; float* Mc = sm + L.mc;
  const float* D = P.dense;
  const int oW1 = 0, ob1 = oW1 + 2 * P.E * H1, og1 = ob1 + H1, obe1 = og1 + H1, oW2 = obe1 + H1, ob2 = oW2 + H1 * H2,
            og2 = ob2 + H2, obe2 = og2 + H2, oW3 = obe2 + H2, ob3 = oW3 + H2 * H3, oW4 = ob3 + H3;

  const int t = threadIdx.x;
  const int64_t row0 = int64_t(blockIdx.x) * NT, row = row0 + t;
  const bool live = row < P.U;

  // ---- per-CTA staging: the users' rows, the weights, BatchNorm folded with the moving statistics ----
  for (int e = t; e < NT * H1; e += NT) {
    const int r = e / H1, c = e - r * H1;
    Au[c * LDU + r] = row0 + r < P.U ? __ldg(P.A + (row0 + r) * H1 + c) : 0.f;
  }
  for (int e = t; e < NT * EMF; e += NT) {
    const int r = e / EMF, f = e - r * EMF;
    Mu[f * LDU + r] = row0 + r < P.U ? __ldg(P.uMF + int64_t(__ldg(P.users + row0 + r)) * EMF + f) : 0.f;
  }
  for (int e = t; e < H1 * H2p; e += NT) {
    const int c = e / H2p, o = e - c * H2p;
    W2[e] = o < H2 ? __ldg(D + oW2 + c * H2 + o) : 0.f;
  }
  for (int e = t; e < H2 * H3p; e += NT) {
    const int c = e / H3p, o = e - c * H3p;
    W3[e] = o < H3 ? __ldg(D + oW3 + c * H3 + o) : 0.f;
  }
  for (int f = t; f < H1; f += NT) {
    float sc = 1.f, sh = 0.f;
    if (P.bn_on) {
      const float rstd = 1.0f / sqrtf(P.bn[H1 + f] + kBnEps);
      sc = D[og1 + f] * rstd; sh = D[obe1 + f] - P.bn[f] * sc;
    }
    st1[2 * f] = sc; st1[2 * f + 1] = sh;
  }
  for (int f = t; f < H2; f += NT) {
    float sc = 1.f, sh = 0.f;
    if (P.bn_on) {
      const float rstd = 1.0f / sqrtf(P.bn[2 * H1 + H2 + f] + kBnEps);
      sc = D[og2 + f] * rstd; sh = D[obe2 + f] - P.bn[2 * H1 + f] * sc;
    }
    p2[4 * f] = D[ob2 + f]; p2[4 * f + 1] = sc; p2[4 * f + 2] = sh; p2[4 * f + 3] = 0.f;
  }
  for (int f = t; f < H3; f += NT) b3[f] = D[ob3 + f];
  for (int f = t; f < H3 + HM + 1; f += NT) w4[f] = D[oW4 + f];

  float vals[K_CAP]; int32_t ids[K_CAP];
#pragma unroll
  for (int j = 0; j < K_CAP; ++j) { vals[j] = -CUDART_INF_F; ids[j] = -1; }
  float thr = -CUDART_INF_F;
  const int64_t i_begin = int64_t(blockIdx.y) * P.items_per_split;
  const int64_t i_end = min(P.I, i_begin + P.items_per_split);
  // exclusion cursor: the first listed id >= this split's first id; rows >= U and calls without a list have none
  const int32_t* cur = nullptr; int32_t left = 0, next = INT_MAX;
  if (P.excl_indptr != nullptr && live) {
    int64_t pos = P.excl_indptr[row], end = P.excl_indptr[row + 1];
    const int64_t first = i_begin + P.id_offset;
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
  const float* au = Au + t;
  const float* mu = Mu + t;

  for (int64_t i0 = i_begin; i0 < i_end; i0 += kChunk) {
    const int n_it = int(min(int64_t(kChunk), i_end - i0));
    __syncthreads();                                        // the previous chunk is consumed (and the staging done)
    for (int e = t; e < kChunk * H1; e += NT) {
      const int j = e / H1, c = e - j * H1;
      Bc[c * LDI + j] = j < n_it ? __ldg(P.B + (i0 + j) * H1 + c) : 0.f;
    }
    for (int e = t; e < kChunk * EMF; e += NT) {
      const int j = e / EMF, f = e - j * EMF;
      Mc[f * LDI + j] = j < n_it ? __ldg(P.iMF + (i0 + j) * EMF + f) : 0.f;
    }
    __syncthreads();

#pragma unroll 1
    for (int j = 0; j < n_it; j += 2) {                     // items j and j + 1 of the chunk
      // ---- layers 1 and 2: z2 = BN1(act(A_u + B_i)) W2, both items per weight row ----
      float z[2][H2C];
#pragma unroll
      for (int o = 0; o < H2C; ++o) { z[0][o] = 0.f; z[1][o] = 0.f; }
#pragma unroll 1
      for (int c = 0; c < H1; ++c) {
        const float a = au[c * LDU];
        const float2 b = *reinterpret_cast<const float2*>(Bc + c * LDI + j);
        const float2 ss = *reinterpret_cast<const float2*>(st1 + 2 * c);
        const float y[2] = {fmaf(act_f<ACT>(a + b.x), ss.x, ss.y), fmaf(act_f<ACT>(a + b.y), ss.x, ss.y)};
        const float4* w = reinterpret_cast<const float4*>(W2 + c * H2p);
#pragma unroll
        for (int q = 0; q < H2C / 4; ++q) {
          if (q < nq2) {
            const float4 wq = w[q];
#pragma unroll
            for (int s = 0; s < 2; ++s) {
              z[s][4 * q] = fmaf(y[s], wq.x, z[s][4 * q]);
              z[s][4 * q + 1] = fmaf(y[s], wq.y, z[s][4 * q + 1]);
              z[s][4 * q + 2] = fmaf(y[s], wq.z, z[s][4 * q + 2]);
              z[s][4 * q + 3] = fmaf(y[s], wq.w, z[s][4 * q + 3]);
            }
          }
        }
      }
      // ---- layer 3: z3 = BN2(act(z2 + b2)) W3 ----
      float z3[2][H3C];
#pragma unroll
      for (int o = 0; o < H3C; ++o) { z3[0][o] = 0.f; z3[1][o] = 0.f; }
#pragma unroll
      for (int c = 0; c < H2C; ++c) {
        if (c < H2) {
          const float4 pc = *reinterpret_cast<const float4*>(p2 + 4 * c);
          const float y[2] = {fmaf(act_f<ACT>(z[0][c] + pc.x), pc.y, pc.z), fmaf(act_f<ACT>(z[1][c] + pc.x), pc.y, pc.z)};
          const float4* w = reinterpret_cast<const float4*>(W3 + c * H3p);
#pragma unroll
          for (int q = 0; q < H3C / 4; ++q) {
            if (q < nq3) {
              const float4 wq = w[q];
#pragma unroll
              for (int s = 0; s < 2; ++s) {
                z3[s][4 * q] = fmaf(y[s], wq.x, z3[s][4 * q]);
                z3[s][4 * q + 1] = fmaf(y[s], wq.y, z3[s][4 * q + 1]);
                z3[s][4 * q + 2] = fmaf(y[s], wq.z, z3[s][4 * q + 2]);
                z3[s][4 * q + 3] = fmaf(y[s], wq.w, z3[s][4 * q + 3]);
              }
            }
          }
        }
      }
      // ---- head: logit = b4 + sum h3 W4[0:H3] + MF term; sigmoid ----
      const float b4 = w4[H3 + HM];
      float logit[2] = {b4, b4};
#pragma unroll
      for (int o = 0; o < H3C; ++o) {
        if (o < H3) {
          const float bo = b3[o], wo = w4[o];
#pragma unroll
          for (int s = 0; s < 2; ++s) logit[s] = fmaf(act_f<ACT>(z3[s][o] + bo), wo, logit[s]);
        }
      }
      if (had) {                                            // sum_f (uMF[f] iMF[f]) W4[H3 + f]
#pragma unroll 2
        for (int f = 0; f < EMF; ++f) {
          const float u = mu[f * LDU], wf = w4[H3 + f];
          const float2 m = *reinterpret_cast<const float2*>(Mc + f * LDI + j);
          logit[0] = fmaf(u * m.x, wf, logit[0]);
          logit[1] = fmaf(u * m.y, wf, logit[1]);
        }
      } else {                                              // W4[H3] <uMF, iMF>
        float dot[2] = {0.f, 0.f};
#pragma unroll 4
        for (int f = 0; f < EMF; ++f) {
          const float u = mu[f * LDU];
          const float2 m = *reinterpret_cast<const float2*>(Mc + f * LDI + j);
          dot[0] = fmaf(u, m.x, dot[0]);
          dot[1] = fmaf(u, m.y, dot[1]);
        }
        const float wf = w4[H3];
        logit[0] = fmaf(dot[0], wf, logit[0]);
        logit[1] = fmaf(dot[1], wf, logit[1]);
      }
      const float o0 = 1.0f / (1.0f + expf(-logit[0]));
      const float o1 = 1.0f / (1.0f + expf(-logit[1]));
      // ---- selection, item j before item j + 1 ----
#pragma unroll 1
      for (int s = 0; s < 2; ++s) {
        const float x = s ? o1 : o0;
        if (j + s < n_it && x > thr) {
          const int32_t id = int32_t(i0 + j + s) + P.id_offset;
          while (next < id) next = (--left > 0) ? *++cur : INT_MAX;
          if (next == id) continue;
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
}

// The instantiation a model takes: from its widths and k only.
struct Choice {
  const void* fn;
  void (*launch)(dim3, size_t, cudaStream_t, const Params&);
};

template <int H2C, int H3C, int ACT, int K_CAP>
void launch_one(dim3 grid, size_t smem, cudaStream_t st, const Params& P) {
  neumf_topk_fp32_kernel<H2C, H3C, ACT, K_CAP><<<grid, NT, smem, st>>>(P);
}

template <int H2C, int H3C, int ACT>
Choice pick_k(int k) {
  if (k <= 10) return {(const void*)neumf_topk_fp32_kernel<H2C, H3C, ACT, 10>, launch_one<H2C, H3C, ACT, 10>};
  if (k <= 16) return {(const void*)neumf_topk_fp32_kernel<H2C, H3C, ACT, 16>, launch_one<H2C, H3C, ACT, 16>};
  return {(const void*)neumf_topk_fp32_kernel<H2C, H3C, ACT, 32>, launch_one<H2C, H3C, ACT, 32>};
}

template <int H2C, int H3C>
Choice pick_act(int act, int k) { return act == 0 ? pick_k<H2C, H3C, 0>(k) : pick_k<H2C, H3C, 1>(k); }

Choice pick(int H2, int H3, int act, int k) {
  if (H2 <= 16 && H3 <= 8) return pick_act<16, 8>(act, k);
  if (H2 <= 32 && H3 <= 16) return pick_act<32, 16>(act, k);
  if (H3 <= 16) return pick_act<64, 16>(act, k);
  return pick_act<64, 32>(act, k);
}

struct Plan {
  Choice c;
  size_t smem;
  int splits;                        // the most splits the launch may use (the workspace holds this many lists)
};

// Item splits so that a few hundred users still fill every SM: as many as keep the grid within one wave of the
// instantiation's resident CTAs (rounding up would leave a nearly empty second wave that costs a whole CTA time),
// at most kMaxSplits.
int plan(brk_ctx* ctx, const brk_neumf_model* m, int64_t U, int32_t k, Plan* out) {
  const int emf = m->EMF > 0 ? m->EMF : m->E;
  const Smem L(m->H1, m->H2, m->H3, emf, m->mf_mode ? emf : 1);
  out->c = pick(m->H2, m->H3, m->act, k);
  out->smem = size_t(L.total) * sizeof(float);
  int per_sm = 0;
  BRK_CUDA(cudaFuncSetAttribute(out->c.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, int(out->smem)));
  BRK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, out->c.fn, NT, out->smem));
  BRK_REQUIRE(per_sm >= 1, BRK_E_ARG, "brk_neumf_score_topk_fp32: %zu bytes of shared memory do not fit an SM", out->smem);
  const int64_t slots = int64_t(per_sm) * ctx->sm_count;
  const int64_t m_tiles = (U + NT - 1) / NT;
  int64_t S = m_tiles < slots ? slots / m_tiles : 1;
  out->splits = int(S > kMaxSplits ? kMaxSplits : S);
  return 0;
}

const char* check_model(const brk_neumf_model* m) {
  static thread_local char msg[512];
  const int emf = m->EMF > 0 ? m->EMF : m->E;
  if (m->tensor_cores) return "the model computes with TF32 tensor-core products (tensor_cores = 1): rank it with brk_neumf_score_topk";
  if (m->E < 1 || m->H1 < 1 || m->H2 < 1 || m->H3 < 1 || emf < 1 || m->H1 > kMaxH1 || m->H2 > kMaxH2 || m->H3 > kMaxH3 ||
      emf > kMaxEMF || (m->act != 0 && m->act != 1)) {
    snprintf(msg, sizeof msg, "no instance for E=%d EMF=%d H=(%d,%d,%d) act=%d; built: H1 <= %d, H2 <= %d, H3 <= %d, "
             "EMF <= %d, relu or sigmoid -- wider models rank through score_all", m->E, emf, m->H1, m->H2, m->H3, m->act,
             kMaxH1, kMaxH2, kMaxH3, kMaxEMF);
    return msg;
  }
  return nullptr;
}

}  // namespace ntf

extern "C" int brk_topk_merge(brk_ctx* ctx, const float* part_vals, const int32_t* part_ids, int32_t n_parts, int64_t U,
                              int32_t k, float* out_vals, int32_t* out_ids, void* stream);

extern "C" int64_t brk_neumf_topk_fp32_workspace_bytes(brk_ctx* ctx, const brk_neumf_model* m, int64_t U, int64_t I,
                                                       int32_t k) {
  if (!ctx || !m || U <= 0 || I <= 0 || k <= 0 || k > 32 || ntf::check_model(m)) return 0;
  ntf::Plan pl;
  if (ntf::plan(ctx, m, U, k, &pl) != 0) return 0;
  return int64_t(pl.splits) * U * k * 8;
}

namespace {

int neumf_score_topk_fp32(brk_ctx* ctx, const brk_neumf_model* m, const float* user_side, const int32_t* users,
                          int64_t U, const float* item_side, const float* item_mf, int64_t I, int32_t k, int32_t id_offset,
                          const int64_t* excl_indptr, const int32_t* excl_ids, float* out_vals, int32_t* out_ids,
                          void* workspace, int64_t workspace_bytes, void* stream) {
  BRK_REQUIRE(ctx && m && user_side && users && item_side && item_mf && out_vals && out_ids, BRK_E_ARG,
              "brk_neumf_score_topk_fp32: null argument");
  BRK_REQUIRE(m->uMF.w && m->dense.w && m->bn_moving, BRK_E_ARG, "brk_neumf_score_topk_fp32: model tables missing");
  if (const char* why = ntf::check_model(m)) {
    brk_set_error("brk_neumf_score_topk_fp32: %s", why);
    return BRK_E_ARG;
  }
  BRK_REQUIRE(U >= 0 && I > 0 && U < (int64_t(1) << 31) && I < (int64_t(1) << 31), BRK_E_ARG,
              "brk_neumf_score_topk_fp32: U=%lld I=%lld", (long long)U, (long long)I);
  BRK_REQUIRE(k >= 1 && k <= 32, BRK_E_ARG, "brk_neumf_score_topk_fp32: k=%d (1..32)", k);
  BRK_REQUIRE(id_offset >= 0 && int64_t(id_offset) + I + ntf::kChunk < int64_t(INT_MAX), BRK_E_ARG,
              "brk_neumf_score_topk_fp32: id_offset=%d + I=%lld reaches INT_MAX", id_offset, (long long)I);
  if (U == 0) return 0;
  ntf::Plan pl;
  if (int rc = ntf::plan(ctx, m, U, k, &pl)) return rc;
  const int64_t need = int64_t(pl.splits) * U * k * 8;
  BRK_REQUIRE(workspace && workspace_bytes >= need, BRK_E_ARG,
              "brk_neumf_score_topk_fp32: workspace of %lld bytes needed, %lld given", (long long)need,
              (long long)workspace_bytes);
  const int emf = m->EMF > 0 ? m->EMF : m->E;
  ntf::Params P;
  P.A = user_side; P.users = users; P.uMF = m->uMF.w; P.B = item_side; P.iMF = item_mf;
  P.dense = m->dense.w; P.bn = m->bn_moving;
  P.U = U; P.I = I;
  P.H1 = m->H1; P.H2 = m->H2; P.H3 = m->H3; P.EMF = emf; P.E = m->E; P.had = m->mf_mode ? 1 : 0;
  P.bn_on = m->no_batch_norm ? 0 : 1;
  P.k = k; P.id_offset = id_offset;
  // whole chunks per split; the splits actually used can be fewer than planned
  const int64_t chunks = (I + ntf::kChunk - 1) / ntf::kChunk;
  const int64_t per = (chunks + pl.splits - 1) / pl.splits;
  P.items_per_split = per * ntf::kChunk;
  const int used = int((chunks + per - 1) / per);
  float* pv = reinterpret_cast<float*>(workspace);
  int32_t* pi = reinterpret_cast<int32_t*>(pv + int64_t(pl.splits) * U * k);
  P.out_vals = pv; P.out_ids = pi;
  P.excl_indptr = excl_indptr; P.excl_ids = excl_ids;
  cudaStream_t st = (cudaStream_t)stream;
  pl.c.launch(dim3(unsigned((U + ntf::NT - 1) / ntf::NT), unsigned(used)), pl.smem, st, P);
  BRK_LAUNCH_CHECK();
  return brk_topk_merge(ctx, pv, pi, used, U, k, out_vals, out_ids, stream);
}

}  // namespace

extern "C" int brk_neumf_score_topk_fp32(brk_ctx* ctx, const brk_neumf_model* m, const float* user_side,
                                         const int32_t* users, int64_t U, const float* item_side, const float* item_mf,
                                         int64_t I, int32_t k, int32_t id_offset, float* out_vals, int32_t* out_ids,
                                         void* workspace, int64_t workspace_bytes, void* stream) {
  return neumf_score_topk_fp32(ctx, m, user_side, users, U, item_side, item_mf, I, k, id_offset, nullptr, nullptr,
                               out_vals, out_ids, workspace, workspace_bytes, stream);
}

extern "C" int brk_neumf_score_topk_fp32_excl(brk_ctx* ctx, const brk_neumf_model* m, const float* user_side,
                                              const int32_t* users, int64_t U, const float* item_side,
                                              const float* item_mf, int64_t I, int32_t k, int32_t id_offset,
                                              const int64_t* excl_indptr, const int32_t* excl_ids, float* out_vals,
                                              int32_t* out_ids, void* workspace, int64_t workspace_bytes, void* stream) {
  BRK_REQUIRE(excl_indptr && excl_ids, BRK_E_ARG, "brk_neumf_score_topk_fp32_excl: null exclusion list");
  return neumf_score_topk_fp32(ctx, m, user_side, users, U, item_side, item_mf, I, k, id_offset, excl_indptr, excl_ids,
                               out_vals, out_ids, workspace, workspace_bytes, stream);
}
