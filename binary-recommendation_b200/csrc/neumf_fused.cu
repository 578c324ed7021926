// NeuMF training / inference step as ONE cooperative launch on the 5th-generation tensor cores.
//
// Stands in for the Keras graph of /root/reference/src/models/NeuMFModel.py:53-100 inside model.fit
// (src/models/RModel.py:130-137), and for the He et al. variant BASELINE.json configs[0] names (GMF Hadamard
// vector + MLP, no BatchNorm).  Same arithmetic as csrc/neumf_tc.cu (TF32 operands, fp32 accumulation in TMEM),
// different schedule: a CTA owns ONE tile of 128 samples for the whole step and keeps everything that the five
// kernels of neumf_tc.cu pass through HBM (h1, h2, dy1, dy2, the re-gathered rows) on chip --
//   * activations h1 / h2 and the BatchNorm-output gradients live in REGISTERS of the thread that read them
//     out of TMEM (thread = sample x column half), across the grid-wide barriers;
//   * x0 stays in shared memory (K-major for the forward product, rewritten MN-major for dW1 from the registers
//     of the gather -- the rows are read from HBM/L2 exactly once);
//   * the weight gradients dW1 / dW2 / dW3 are tensor-core products accumulated in TMEM; bias / head gradients are
//     warp-butterfly reductions into shared-memory accumulators;
//   * NO atomics on shared addresses: every CTA stores its tile's partial sums (BatchNorm statistics, the whole
//     dense-gradient block, the loss) into its own slot of a small HBM/L2 scratch, and after a grid barrier the
//     slots are summed in a fixed order -- the BatchNorm totals by every CTA, the dense gradients by the CTA that
//     owns that slice of the parameter block.  (First version: float atomics on the 2.7 k dense-gradient words
//     from 128 CTAs took 17 us of a 49 us step, the double atomics of the statistics ~2 us per barrier.)  Results
//     are bit-reproducible run to run except for the embedding-row REDs.
//   * four grid-wide barriers for training-mode BatchNorm (sum h, sum h^2 after layers 1 and 2; sum dy, sum dy*xhat
//     before them in the backward pass) and one before the dense-gradient reduction; without BatchNorm (He et al.)
//     only the last one.
//
// Thread roles (256 threads): warp w reads TMEM lane quadrant q = w & 3 (sample s = 32 q + lane) and column half
// hf = w >> 2 of every accumulator; one elected thread issues the MMAs.
#include <stdlib.h>
#include <string.h>
#include "neumf_common.cuh"
#include "tc.cuh"
#include "tc_tiles.cuh"

namespace nfz {

using ntc::issue_gemm; using ntc::km_off16; using ntc::mn_off16; using ntc::pad32; using ntc::row_of_lane;
using v2::Acc; using v2::Args; using v2::RowRef; using v2::TabRef;
using v2::act_f; using v2::act_grad; using v2::drop16_bits; using v2::locate; using v2::mark_row;
using v2::kBnEps; using v2::kBnMomentum; using v2::kDropScale;

constexpr int TS = 128;          // samples per tile = TMEM lanes
constexpr int NT = 256;          // threads per CTA
__host__ __device__ constexpr int pad4(int x) { return (x + 3) & ~3; }
__host__ __device__ constexpr int ilog2(int x) { return x <= 1 ? 0 : 1 + ilog2(x >> 1); }
__host__ __device__ constexpr int imax(int a, int b) { return a > b ? a : b; }

template <int E_, int EMF_, int H1_, int H2_, int H3_, int ACT_, int BN_, int HAD_>
struct Spec {
  static constexpr int E = E_, EMF = EMF_, H1 = H1_, H2 = H2_, H3 = H3_, ACT = ACT_, BN = BN_, HAD = HAD_;
  static constexpr int K0 = 2 * E, N3 = H3 < 16 ? 16 : H3, HM = HAD ? EMF : 1;
  static constexpr int HC1 = H1 / 2, HC2 = H2 / 2;
  static constexpr int PH = pad32(H1);                                   // column pitch of the Q / R / S tiles
  // TMEM columns: [0, K0) the product being read back (z1, z2, z3, da2, da1, dx0 in turn), then dW1, dW2, dW3
  static constexpr int CW1 = K0, CW2 = CW1 + H1, CW3 = CW2 + H2, CEND = CW3 + N3;
  static constexpr int TCOLS = CEND <= 128 ? 128 : 256;
  static constexpr int MW2 = H1 >= 64 ? H1 : 64, MW3 = H2 >= 64 ? H2 : 64;   // M of the dW2 / dW3 products
  // dense parameter block (include/brk_b200.h): W4 has H3 + HM rows
  static constexpr int oW1 = 0, ob1 = oW1 + K0 * H1, og1 = ob1 + H1, obe1 = og1 + H1;
  static constexpr int oW2 = obe1 + H1, ob2 = oW2 + H1 * H2, og2 = ob2 + H2, obe2 = og2 + H2;
  static constexpr int oW3 = obe2 + H2, ob3 = oW3 + H2 * H3, oW4 = ob3 + H3, ob4 = oW4 + H3 + HM;
  static constexpr int NW4 = H3 + HM + 1;                                // head weights + b4
  static constexpr int ND = ob4 + 1, NDP = (ND + 3) & ~3;                // dense block length
  // per-tile slot of partial sums (floats): BN forward sums of layers 1, 2; BN backward sums of layers 2, 1; the
  // tile's dense gradients; the tile's loss (a double)
  // the four BatchNorm exchanges use TAGGED 64-bit words {value | launch tag << 32} (2 H words each: sum A, sum B):
  // readers poll the data itself, there is no separate barrier for them
  static constexpr int pS1 = 0, pS2 = pS1 + 4 * H1, pD2 = pS2 + 4 * H2, pD1 = pD2 + 4 * H2, pDense = pD1 + 4 * H1;
  static constexpr int pLoss = pDense + NDP, PT = pLoss + 4;             // all multiples of 4 floats
  // shared memory (bytes); every tile is a multiple of 1024 B
  static constexpr int szP = TS * K0 * 4, szT = TS * PH * 4;
  static constexpr int szWB = imax(H1 * pad32(K0), K0 * pad32(H1)) * 4;
  static constexpr int szW2t = H2 * pad32(H1) * 4, szW3t = N3 * pad32(H2) * 4;
  static constexpr int szW2i = H1 * pad32(H2) * 4, szW3i = H2 * pad32(H3) * 4;
  static constexpr int nFloats = H1 + H2 + N3 + pad4(NW4)                // b1 b2 b3 w4
                                 + 7 * H1 + 7 * H2                       // mean rstd var gamma beta sdy sdyx per BN layer
                                 + H1 + H2 + N3 + pad4(NW4)              // gradient accumulators gb1 gb2 gb3 gw4
                                 + 2 * 8 * 32 + 2 * TS;                  // part, dl, mfs
  static constexpr int nInts = 2 * TS + TS * (K0 / 32);                  // ids, layer-0 keep masks
  static constexpr size_t smem = size_t(szP) + 3 * size_t(szT) + szWB + szW2t + szW3t + szW2i + szW3i +
                                 size_t(nFloats + nInts) * 4 + 1024;
  static_assert(K0 % 32 == 0 && H1 % 32 == 0 && H2 % 16 == 0 && H3 % 8 == 0, "widths");
  static_assert(HC1 <= 32 && HC2 <= 32 && (HC1 & (HC1 - 1)) == 0 && (HC2 & (HC2 - 1)) == 0 && (H3 & (H3 - 1)) == 0, "halves");
  static_assert(EMF % 4 == 0 && EMF <= 128 && E % 32 == 0 && (!HAD_ || EMF <= 32), "embedding widths");
  static_assert(CEND <= 256, "TMEM columns");
};

struct Extra {
  unsigned int* ticket;
  float* part;                 // [n_tiles][S::PT] per-tile partial sums (cooperative launches)
  int32_t coop;                // 1: cooperative launch (slots + grid barriers); 0: independent tiles (atomics + last-CTA ticket)
  unsigned int* bar;           // grid-barrier words {count, error, base, tag} of the context (cooperative launches; common.cuh)
  // exact Keras Adam inside the same launch (after the last barrier): do_adam != 0
  int32_t do_adam;
  brk_adam_hyper hyp;
  int64_t* adam_state;         // [0] t, [1] beta1^t, [2] beta2^t (include/brk_b200.h); advanced by block 0
  float* tm[4]; float* tv[4]; float* tw[4]; float* tg[4]; uint32_t* tt[4]; int64_t tn[4];   // tables: moments, weights, gradients, touched, elements
  int64_t trows[4];
  float* dm; float* dv; float* dw;                                                           // dense block
  unsigned long long* trace;   // BRK_NEUMF_TRACE: %globaltimer stamps of block 0 at the phase boundaries (profiles/neumf_fused_trace.py)
  int32_t n_tiles;
};
__device__ __forceinline__ void stamp(const Extra& X, int k) {
  if (X.trace != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    X.trace[k] = t;
  }
}

extern __shared__ __align__(1024) uint8_t nfz_smem_raw[];

// ---- TMEM -> registers: N consecutive columns of this thread's lane ---------------------------------------------
template <int N>
__device__ __forceinline__ void tmem_load(uint32_t taddr, float (&v)[N]) {
  static_assert(N == 8 || N == 16 || N == 32, "tmem_load width");
  uint32_t r[N];
  if constexpr (N == 32) { tc::tmem_ld_32x32_issue(taddr, r); tc::tmem_ld_wait(r); }
  else if constexpr (N == 16) tc::tmem_ld_32x32_x16(taddr, r);
  else tc::tmem_ld_32x32_x8(taddr, r);
#pragma unroll
  for (int j = 0; j < N; ++j) v[j] = __uint_as_float(r[j]);
}

// ---- per-feature sums over the 32 samples of a warp: butterfly that halves the value count at every exchange -----
// After the call r[0] of lane l holds the sum of feature  l >> (5 - log2 N)  (N - 1 + 5 - log2 N shuffles).
template <int N>
__device__ __forceinline__ void warp_feat_reduce(float (&r)[N]) {
  static_assert(N >= 1 && N <= 32 && (N & (N - 1)) == 0, "power of two");
  const int lane = threadIdx.x & 31;
  int n = N;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    if (n > 1) {
      const int half = n >> 1;
      const bool upper = (lane & off) != 0;
#pragma unroll
      for (int i = 0; i < N / 2; ++i)
        if (i < half) {
          const float mine = upper ? r[i + half] : r[i];
          const float theirs = upper ? r[i] : r[i + half];
          r[i] = mine + __shfl_xor_sync(0xffffffffu, theirs, off);
        }
      n = half;
    } else {
      r[0] += __shfl_xor_sync(0xffffffffu, r[0], off);
    }
  }
}
// Two quantities per feature summed over the tile's 128 samples -> this tile's slot (slotA[f], slotB[f], f < 2 HC).
// Thread (q, hf) holds columns [hf * HC, (hf + 1) * HC) of its sample; part: [2][8 warps][32] floats.
template <int HC>
__device__ __forceinline__ void cta_feature_sums(float (&a)[HC], float (&b)[HC], float* part, float* slotA, float* slotB) {
  constexpr int SH = 5 - ilog2(HC);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  warp_feat_reduce<HC>(a);
  warp_feat_reduce<HC>(b);
  if ((lane & ((1 << SH) - 1)) == 0) {
    part[(0 * 8 + warp) * 32 + (lane >> SH)] = a[0];
    part[(1 * 8 + warp) * 32 + (lane >> SH)] = b[0];
  }
  __syncthreads();
  if (t < 2 * HC) {
    const int hh = t / HC, j = t % HC;
    float sa = 0.f, sb = 0.f;
#pragma unroll
    for (int qq = 0; qq < 4; ++qq) { sa += part[(0 * 8 + hh * 4 + qq) * 32 + j]; sb += part[(1 * 8 + hh * 4 + qq) * 32 + j]; }
    slotA[t] = sa;
    slotB[t] = sb;
  }
  __syncthreads();
}
// The same two sums as SELF-VALIDATING words: word f (f < 2 HC) = {sum A of feature f | tag << 32}, word 2 HC + f = sum B.
// A 64-bit store is single-copy atomic, so a reader that sees the tag sees the value: no fence, no flag, no barrier.
// plainA / plainB (optional): the same sums as plain floats (the tile's BatchNorm parameter gradients in its dense slot).
template <int HC>
__device__ __forceinline__ void cta_feature_sums_tagged(float (&a)[HC], float (&b)[HC], float* part, unsigned long long* words,
                                                        uint32_t tag, float* plainA, float* plainB) {
  constexpr int SH = 5 - ilog2(HC);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  warp_feat_reduce<HC>(a);
  warp_feat_reduce<HC>(b);
  if ((lane & ((1 << SH) - 1)) == 0) {
    part[(0 * 8 + warp) * 32 + (lane >> SH)] = a[0];
    part[(1 * 8 + warp) * 32 + (lane >> SH)] = b[0];
  }
  __syncthreads();
  if (t < 2 * HC) {
    const int hh = t / HC, j = t % HC;
    float sa = 0.f, sb = 0.f;
#pragma unroll
    for (int qq = 0; qq < 4; ++qq) { sa += part[(0 * 8 + hh * 4 + qq) * 32 + j]; sb += part[(1 * 8 + hh * 4 + qq) * 32 + j]; }
    const unsigned long long hi = static_cast<unsigned long long>(tag) << 32;
    asm volatile("st.global.cg.u64 [%0], %1;" ::"l"(words + t), "l"(hi | __float_as_uint(sa)) : "memory");
    asm volatile("st.global.cg.u64 [%0], %1;" ::"l"(words + 2 * HC + t), "l"(hi | __float_as_uint(sb)) : "memory");
    if (plainA != nullptr) { plainA[t] = sa; plainB[t] = sb; }
  }
  __syncthreads();
}
// Totals over all tiles of W tagged words (W = 2 H): every thread takes one 16-byte pair of words and every
// (NT / (W / 2))-th tile, eight loads in flight, and re-reads a word until it carries this launch's tag -- the wait for
// the slowest tile and the data transfer are the same round trip.  Summed per thread in tile order, in double.
// scratch: (NT / (W / 2)) * W doubles of shared memory; tot: W doubles.  Bounded: a tile that never arrives raises err.
template <int W>
__device__ __forceinline__ void gather_tagged(const unsigned long long* base, int stride64, int n_tiles, uint32_t tag, double* scratch,
                                              double* tot, unsigned int* err) {
  constexpr int C2 = W / 2, G = NT / C2;
  static_assert(W % 2 == 0 && NT % C2 == 0, "slot width");
  const int t = threadIdx.x, f2 = t % C2, g = t / C2;
  double a0 = 0.0, a1 = 0.0;
  const long long t0 = clock64();
  for (int j0 = g; j0 < n_tiles; j0 += 8 * G) {
    ulonglong2 v[8];
#pragma unroll
    for (int q8 = 0; q8 < 8; ++q8) {
      const int j = j0 + q8 * G;
      if (j < n_tiles) v[q8] = __ldcg(reinterpret_cast<const ulonglong2*>(base + size_t(j) * stride64) + f2);
    }
#pragma unroll
    for (int q8 = 0; q8 < 8; ++q8) {
      const int j = j0 + q8 * G;
      if (j < n_tiles) {
        while (uint32_t(v[q8].x >> 32) != tag || uint32_t(v[q8].y >> 32) != tag) {
          if (clock64() - t0 > 4000000000LL) { atomicExch(err, 1u); __trap(); }
          v[q8] = __ldcg(reinterpret_cast<const ulonglong2*>(base + size_t(j) * stride64) + f2);
        }
        a0 += double(__uint_as_float(uint32_t(v[q8].x))); a1 += double(__uint_as_float(uint32_t(v[q8].y)));
      }
    }
  }
  scratch[g * W + 2 * f2] = a0; scratch[g * W + 2 * f2 + 1] = a1;
  __syncthreads();
  if (t < W) {
    double tt = 0.0;
#pragma unroll
    for (int gg = 0; gg < G; ++gg) tt += scratch[gg * W + t];
    tot[t] = tt;
  }
  __syncthreads();
}
// After the grid barrier: totals over all tiles of W consecutive slot words, summed in a fixed order in double.
// base = first tile's word 0 (16-byte aligned); tiles are PT floats apart.  Every thread takes one float4 of the slot
// and every (NT / (W / 4))-th tile, so that a tile's slot is one coalesced request and all of a thread's loads are
// in flight together.  scratch: NT * 4 doubles of shared memory (the Q tile, dead at every barrier); tot: W doubles.
template <int W>
__device__ __forceinline__ void reduce_slots(const float* base, int PT, int n_tiles, double* scratch, double* tot) {
  constexpr int C4 = W / 4, G = NT / C4;
  static_assert(W % 4 == 0 && NT % C4 == 0, "slot width");
  const int t = threadIdx.x, f4 = t % C4, g = t / C4;
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll 8
  for (int j = g; j < n_tiles; j += G) {
    const float4 v = __ldcg(reinterpret_cast<const float4*>(base + size_t(j) * PT) + f4);
    a0 += double(v.x); a1 += double(v.y); a2 += double(v.z); a3 += double(v.w);
  }
  scratch[g * W + 4 * f4 + 0] = a0; scratch[g * W + 4 * f4 + 1] = a1;
  scratch[g * W + 4 * f4 + 2] = a2; scratch[g * W + 4 * f4 + 3] = a3;
  __syncthreads();
  if (t < W) {
    double tt = 0.0;
#pragma unroll
    for (int gg = 0; gg < G; ++gg) tt += scratch[gg * W + t];
    tot[t] = tt;
  }
  __syncthreads();
}
// One quantity per feature, added to a shared-memory accumulator of this CTA (bias gradients).
template <int HC>
__device__ __forceinline__ void cta_feature_sum_local(float (&a)[HC], float* part, float* dst) {
  constexpr int SH = 5 - ilog2(HC);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  warp_feat_reduce<HC>(a);
  if ((lane & ((1 << SH) - 1)) == 0) part[warp * 32 + (lane >> SH)] = a[0];
  __syncthreads();
  if (t < 2 * HC) {
    const int hh = t / HC, j = t % HC;
    float sa = 0.f;
#pragma unroll
    for (int qq = 0; qq < 4; ++qq) sa += part[(hh * 4 + qq) * 32 + j];
    dst[t] += sa;
  }
  __syncthreads();
}

// keep bits of features [c0, c0 + HC) of `layer` for sample idx (bit j = feature c0 + j); c0 a multiple of HC
template <int HC>
__device__ __forceinline__ uint32_t drop_bits_range(uint64_t idx, int c0, int layer, uint32_t seed, uint32_t epoch) {
  uint32_t bits = 0;
#pragma unroll
  for (int c = 0; c < (HC + 15) / 16; ++c) {
    const uint32_t b = drop16_bits(idx, c0 / 16 + c, layer, seed, epoch);
    bits |= (HC >= 16) ? (b << (16 * c)) : ((b >> (c0 & 15)) & ((1u << HC) - 1u));
  }
  return bits;
}

// swizzled K-major image of a small matrix: value(r, c) for r < ROWS, c < COLS_PAD (a multiple of 32)
template <int ROWS, int COLS_PAD, class F>
__device__ __forceinline__ void build_image(uint8_t* dst, F value) {
  for (int idx = threadIdx.x; idx < ROWS * COLS_PAD; idx += NT) {
    const int r = idx / COLS_PAD, c = idx % COLS_PAD;
    *reinterpret_cast<float*>(dst + km_off16(ROWS, r, c >> 2) + (c & 3) * 4) = value(r, c);
  }
}

// ---- after the tiles: the dense gradients -- the slots of all tiles, summed in tile order by the CTA that owns the
//      parameter slice (float4 granularity) -- and, with do_adam, the exact Keras Adam of optim.cu over the dense block and
//      the four tables in the same pass.  Run by EVERY CTA of a cooperative launch: the tile CTAs and the helper CTAs that
//      only exist so that a small batch does not leave this phase (20 MB of optimizer traffic) to a handful of SMs.
template <class S>
__device__ __forceinline__ void dense_reduce_and_adam(const Args& A, const Extra& X, unsigned int bar_target, uint32_t tag,
                                                      float4* f4red, float alpha) {
  const int t = threadIdx.x;
  brk_grid_barrier(X.bar, bar_target);
  if (blockIdx.x == 0 && t == 0) { X.bar[2] = bar_target; X.bar[3] = tag; }   // the next launch's barrier base and last tag
  const float b1c = X.hyp.beta1, b2c = X.hyp.beta2, ob1c = 1.0f - X.hyp.beta1, ob2c = 1.0f - X.hyp.beta2, epsc = X.hyp.eps;
  auto adam1 = [&](float& w, float& m, float& v, float g) {
    m = b1c * m + ob1c * g;
    v = b2c * v + ob2c * g * g;
    w -= alpha * m / (sqrtf(v) + epsc);
  };
  auto adam4 = [&](float4* w, float4* m, float4* v, float4 g4) {
    float4 w4 = *w, m4 = *m, v4 = *v;
    adam1(w4.x, m4.x, v4.x, g4.x); adam1(w4.y, m4.y, v4.y, g4.y); adam1(w4.z, m4.z, v4.z, g4.z); adam1(w4.w, m4.w, v4.w, g4.w);
    *w = w4; *m = m4; *v = v4;
  };
  constexpr int n4 = S::NDP / 4;
  const int per4 = (n4 + int(gridDim.x) - 1) / int(gridDim.x);
  const int lo4 = int(blockIdx.x) * per4, hi4 = lo4 + per4 < n4 ? lo4 + per4 : n4;
  int PP = 1;
  while (PP < per4 && PP < NT) PP <<= 1;
  const int groups = NT / PP, grp = t / PP, pl = t % PP;
  float4* G4 = reinterpret_cast<float4*>(A.dense.g);
  for (int p0 = lo4; p0 < hi4; p0 += PP) {
    const int pp = p0 + pl;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (pp < hi4)
#pragma unroll 8
      for (int j = grp; j < X.n_tiles; j += groups) {
        const float4 v = __ldcg(reinterpret_cast<const float4*>(X.part + size_t(j) * S::PT + S::pDense) + pp);
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      }
    f4red[t] = acc;
    __syncthreads();
    if (grp == 0 && pp < hi4) {
      // with Adam in this launch the block's accumulator is not read: it is zero between steps (include/brk_b200.h)
      float4 g4 = X.do_adam ? make_float4(0.f, 0.f, 0.f, 0.f) : G4[pp];
      for (int gg = 0; gg < groups; ++gg) {
        const float4 v = f4red[gg * PP + pl];
        g4.x += v.x; g4.y += v.y; g4.z += v.z; g4.w += v.w;
      }
      if (X.do_adam) {
        adam4(reinterpret_cast<float4*>(X.dw) + pp, reinterpret_cast<float4*>(X.dm) + pp, reinterpret_cast<float4*>(X.dv) + pp, g4);
      } else {
        G4[pp] = g4;
      }
    }
    __syncthreads();
  }
  stamp(X, 10);
  if (X.do_adam) {                                      // the four tables: every element moves (Keras' sparse Adam is dense-equivalent)
    const int64_t gtid = int64_t(blockIdx.x) * NT + t, nthr = int64_t(gridDim.x) * NT;
#pragma unroll 1
    for (int k = 0; k < 4; ++k) {
      const int64_t e4 = X.tn[k] >> 2;
      float4* w = reinterpret_cast<float4*>(X.tw[k]); float4* m = reinterpret_cast<float4*>(X.tm[k]);
      float4* v = reinterpret_cast<float4*>(X.tv[k]); float4* g = reinterpret_cast<float4*>(X.tg[k]);
      // four elements per thread and pass: all sixteen loads are issued before the first store (the compiler
      // cannot hoist them itself past stores through pointers it must assume to alias)
      for (int64_t i0 = gtid; i0 < e4; i0 += 4 * nthr) {
        float4 gq[4], wq[4], mq[4], vq[4];
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          const int64_t i = i0 + q4 * nthr;
          if (i < e4) { gq[q4] = g[i]; wq[q4] = w[i]; mq[q4] = m[i]; vq[q4] = v[i]; }
        }
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          const int64_t i = i0 + q4 * nthr;
          if (i < e4) {
            adam1(wq[q4].x, mq[q4].x, vq[q4].x, gq[q4].x); adam1(wq[q4].y, mq[q4].y, vq[q4].y, gq[q4].y);
            adam1(wq[q4].z, mq[q4].z, vq[q4].z, gq[q4].z); adam1(wq[q4].w, mq[q4].w, vq[q4].w, gq[q4].w);
            w[i] = wq[q4]; m[i] = mq[q4]; v[i] = vq[q4]; g[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
      }
      if (X.tt[k] != nullptr) {
        const int64_t nwords = (X.trows[k] + 31) >> 5;
        for (int64_t i = gtid; i < nwords; i += nthr) X.tt[k][i] = 0u;
      }
    }
    if (blockIdx.x == 0 && t == 0) {                    // every CTA read the state during set-up, before the barriers
      double* pw = reinterpret_cast<double*>(X.adam_state);
      X.adam_state[0] += 1;
      pw[1] *= double(X.hyp.beta1);
      pw[2] *= double(X.hyp.beta2);
    }
  }
}

#define NFZ_OPERANDS_READY() do { tc::fence_proxy_async_smem(); tc::fence_before_sync(); __syncthreads(); tc::fence_after_sync(); } while (0)

template <class S>
__global__ void __launch_bounds__(NT, (S::smem <= 110 * 1024) ? 2 : 1) fused_step(const Args A, const Extra X) {
  using AC = Acc<S::H1, S::H2>;
  constexpr int E = S::E, EMF = S::EMF, H1 = S::H1, H2 = S::H2, H3 = S::H3, ACT = S::ACT, N3 = S::N3, HM = S::HM;
  constexpr int K0 = S::K0, HC1 = S::HC1, HC2 = S::HC2;
  constexpr bool BN = S::BN != 0, HAD = S::HAD != 0;
  
  uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(nfz_smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* P = sm;                                   // x0: K-major (forward), then MN-major (dW1)
  uint8_t* Q = P + S::szP;                           // K-major operand of the running product (a1, a2, dz3, dz2, dz1)
  uint8_t* R = Q + S::szT;                           // MN-major activation (a2 for dW3, a1 for dW2)
  uint8_t* Sb = R + S::szT;                          // MN-major dz (B operand of the weight-gradient products)
  uint8_t* WB = Sb + S::szT;                         // W1^T image (forward), then W1 image (dx0)
  uint8_t* W2t = WB + S::szWB;
  uint8_t* W3t = W2t + S::szW2t;
  uint8_t* W2i = W3t + S::szW3t;
  uint8_t* W3i = W2i + S::szW2i;
  float* fl = reinterpret_cast<float*>(W3i + S::szW3i);
  float* b1 = fl;            float* b2 = b1 + H1;      float* b3 = b2 + H2;       float* w4 = b3 + N3;
  float* mean1 = w4 + pad4(S::NW4); float* rstd1 = mean1 + H1; float* gam1 = rstd1 + H1; float* bet1 = gam1 + H1;
  float* sdy1 = bet1 + H1;   float* sdyx1 = sdy1 + H1; float* var1 = sdyx1 + H1;
  float* mean2 = var1 + H1;  float* rstd2 = mean2 + H2; float* gam2 = rstd2 + H2; float* bet2 = gam2 + H2;
  float* sdy2 = bet2 + H2;   float* sdyx2 = sdy2 + H2; float* var2 = sdyx2 + H2;
  float* gb1 = var2 + H2;   float* gb2 = gb1 + H1;    float* gb3 = gb2 + H2;     float* gw4 = gb3 + N3;
  float* part = gw4 + pad4(S::NW4);
  float* dl = part + 2 * 8 * 32; float* mfs = dl + TS;
  // scratch of the cross-tile reductions, aliased onto arrays that are dead whenever a reduction runs: `part` is
  // only live inside cta_feature_sums (before the barrier), dl / mfs only between the head and the MF gradient REDs
  double* dred = reinterpret_cast<double*>(Q);             // NT * 4 doubles = 8 KB: the Q tile is dead at every barrier
  double* tot = reinterpret_cast<double*>(dl);             // <= 128 doubles = 1 KB
  static_assert(((3 * (H1 + H2) + 2 * N3 + 2 * pad4(S::NW4) + 6 * (H1 + H2)) % 2) == 0 && 2 * H1 <= 128 && S::szT >= NT * 32,
                "alignment / size of the aliases");
  int32_t* ids_s = reinterpret_cast<int32_t*>(mfs + TS);
  uint32_t* masks = reinterpret_cast<uint32_t*>(ids_s + 2 * TS);
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_slot;
  __shared__ double red[32];
  __shared__ bool last;
  __shared__ float alpha_s;
  __shared__ uint32_t base_s, tag_s;

  const int t = threadIdx.x, warp = t >> 5, lane = t & 31, q = warp & 3, hf = warp >> 2, s = q * 32 + lane;
  const int64_t b0 = int64_t(blockIdx.x) * TS;
  const int valid = int((A.B - b0) < int64_t(TS) ? (A.B - b0) : int64_t(TS));
  const bool ok = s < valid;
  const bool training = A.training != 0, dropout = A.dropout != 0;
  const uint64_t sidx = uint64_t(A.first_index + b0 + s);
  const bool coop = X.coop != 0;
  float* slot = X.part + size_t(blockIdx.x) * S::PT;  // this tile's partial sums (cooperative launches)
  float* dp = slot + S::pDense;
  // cooperative launches: the barrier base and the last launch's slot-word tag, loaded here and published to shared memory
  // (registers are the kernel's limit) just before the first __syncthreads, so that the round trip overlaps the set-up
  // loads; dense_reduce_and_adam writes both back after the barrier
  unsigned int base = 0u, last_tag = 0u;
  if (coop && t == 0) {
    base = *reinterpret_cast<volatile unsigned int*>(X.bar + 2);
    last_tag = *reinterpret_cast<volatile unsigned int*>(X.bar + 3);
  }
  auto publish_launch_words = [&]() {
    if (coop && t == 0) { base_s = base; tag_s = last_tag + 1u != 0u ? last_tag + 1u : 1u; }   // zeroed slots carry tag 0
  };
  const uint32_t bar_a = tc::smem_u32(&bar);
  uint32_t phase = 0;
  const int c1 = hf * HC1, c2 = hf * HC2;            // first column of this thread's half in layers 1 / 2
  stamp(X, 0);
  if (X.trace != nullptr && t == 0 && blockIdx.x < 480) {   // which SM runs this CTA (trace words 32 ..)
    unsigned int smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    X.trace[32 + blockIdx.x] = smid;
  }

  if (int(blockIdx.x) >= X.n_tiles) {
    // helper CTA of a cooperative training launch (grid = max(tiles, SMs)): no tile, only the barriers and its share of
    // the dense-gradient reduction and of the Adam pass
    if (t == 64 && X.do_adam) {
      const double* pw = reinterpret_cast<const double*>(X.adam_state);
      const double p1 = pw[1] * double(X.hyp.beta1), p2 = pw[2] * double(X.hyp.beta2);
      alpha_s = float(double(X.hyp.lr) * sqrt(1.0 - p2) / (1.0 - p1));
    }
    publish_launch_words();
    __syncthreads();
    dense_reduce_and_adam<S>(A, X, base_s, tag_s, reinterpret_cast<float4*>(Q), alpha_s);
    return;
  }

  // ---- set-up: ids and the dense parameter block (one coalesced copy into the R / S tile space, free until phase C;
  //      the operand images and small vectors are then built from shared memory) -----------------------------------
  static_assert(S::NDP * 4 <= 2 * S::szT, "dense block fits the R + S tiles");
  float* Wd = reinterpret_cast<float*>(R);
  if (t < 2 * TS) {
    const int r = t & (TS - 1);
    ids_s[t] = r < valid ? __ldg((t < TS ? A.u : A.i) + b0 + r) : 0;
  }
  for (int i4 = t; i4 < S::ND / 4; i4 += NT)
    reinterpret_cast<float4*>(Wd)[i4] = __ldg(reinterpret_cast<const float4*>(A.dense.w) + i4);
  if (t < S::ND % 4) Wd[(S::ND / 4) * 4 + t] = __ldg(A.dense.w + (S::ND / 4) * 4 + t);
  if (t == 0) { tc::mbar_init(bar_a, 1); tc::fence_barrier_init(); }
  if (t < 32) tc::tmem_alloc<S::TCOLS>(tc::smem_u32(&tmem_slot));
  if (t == 64 && X.do_adam) {                               // Keras Adam step size of this step (the state is advanced at the end)
    const double* pw = reinterpret_cast<const double*>(X.adam_state);
    const double p1 = pw[1] * double(X.hyp.beta1), p2 = pw[2] * double(X.hyp.beta2);
    alpha_s = float(double(X.hyp.lr) * sqrt(1.0 - p2) / (1.0 - p1));
  }
  publish_launch_words();
  __syncthreads();                                          // ids, Wd, launch words
  // x0 rows: every load of the thread is issued here and lands while the images are being built
  constexpr int LPR = E / 4, RPP = NT / LPR, NP = TS / RPP;
  const int gc4 = t % LPR, grr = t / LPR;
  float4 xv[2 * NP];
#pragma unroll
  for (int tab = 0; tab < 2; ++tab)
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      const int r = p * RPP + grr;
      xv[tab * NP + p] = r < valid ? __ldg(reinterpret_cast<const float4*>(locate<E>(tab == 0 ? A.uMLP : A.iMLP, ids_s[tab * TS + r]).w) + gc4)
                                   : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  for (int f = t; f < H1; f += NT) { b1[f] = Wd[S::ob1 + f]; gam1[f] = Wd[S::og1 + f]; bet1[f] = Wd[S::obe1 + f]; gb1[f] = 0.f; }
  for (int f = t; f < H2; f += NT) { b2[f] = Wd[S::ob2 + f]; gam2[f] = Wd[S::og2 + f]; bet2[f] = Wd[S::obe2 + f]; gb2[f] = 0.f; }
  for (int f = t; f < N3; f += NT) { b3[f] = f < H3 ? Wd[S::ob3 + f] : 0.f; gb3[f] = 0.f; }
  for (int f = t; f < S::NW4; f += NT) { w4[f] = Wd[S::oW4 + f]; gw4[f] = 0.f; }
  // the two transposed images are written in SOURCE order (conflict-free reads of the staged block; in image order
  // the reads stride by the layer width and serialise 16- to 32-fold); K0 and H1 are multiples of 32: no pad columns
  for (int idx = t; idx < K0 * H1; idx += NT) {
    const int c = idx / H1, r = idx % H1;
    *reinterpret_cast<float*>(WB + km_off16(H1, r, c >> 2) + (c & 3) * 4) = Wd[S::oW1 + idx];
  }
  for (int idx = t; idx < H1 * H2; idx += NT) {
    const int c = idx / H2, r = idx % H2;
    *reinterpret_cast<float*>(W2t + km_off16(H2, r, c >> 2) + (c & 3) * 4) = Wd[S::oW2 + idx];
  }
  build_image<N3, pad32(H2)>(W3t, [&](int r, int c) { return (c < H2 && r < H3) ? Wd[S::oW3 + c * H3 + r] : 0.f; });
  build_image<H1, pad32(H2)>(W2i, [&](int r, int c) { return c < H2 ? Wd[S::oW2 + r * H2 + c] : 0.f; });
  build_image<H2, pad32(H3)>(W3i, [&](int r, int c) { return c < H3 ? Wd[S::oW3 + r * H3 + c] : 0.f; });
  if (dropout) {                                           // layer-0 keep bits: K0 / 16 Philox calls per sample, half per thread
    for (int c = hf * (K0 / 32); c < (hf + 1) * (K0 / 32); ++c) {
      const uint32_t bits = ok ? drop16_bits(sidx, c, 0, A.drop_seed, A.drop_epoch) : 0u;
      reinterpret_cast<uint16_t*>(masks + s * (K0 / 32))[c] = uint16_t(bits);
    }
  }
  // keep bits of this thread's columns in layers 1 and 2: drawn here, off the critical path between the barriers
  const uint32_t m1 = (dropout && ok) ? drop_bits_range<HC1>(sidx, c1, 1, A.drop_seed, A.drop_epoch) : 0xFFFFFFFFu;
  const uint32_t m2 = (dropout && ok) ? drop_bits_range<HC2>(sidx, c2, 2, A.drop_seed, A.drop_epoch) : 0xFFFFFFFFu;
  if (!training || !BN) {                                  // BatchNorm with the moving statistics (inference)
    for (int f = t; f < H1; f += NT) { mean1[f] = BN ? A.bn_moving[f] : 0.f; rstd1[f] = BN ? 1.0f / sqrtf(A.bn_moving[H1 + f] + kBnEps) : 1.f; }
    for (int f = t; f < H2; f += NT) { mean2[f] = BN ? A.bn_moving[2 * H1 + f] : 0.f; rstd2[f] = BN ? 1.0f / sqrtf(A.bn_moving[2 * H1 + H2 + f] + kBnEps) : 1.f; }
  }
  tc::fence_before_sync();
  __syncthreads();                                          // masks, TMEM address
  tc::fence_after_sync();
  const uint32_t tmem = tmem_slot;
  const uint32_t tlane = tmem + (uint32_t(q * 32) << 16);  // this warp's lane quadrant
  stamp(X, 1);

  // ---- phase A: x0 = dropout([uMLP[u], iMLP[i]]);  h1 = act(x0 W1 + b1) ---------------------------------------
#pragma unroll
  for (int tab = 0; tab < 2; ++tab)
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      const int r = p * RPP + grr;
      float4 x = xv[tab * NP + p];
      if (dropout) {
        const int f = tab * E + 4 * gc4;
        const uint32_t m = masks[r * (K0 / 32) + (f >> 5)] >> (f & 31);
        x.x = (m & 1u) ? x.x * kDropScale : 0.f; x.y = (m & 2u) ? x.y * kDropScale : 0.f;
        x.z = (m & 4u) ? x.z * kDropScale : 0.f; x.w = (m & 8u) ? x.w * kDropScale : 0.f;
      }
      xv[tab * NP + p] = x;
      *reinterpret_cast<float4*>(P + km_off16(TS, r, tab * LPR + gc4)) = x;
    }
  stamp(X, 2);
  NFZ_OPERANDS_READY();
  if (t == 0) {
    issue_gemm<128, H1, 0, 0>(tmem, tc::smem_u32(P), TS, tc::smem_u32(WB), H1, K0, false);
    tc::mma_commit(bar_a);
  }
  tc::mbar_wait(bar_a, phase); phase ^= 1u;
  tc::fence_after_sync();
  stamp(X, 3);
  float h1[HC1];
  {
    float v[HC1];
    tmem_load<HC1>(tlane + uint32_t(c1), v);
#pragma unroll
    for (int j = 0; j < HC1; ++j) h1[j] = ok ? act_f<ACT>(v[j] + b1[c1 + j]) : 0.f;
  }
  if (training) {
    // the product has read P and WB: x0 goes back MN-major (A operand of dW1), WB becomes the W1 image of dx0
#pragma unroll
    for (int tab = 0; tab < 2; ++tab)
#pragma unroll
      for (int p = 0; p < NP; ++p)
        *reinterpret_cast<float4*>(P + mn_off16(TS, p * RPP + grr, tab * LPR + gc4)) = xv[tab * NP + p];
    build_image<K0, pad32(H1)>(WB, [&](int r, int c) { return c < H1 ? Wd[S::oW1 + r * H1 + c] : 0.f; });
  }
  if (training && BN) {
    float a[HC1], b[HC1];
#pragma unroll
    for (int j = 0; j < HC1; ++j) { a[j] = h1[j]; b[j] = h1[j] * h1[j]; }
    cta_feature_sums_tagged<HC1>(a, b, part, reinterpret_cast<unsigned long long*>(slot + S::pS1), tag_s, nullptr, nullptr);
    gather_tagged<2 * H1>(reinterpret_cast<const unsigned long long*>(X.part + S::pS1), S::PT / 2, X.n_tiles, tag_s, dred, tot, X.bar + 1);
    for (int f = t; f < H1; f += NT) {
      const double m = tot[f] / double(A.B);
      const double var = fmax(tot[H1 + f] / double(A.B) - m * m, 0.0);
      mean1[f] = float(m); var1[f] = float(var); rstd1[f] = 1.0f / sqrtf(float(var) + kBnEps);
    }
    __syncthreads();
  }

  stamp(X, 4);
  // ---- phase B: a1 = dropout(bn1(h1));  h2 = act(a1 W2 + b2) ---------------------------------------------------
  auto a1_value = [&](int j) {                              // column c1 + j of a1 for this thread's sample
    const int f = c1 + j;
    float y = BN ? gam1[f] * ((h1[j] - mean1[f]) * rstd1[f]) + bet1[f] : h1[j];
    if (dropout) y = ((m1 >> j) & 1u) ? y * kDropScale : 0.f;
    return ok ? y : 0.f;
  };
#pragma unroll
  for (int f4 = 0; f4 < HC1 / 4; ++f4)
    *reinterpret_cast<float4*>(Q + km_off16(TS, s, c1 / 4 + f4)) =
        make_float4(a1_value(4 * f4), a1_value(4 * f4 + 1), a1_value(4 * f4 + 2), a1_value(4 * f4 + 3));
  NFZ_OPERANDS_READY();
  if (t == 0) {
    issue_gemm<128, H2, 0, 0>(tmem, tc::smem_u32(Q), TS, tc::smem_u32(W2t), H2, H1, false);
    tc::mma_commit(bar_a);
  }
  tc::mbar_wait(bar_a, phase); phase ^= 1u;
  tc::fence_after_sync();
  float h2[HC2];
  {
    float v[HC2];
    tmem_load<HC2>(tlane + uint32_t(c2), v);
#pragma unroll
    for (int j = 0; j < HC2; ++j) h2[j] = ok ? act_f<ACT>(v[j] + b2[c2 + j]) : 0.f;
  }
  // MF rows: the loads are issued here, in front of the barrier, and land while this CTA waits (MLPR lanes per row
  // pair; the chunks stay in registers for the head and for the gradient REDs)
  constexpr int MLPR = EMF / 4, MRPP = NT / MLPR, MNP = (TS + MRPP - 1) / MRPP;
  const int mc4 = t % MLPR, mrr = t / MLPR;
  float4 mu[MNP], mi[MNP];
#pragma unroll
  for (int p = 0; p < MNP; ++p) {
    const int r = p * MRPP + mrr;
    mu[p] = mi[p] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < valid) {
      mu[p] = __ldg(reinterpret_cast<const float4*>(locate<EMF>(A.uMF, ids_s[r]).w) + mc4);
      mi[p] = __ldg(reinterpret_cast<const float4*>(locate<EMF>(A.iMF, ids_s[TS + r]).w) + mc4);
    }
  }
  if (training && BN) {
    float a[HC2], b[HC2];
#pragma unroll
    for (int j = 0; j < HC2; ++j) { a[j] = h2[j]; b[j] = h2[j] * h2[j]; }
    stamp(X, 12);
    cta_feature_sums_tagged<HC2>(a, b, part, reinterpret_cast<unsigned long long*>(slot + S::pS2), tag_s, nullptr, nullptr);
    stamp(X, 13);
    stamp(X, 14);
    gather_tagged<2 * H2>(reinterpret_cast<const unsigned long long*>(X.part + S::pS2), S::PT / 2, X.n_tiles, tag_s, dred, tot, X.bar + 1);
    stamp(X, 15);
    for (int f = t; f < H2; f += NT) {
      const double m = tot[f] / double(A.B);
      const double var = fmax(tot[H2 + f] / double(A.B) - m * m, 0.0);
      mean2[f] = float(m); var2[f] = float(var); rstd2[f] = 1.0f / sqrtf(float(var) + kBnEps);
    }
    __syncthreads();
  }

  stamp(X, 5);
  // ---- phase C: a2 = dropout(bn2(h2));  h3 = act(a2 W3 + b3);  MF part;  logit, prediction, loss ------------------
#pragma unroll
  for (int f4 = 0; f4 < HC2 / 4; ++f4) {
    float v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int j = 4 * f4 + k, f = c2 + j;
      float y = BN ? gam2[f] * ((h2[j] - mean2[f]) * rstd2[f]) + bet2[f] : h2[j];
      if (dropout) y = ((m2 >> j) & 1u) ? y * kDropScale : 0.f;
      v[k] = ok ? y : 0.f;
    }
    const float4 v4 = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(Q + km_off16(TS, s, c2 / 4 + f4)) = v4;
    if (training) *reinterpret_cast<float4*>(R + mn_off16(TS, s, c2 / 4 + f4)) = v4;
  }
  NFZ_OPERANDS_READY();
  if (t == 0) {
    issue_gemm<128, N3, 0, 0>(tmem, tc::smem_u32(Q), TS, tc::smem_u32(W3t), N3, H2, false);
    tc::mma_commit(bar_a);
  }
  float4 wmf = make_float4(1.f, 1.f, 1.f, 1.f);            // head weights of this thread's four MF features
  if (HAD) wmf = make_float4(w4[H3 + 4 * mc4], w4[H3 + 4 * mc4 + 1], w4[H3 + 4 * mc4 + 2], w4[H3 + 4 * mc4 + 3]);
#pragma unroll
  for (int p = 0; p < MNP; ++p) {
    float pr;
    if (HAD) pr = fmaf(mu[p].x * mi[p].x, wmf.x, fmaf(mu[p].y * mi[p].y, wmf.y, fmaf(mu[p].z * mi[p].z, wmf.z, mu[p].w * mi[p].w * wmf.w)));
    else     pr = fmaf(mu[p].x, mi[p].x, fmaf(mu[p].y, mi[p].y, fmaf(mu[p].z, mi[p].z, mu[p].w * mi[p].w)));
    pr = group_sum<MLPR>(pr);
    const int r = p * MRPP + mrr;
    if (mc4 == 0 && r < TS) mfs[r] = pr;
  }
  tc::mbar_wait(bar_a, phase); phase ^= 1u;
  tc::fence_after_sync();
  __syncthreads();                                          // mfs visible
  float loss_local = 0.f;
  if (hf == 0) {                                            // one thread per sample
    float v[N3];
    tmem_load<N3>(tlane, v);
    float h3[H3], dlogit = 0.f;
    if (ok) {
      float logit = w4[H3 + HM];
#pragma unroll
      for (int j = 0; j < H3; ++j) { h3[j] = act_f<ACT>(v[j] + b3[j]); logit = fmaf(h3[j], w4[j], logit); }
      logit = HAD ? logit + mfs[s] : fmaf(mfs[s], w4[H3], logit);
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
    if (training) {
      dl[s] = dlogit;
      float dz3[H3], pw[H3];
#pragma unroll
      for (int j = 0; j < H3; ++j) { dz3[j] = dlogit * w4[j] * act_grad<ACT>(h3[j]); pw[j] = h3[j] * dlogit; }
      // dz3 rows in both operand forms, columns [H3, 32) zero
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) {
        float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        if (4 * c4 < H3) z = make_float4(dz3[(4 * c4) % H3], dz3[(4 * c4 + 1) % H3], dz3[(4 * c4 + 2) % H3], dz3[(4 * c4 + 3) % H3]);
        *reinterpret_cast<float4*>(Q + km_off16(TS, s, c4)) = z;
        *reinterpret_cast<float4*>(Sb + mn_off16(TS, s, c4)) = z;
      }
      // head / layer-3 bias gradients of this warp's 32 samples -> the CTA's shared-memory accumulators
      constexpr int SH3 = 5 - ilog2(H3);
      warp_feat_reduce<H3>(pw);
      warp_feat_reduce<H3>(dz3);
      // per-warp partials into `part` (combined in warp order after the barrier below: no atomics, reproducible bits)
      if ((lane & ((1 << SH3) - 1)) == 0) { part[(0 * 8 + warp) * 32 + (lane >> SH3)] = pw[0]; part[(1 * 8 + warp) * 32 + (lane >> SH3)] = dz3[0]; }
      const float sdl = warp_sum(dlogit);
      const float smf = HAD ? 0.f : warp_sum(ok ? mfs[s] * dlogit : 0.f);
      if (lane == 0) { part[(0 * 8 + warp) * 32 + 30] = sdl; part[(0 * 8 + warp) * 32 + 31] = smf; }
    }
  }
  {
    const double lsum = block_sum_double(double(loss_local), red);
    if (t == 0) {
      if (coop) *reinterpret_cast<double*>(slot + S::pLoss) = lsum;
      else atomicAdd(A.acc + AC::loss, lsum);
    }
  }

  stamp(X, 6);
  if (training) {
    __syncthreads();                                        // dl and the warps' head partials visible
    if (t < H3) {
      float sw = 0.f, sb = 0.f;
#pragma unroll
      for (int w = 0; w < 4; ++w) { sw += part[(0 * 8 + w) * 32 + t]; sb += part[(1 * 8 + w) * 32 + t]; }
      gw4[t] += sw; gb3[t] += sb;
    }
    if (t == 32) {
      float sl = 0.f, sm_ = 0.f;
#pragma unroll
      for (int w = 0; w < 4; ++w) { sl += part[(0 * 8 + w) * 32 + 30]; sm_ += part[(0 * 8 + w) * 32 + 31]; }
      gw4[H3 + HM] += sl;
      if (!HAD) gw4[H3] += sm_;
    }
    // MF embedding gradients: 16-byte REDs into the owners' accumulators; Hadamard head weights
    float4 hw = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int p = 0; p < MNP; ++p) {
      const int r = p * MRPP + mrr;
      if (r < valid) {
        const RowRef ru = locate<EMF>(A.uMF, ids_s[r]), ri = locate<EMF>(A.iMF, ids_s[TS + r]);
        const float d = dl[r];
        const float4 cf = HAD ? make_float4(d * wmf.x, d * wmf.y, d * wmf.z, d * wmf.w)
                              : make_float4(d * w4[H3], d * w4[H3], d * w4[H3], d * w4[H3]);
        red_add_f4(ru.g + 4 * mc4, make_float4(cf.x * mi[p].x, cf.y * mi[p].y, cf.z * mi[p].z, cf.w * mi[p].w));
        red_add_f4(ri.g + 4 * mc4, make_float4(cf.x * mu[p].x, cf.y * mu[p].y, cf.z * mu[p].z, cf.w * mu[p].w));
        if (mc4 == 0) { mark_row(ru); mark_row(ri); }
        if (HAD) { hw.x = fmaf(d, mu[p].x * mi[p].x, hw.x); hw.y = fmaf(d, mu[p].y * mi[p].y, hw.y);
                   hw.z = fmaf(d, mu[p].z * mi[p].z, hw.z); hw.w = fmaf(d, mu[p].w * mi[p].w, hw.w); }
      }
    }
    if (HAD) {                                              // lanes with equal mc4 hold the same four features
#pragma unroll
      for (int o = MLPR; o < 32; o <<= 1) {
        hw.x += __shfl_xor_sync(0xffffffffu, hw.x, o); hw.y += __shfl_xor_sync(0xffffffffu, hw.y, o);
        hw.z += __shfl_xor_sync(0xffffffffu, hw.z, o); hw.w += __shfl_xor_sync(0xffffffffu, hw.w, o);
      }
      __syncthreads();                                      // the head partials above have been consumed
      if (lane < MLPR) {
        float* pr = part + (1 * 8 + warp) * 32 + 4 * mc4;
        pr[0] = hw.x; pr[1] = hw.y; pr[2] = hw.z; pr[3] = hw.w;
      }
      __syncthreads();
      if (t < EMF) {
        float sw = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) sw += part[(1 * 8 + w) * 32 + t];
        gw4[H3 + t] += sw;
      }
    }
    // da2 = dz3 W3^T;  dW3 = a2^T dz3 (M = 64: rows >= H2 alias / are ignored)
    NFZ_OPERANDS_READY();
    if (t == 0) {
      issue_gemm<128, H2, 0, 0>(tmem, tc::smem_u32(Q), TS, tc::smem_u32(W3i), H2, (H3 + 7) & ~7, false);
      constexpr uint32_t idesc = tc::idesc_tf32_f32(S::MW3, N3, 1, 1);
      for (int ks = 0; ks < TS / 8; ++ks) {
        const uint64_t ad = tc::smem_desc_sw128_base32(tc::smem_u32(R) + uint32_t(ks) * 1024u, H2 >= 64 ? TS * 128u : 0u, 512);
        const uint64_t bd = tc::smem_desc_sw128_base32(tc::smem_u32(Sb) + uint32_t(ks) * 1024u, TS * 128u, 512);
        tc::mma_tf32_ss(tmem + S::CW3, ad, bd, idesc, ks != 0 ? 1u : 0u);
      }
      tc::mma_commit(bar_a);
    }
    tc::mbar_wait(bar_a, phase); phase ^= 1u;
    tc::fence_after_sync();
    float dy2[HC2];
    {
      float v[HC2];
      tmem_load<HC2>(tlane + uint32_t(c2), v);
#pragma unroll
      for (int j = 0; j < HC2; ++j) {
        float d = v[j];
        if (dropout) d = ((m2 >> j) & 1u) ? d * kDropScale : 0.f;
        dy2[j] = ok ? d : 0.f;
      }
    }
    if (BN) {
      float a[HC2], b[HC2];
#pragma unroll
      for (int j = 0; j < HC2; ++j) { a[j] = dy2[j]; b[j] = dy2[j] * ((h2[j] - mean2[c2 + j]) * rstd2[c2 + j]); }
      // the tile's sums are also its share of the BatchNorm parameter gradients: d beta = sum dy, d gamma = sum dy xhat
      cta_feature_sums_tagged<HC2>(a, b, part, reinterpret_cast<unsigned long long*>(slot + S::pD2), tag_s, dp + S::obe2, dp + S::og2);
      gather_tagged<2 * H2>(reinterpret_cast<const unsigned long long*>(X.part + S::pD2), S::PT / 2, X.n_tiles, tag_s, dred, tot, X.bar + 1);
      for (int f = t; f < H2; f += NT) { sdy2[f] = float(tot[f] / double(A.B)); sdyx2[f] = float(tot[H2 + f] / double(A.B)); }
      __syncthreads();
    }

    stamp(X, 7);
    // ---- phase D: dz2 = bn2-backward(dy2) * act'(h2);  dW2 += a1^T dz2;  da1 = dz2 W2^T -------------------------
    {
      float dz[HC2];
#pragma unroll
      for (int j = 0; j < HC2; ++j) {
        const int f = c2 + j;
        float dh = dy2[j];
        if (BN) { const float xh = (h2[j] - mean2[f]) * rstd2[f]; dh = gam2[f] * rstd2[f] * (dy2[j] - sdy2[f] - xh * sdyx2[f]); }
        dz[j] = ok ? dh * act_grad<ACT>(h2[j]) : 0.f;
      }
#pragma unroll
      for (int f4 = 0; f4 < HC2 / 4; ++f4) {
        const float4 v4 = make_float4(dz[4 * f4], dz[4 * f4 + 1], dz[4 * f4 + 2], dz[4 * f4 + 3]);
        *reinterpret_cast<float4*>(Q + km_off16(TS, s, c2 / 4 + f4)) = v4;
        *reinterpret_cast<float4*>(Sb + mn_off16(TS, s, c2 / 4 + f4)) = v4;
      }
#pragma unroll
      for (int f4 = 0; f4 < HC1 / 4; ++f4)                  // a1 again, MN-major (A operand of dW2)
        *reinterpret_cast<float4*>(R + mn_off16(TS, s, c1 / 4 + f4)) =
            make_float4(a1_value(4 * f4), a1_value(4 * f4 + 1), a1_value(4 * f4 + 2), a1_value(4 * f4 + 3));
      cta_feature_sum_local<HC2>(dz, part, gb2);
    }
    NFZ_OPERANDS_READY();
    if (t == 0) {
      issue_gemm<128, H1, 0, 0>(tmem, tc::smem_u32(Q), TS, tc::smem_u32(W2i), H1, H2, false);
      constexpr uint32_t idesc = tc::idesc_tf32_f32(S::MW2, H2, 1, 1);
      for (int ks = 0; ks < TS / 8; ++ks) {
        const uint64_t ad = tc::smem_desc_sw128_base32(tc::smem_u32(R) + uint32_t(ks) * 1024u, H1 >= 64 ? TS * 128u : 0u, 512);
        const uint64_t bd = tc::smem_desc_sw128_base32(tc::smem_u32(Sb) + uint32_t(ks) * 1024u, TS * 128u, 512);
        tc::mma_tf32_ss(tmem + S::CW2, ad, bd, idesc, ks != 0 ? 1u : 0u);
      }
      tc::mma_commit(bar_a);
    }
    tc::mbar_wait(bar_a, phase); phase ^= 1u;
    tc::fence_after_sync();
    float dy1[HC1];
    {
      float v[HC1];
      tmem_load<HC1>(tlane + uint32_t(c1), v);
#pragma unroll
      for (int j = 0; j < HC1; ++j) {
        float d = v[j];
        if (dropout) d = ((m1 >> j) & 1u) ? d * kDropScale : 0.f;
        dy1[j] = ok ? d : 0.f;
      }
    }
    if (BN) {
      float a[HC1], b[HC1];
#pragma unroll
      for (int j = 0; j < HC1; ++j) { a[j] = dy1[j]; b[j] = dy1[j] * ((h1[j] - mean1[c1 + j]) * rstd1[c1 + j]); }
      cta_feature_sums_tagged<HC1>(a, b, part, reinterpret_cast<unsigned long long*>(slot + S::pD1), tag_s, dp + S::obe1, dp + S::og1);
      gather_tagged<2 * H1>(reinterpret_cast<const unsigned long long*>(X.part + S::pD1), S::PT / 2, X.n_tiles, tag_s, dred, tot, X.bar + 1);
      for (int f = t; f < H1; f += NT) { sdy1[f] = float(tot[f] / double(A.B)); sdyx1[f] = float(tot[H1 + f] / double(A.B)); }
      __syncthreads();
    }

    stamp(X, 8);
    // ---- phase E: dz1 = bn1-backward(dy1) * act'(h1);  dW1 += x0^T dz1;  dx0 = dz1 W1^T -> row-gradient REDs ------
    {
      float dz[HC1];
#pragma unroll
      for (int j = 0; j < HC1; ++j) {
        const int f = c1 + j;
        float dh = dy1[j];
        if (BN) { const float xh = (h1[j] - mean1[f]) * rstd1[f]; dh = gam1[f] * rstd1[f] * (dy1[j] - sdy1[f] - xh * sdyx1[f]); }
        dz[j] = ok ? dh * act_grad<ACT>(h1[j]) : 0.f;
      }
#pragma unroll
      for (int f4 = 0; f4 < HC1 / 4; ++f4) {
        const float4 v4 = make_float4(dz[4 * f4], dz[4 * f4 + 1], dz[4 * f4 + 2], dz[4 * f4 + 3]);
        *reinterpret_cast<float4*>(Q + km_off16(TS, s, c1 / 4 + f4)) = v4;
        *reinterpret_cast<float4*>(Sb + mn_off16(TS, s, c1 / 4 + f4)) = v4;
      }
      cta_feature_sum_local<HC1>(dz, part, gb1);
    }
    NFZ_OPERANDS_READY();
    if (t == 0) {
      issue_gemm<128, K0, 0, 0>(tmem, tc::smem_u32(Q), TS, tc::smem_u32(WB), K0, H1, false);
      constexpr uint32_t idesc = tc::idesc_tf32_f32(K0, H1, 1, 1);
      for (int ks = 0; ks < TS / 8; ++ks) {
        const uint64_t ad = tc::smem_desc_sw128_base32(tc::smem_u32(P) + uint32_t(ks) * 1024u, TS * 128u, 512);
        const uint64_t bd = tc::smem_desc_sw128_base32(tc::smem_u32(Sb) + uint32_t(ks) * 1024u, TS * 128u, 512);
        tc::mma_tf32_ss(tmem + S::CW1, ad, bd, idesc, ks != 0 ? 1u : 0u);
      }
      tc::mma_commit(bar_a);
    }
    tc::mbar_wait(bar_a, phase); phase ^= 1u;
    tc::fence_after_sync();
    {                                                       // dx0: warps 0..3 carry the user half, warps 4..7 the item half
      const int tab = hf;
      RowRef rr; rr.w = nullptr; rr.g = nullptr; rr.t = nullptr; rr.lrow = 0;
      if (ok) rr = locate<E>(tab == 0 ? A.uMLP : A.iMLP, ids_s[tab * TS + s]);
#pragma unroll
      for (int cc = 0; cc < E; cc += 32) {
        float v[32];
        tmem_load<32>(tlane + uint32_t(tab * E + cc), v);
        if (ok) {
          const int f0 = tab * E + cc;
          const uint32_t m = dropout ? masks[s * (K0 / 32) + (f0 >> 5)] : 0xFFFFFFFFu;
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            float4 g4;
            g4.x = ((m >> (j + 0)) & 1u) ? v[j + 0] : 0.f; g4.y = ((m >> (j + 1)) & 1u) ? v[j + 1] : 0.f;
            g4.z = ((m >> (j + 2)) & 1u) ? v[j + 2] : 0.f; g4.w = ((m >> (j + 3)) & 1u) ? v[j + 3] : 0.f;
            if (dropout) { g4.x *= kDropScale; g4.y *= kDropScale; g4.z *= kDropScale; g4.w *= kDropScale; }
            red_add_f4(rr.g + cc + j, g4);
          }
        }
      }
      if (ok) mark_row(rr);
    }
    stamp(X, 9);
    // ---- flush the dense gradients of this tile -----------------------------------------------------------------
    float* __restrict__ G = A.dense.g;
    // coop: plain stores into this tile's slot (summed over tiles after the barrier below); otherwise float atomics
    auto put = [&](int off, float v) { if (coop) dp[off] = v; else atomicAdd(G + off, v); };
    {                                                       // dW1: lane = row k of [K0][H1], this warp's column half
      const int k = row_of_lane<K0>(q * 32 + lane);
      float v[HC1];
      tmem_load<HC1>(tlane + uint32_t(S::CW1 + c1), v);
      if (k >= 0 && k < K0) {
        if (coop) {
#pragma unroll
          for (int j = 0; j < HC1; j += 4) *reinterpret_cast<float4*>(dp + S::oW1 + k * H1 + c1 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        } else {
#pragma unroll
          for (int j = 0; j < HC1; ++j) put(S::oW1 + k * H1 + c1 + j, v[j]);
        }
      }
    }
    {                                                       // dW2: rows of [H1][H2]
      const int k = row_of_lane<S::MW2>(q * 32 + lane);
      float v[HC2];
      tmem_load<HC2>(tlane + uint32_t(S::CW2 + c2), v);
      if (k >= 0 && k < H1) {
        if (coop) {
#pragma unroll
          for (int j = 0; j < HC2; j += 4) *reinterpret_cast<float4*>(dp + S::oW2 + k * H2 + c2 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        } else {
#pragma unroll
          for (int j = 0; j < HC2; ++j) put(S::oW2 + k * H2 + c2 + j, v[j]);
        }
      }
    }
    if (hf == 0) {                                          // dW3: rows of [H2][H3]
      const int k = row_of_lane<S::MW3>(q * 32 + lane);
      float v[N3];
      tmem_load<N3>(tlane + uint32_t(S::CW3), v);
      if (k >= 0 && k < H2)
#pragma unroll
        for (int j = 0; j < H3; ++j) put(S::oW3 + k * H3 + j, v[j]);
    }
    __syncthreads();                                        // shared-memory accumulators complete
    for (int f = t; f < H1; f += NT) put(S::ob1 + f, gb1[f]);
    for (int f = t; f < H2; f += NT) put(S::ob2 + f, gb2[f]);
    for (int f = t; f < H3; f += NT) put(S::ob3 + f, gb3[f]);
    for (int f = t; f < S::NW4; f += NT) put(S::oW4 + f, gw4[f]);
    if (coop && !BN) {                                      // unused BatchNorm slots of the block
      for (int f = t; f < 2 * H1; f += NT) dp[S::og1 + f] = 0.f;
      for (int f = t; f < 2 * H2; f += NT) dp[S::og2 + f] = 0.f;
    }
    if (coop) {
      for (int f = S::ND + t; f < S::NDP; f += NT) dp[f] = 0.f;           // pad words of the block
      dense_reduce_and_adam<S>(A, X, base_s, tag_s, reinterpret_cast<float4*>(Q), alpha_s);   // every tile buffer is dead by now
      if (blockIdx.x == 0) {                                // BN moving statistics, loss
        if (BN) {
          for (int f = t; f < H1; f += NT) {
            A.bn_moving[f] = A.bn_moving[f] * kBnMomentum + mean1[f] * (1.f - kBnMomentum);
            A.bn_moving[H1 + f] = A.bn_moving[H1 + f] * kBnMomentum + var1[f] * (1.f - kBnMomentum);
          }
          for (int f = t; f < H2; f += NT) {
            A.bn_moving[2 * H1 + f] = A.bn_moving[2 * H1 + f] * kBnMomentum + mean2[f] * (1.f - kBnMomentum);
            A.bn_moving[2 * H1 + H2 + f] = A.bn_moving[2 * H1 + H2 + f] * kBnMomentum + var2[f] * (1.f - kBnMomentum);
          }
        }
        if (warp == 0 && A.loss_out) {
          double l = 0.0;
          for (int j = lane; j < X.n_tiles; j += 32) l += __ldcg(reinterpret_cast<const double*>(X.part + size_t(j) * S::PT + S::pLoss));
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
          if (lane == 0) A.loss_out[0] = float(l / double(A.B));
        }
      }
    }
  }

  // ---- independent tiles (inference; training without BatchNorm on a grid too large to be co-resident): the last
  //      CTA to finish writes the loss and re-zeroes the accumulator
  if (!(coop && training)) {
    __syncthreads();
    if (t == 0) { __threadfence(); last = atomicAdd(X.ticket, 1u) == gridDim.x - 1; }
    __syncthreads();
    if (last) {
      __threadfence();
      if (t == 0 && A.loss_out) A.loss_out[0] = float(__ldcg(A.acc + AC::loss) / double(A.B));
      __syncthreads();
      if (t == 0) { A.acc[AC::loss] = 0.0; *X.ticket = 0u; }
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (t < 32) tc::tmem_dealloc<S::TCOLS>(tmem);
  stamp(X, 11);
}

struct AdamReq {                 // optional: exact Keras Adam in the same launch (single process, mirrored tables)
  const brk_neumf_model* m;
  brk_adam_hyper h;
  int64_t* state;
};

template <class S>
int run(brk_ctx* ctx, const Args& A, const AdamReq* adam, cudaStream_t st, int* handled) {
  auto fn = fused_step<S>;
  // the shared-memory opt-in is per device: set it for the current one; occupancy is a property of the kernel, queried once
  BRK_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, int(S::smem > 120 * 1024 ? S::smem : 120 * 1024)));
  static int per_sm = -1;
  if (per_sm < 0) {
    int occ = 0;
    BRK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, NT, S::smem));
    const int by_tmem = 512 / S::TCOLS;                     // TMEM columns per SM
    per_sm = occ < by_tmem ? occ : by_tmem;
  }
  const int max_blocks = per_sm * ctx->sm_count;
  const int64_t n_tiles = (A.B + TS - 1) / TS;
  Extra X;
  memset(&X, 0, sizeof(X));
  X.ticket = ctx->tickets + 6; X.n_tiles = int(n_tiles);
  const char* tr = getenv("BRK_NEUMF_TRACE");               // hex address of a device buffer of >= 16 uint64
  X.trace = tr ? reinterpret_cast<unsigned long long*>(strtoull(tr, nullptr, 16)) : nullptr;
  Args Ac = A;
  const bool fits = n_tiles <= max_blocks;
  const bool aligned = brk_aligned16(A.dense.w) && brk_aligned16(A.dense.g) && A.dense.d >= S::NDP;
  if (!aligned) { *handled = 0; return 0; }
  if (A.training != 0 && S::BN != 0 && !fits) { *handled = 0; return 0; }   // BatchNorm needs every tile on chip at once
  if (adam != nullptr && (A.training == 0 || !fits)) { *handled = 0; return 0; }
  *handled = 1;
  if (A.training == 0 || !fits) {                           // independent tiles: any grid, ordinary launch
    fn<<<unsigned(n_tiles), NT, S::smem, st>>>(Ac, X);
    BRK_LAUNCH_CHECK();
    return 0;
  }
  const size_t need = size_t(max_blocks) * S::PT;
  if (ctx->neumf_part_floats < need) {
    if (ctx->neumf_part) BRK_CUDA(cudaFree(ctx->neumf_part));
    ctx->neumf_part = nullptr; ctx->neumf_part_floats = 0;
    BRK_CUDA(cudaMalloc(&ctx->neumf_part, need * sizeof(float)));
    BRK_CUDA(cudaMemsetAsync(ctx->neumf_part, 0, need * sizeof(float), st));   // no stale word may carry a future tag
    ctx->neumf_part_floats = need;
  }
  X.part = ctx->neumf_part; X.coop = 1;
  // helper CTAs up to one per SM: the final reduction / Adam phase is spread over the whole GPU even for a small batch
  const unsigned grid = unsigned(n_tiles > ctx->sm_count ? n_tiles : (ctx->sm_count < max_blocks ? ctx->sm_count : max_blocks));
  X.bar = ctx->bar[BRK_BAR_NEUMF];
  if (adam != nullptr) {
    const brk_table* tb[4] = {&adam->m->uMLP, &adam->m->iMLP, &adam->m->uMF, &adam->m->iMF};
    for (int k = 0; k < 4; ++k) {
      const int64_t n = tb[k]->rows * tb[k]->d;
      BRK_REQUIRE(tb[k]->m && tb[k]->v && tb[k]->g && (n & 3) == 0 && brk_aligned16(tb[k]->w) && brk_aligned16(tb[k]->g) &&
                      brk_aligned16(tb[k]->m) && brk_aligned16(tb[k]->v),
                  BRK_E_ARG, "brk_neumf_train_step: table %d needs Adam moments and 16-byte aligned storage", k);
      X.tw[k] = tb[k]->w; X.tg[k] = tb[k]->g; X.tm[k] = tb[k]->m; X.tv[k] = tb[k]->v; X.tt[k] = tb[k]->touched;
      X.tn[k] = n; X.trows[k] = tb[k]->rows;
    }
    BRK_REQUIRE(adam->m->dense.m && adam->m->dense.v && brk_aligned16(adam->m->dense.m) && brk_aligned16(adam->m->dense.v),
                BRK_E_ARG, "brk_neumf_train_step: dense block needs Adam moments");
    X.dw = adam->m->dense.w; X.dm = adam->m->dense.m; X.dv = adam->m->dense.v;
    X.do_adam = 1; X.hyp = adam->h; X.adam_state = adam->state;
  }
  void* args[] = {(void*)&Ac, (void*)&X};
  // A grid of at most one CTA per SM must also RUN one per SM: with room for two CTAs the block scheduler may pack pairs
  // onto one SM and leave others idle, and every barrier then waits for the slow pairs.  Asking for more than half of the
  // SM's shared memory forces the spread.
  size_t smem = S::smem;
  if (int(grid) <= ctx->sm_count && smem < size_t(120) * 1024) smem = size_t(120) * 1024;
  BRK_CUDA(cudaLaunchCooperativeKernel((const void*)fn, dim3(grid), dim3(NT), args, smem, st));
  return 0;
}

}  // namespace nfz

void brk_neumf_fill_args(v2::Args& A, const brk_neumf_model* m, const brk_neumf_shards* sh, const int32_t* u,
                         const int32_t* i, const float* y, int64_t batch, int64_t global_batch, int64_t first_index,
                         int32_t training, uint32_t dropout_seed, uint32_t dropout_epoch, const brk_neumf_workspace* ws,
                         float* out, float* loss_out);

// One-launch tensor-core step.  Returns 0 with *handled = 1 when it ran (rc in *rc_out), *handled = 0 when the
// model is not one of the built instances or the batch does not fit on chip (callers fall back to the five-kernel
// path of neumf_tc.cu).  Built: class spec numFactor 32 and 64 (relu), He et al. (E 32, EMF 8, Hadamard, no BN).
int brk_neumf_step_fused(brk_ctx* ctx, const brk_neumf_model* m, const brk_neumf_shards* sh, const int32_t* u,
                         const int32_t* i, const float* y, int64_t batch, int64_t global_batch, int64_t first_index,
                         int32_t training, uint32_t dropout_seed, uint32_t dropout_epoch, const brk_neumf_workspace* ws,
                         float* out, float* loss_out, cudaStream_t st, int* rc_out, int* handled,
                         const brk_adam_hyper* adam_h, int64_t* adam_state) {
  *handled = 0; *rc_out = 0;
  nfz::AdamReq areq; areq.m = m; areq.state = adam_state;
  if (adam_h) areq.h = *adam_h;
  const nfz::AdamReq* adam = (adam_h != nullptr && adam_state != nullptr && sh == nullptr) ? &areq : nullptr;
  if (getenv("BRK_NEUMF_NO_FUSED") != nullptr) return 0;
  v2::Args A;
  brk_neumf_fill_args(A, m, sh, u, i, y, batch, global_batch, first_index, training, dropout_seed, dropout_epoch, ws, out, loss_out);
  const int emf = m->EMF > 0 ? m->EMF : m->E;
#define BRK_FUSED_SPEC(E_, EMF_, A_, B_, C_, ACT_, BN_, HAD_)                                                         \
  if (m->E == E_ && emf == EMF_ && m->H1 == A_ && m->H2 == B_ && m->H3 == C_ && m->act == ACT_ &&                     \
      (m->no_batch_norm ? 0 : 1) == BN_ && m->mf_mode == HAD_) {                                                      \
    *rc_out = nfz::run<nfz::Spec<E_, EMF_, A_, B_, C_, ACT_, BN_, HAD_>>(ctx, A, adam, st, handled);                  \
    return 0;                                                                                                         \
  }
  BRK_FUSED_SPEC(32, 32, 32, 16, 8, 0, 1, 0)       // reference class spec, numFactor 32 (RModel.py:35)
  BRK_FUSED_SPEC(64, 64, 64, 32, 16, 0, 1, 0)      // BASELINE.json configs[3] widths
  BRK_FUSED_SPEC(32, 8, 32, 16, 8, 0, 0, 1)        // He et al.: MLP 64-32-16-8, GMF 8 (BASELINE.json configs[0])
#undef BRK_FUSED_SPEC
  return 0;
}
