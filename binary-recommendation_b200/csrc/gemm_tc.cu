// General dense product on the 5th-generation tensor cores: C (+)= alpha * opA(A) opB(B) (+ bias), TF32 operands
// (fp32 bits in shared memory, 10 mantissa bits used), fp32 accumulation in TMEM.  Used by the two-tower step
// (trainers/twoTower.py:77-102: tower Dense layers, the in-batch score matrix Q C^T, and the three gradient
// products) where the CUDA-core SGEMM of twotower.cu is the exact-fp32 alternative.
//
// A CTA owns a 128 x BN output tile.  K is walked in chunks of 32 (one 128-byte swizzle block): 256 threads copy
// the A and B chunks from global memory into shared memory with 16-byte loads, written directly in the swizzle of
// the view the tensor core needs --
//   operand stored with K contiguous  ([M][K] / [N][K])  -> K-major,  SWIZZLE_128B
//   operand stored with M/N contiguous ([K][M] / [K][N]) -> MN-major, SWIZZLE_128B_BASE32B
// -- so transposed operands cost nothing.  Two chunk buffers: while the tensor core consumes chunk c (4
// tcgen05.mma of K = 8, committed to an mbarrier), the threads stage chunk c+1.  Epilogue: tcgen05.ld, one output
// row per thread, bias / alpha, plain stores or REDs (split-K).
#include "common.cuh"
#include "tc.cuh"
#include <stdlib.h>

namespace gtc {

constexpr int NT = 256, BM = 128, KC = 32;

__device__ __forceinline__ uint32_t km_off16(int rows, int row, int c4) {
  const int c = c4 & 7, r8 = row & 7;
  return uint32_t(row >> 3) * 1024u + uint32_t(r8) * 128u + uint32_t((c ^ r8) << 4) + uint32_t(c4 >> 3) * uint32_t(rows) * 128u;
}
__device__ __forceinline__ uint32_t mn_off16(int rows, int row, int c4) {
  const int c32 = (c4 & 7) >> 1, half = c4 & 1, r4 = row & 3;
  return uint32_t(c4 >> 3) * uint32_t(rows) * 128u + uint32_t(row >> 2) * 512u + uint32_t(r4) * 128u + uint32_t((c32 ^ r4) << 5) +
         uint32_t(half << 4);
}

struct Params {
  const float* A; const float* B; float* C; const float* bias;
  int M, N, K, lda, ldb, ldc;
  float alpha;
  int accumulate;          // 0: C = ..., 1: C += ... (REDs when split-K)
  int k_per_split;         // multiple of KC
  unsigned long long* trace;   // optional [8] globaltimer stamps of CTA 0 (brk_gemm_tf32_trace), else null
};
__device__ __forceinline__ void stamp(const Params& P, int k) {
  if (P.trace && blockIdx.x == 0 && blockIdx.z == 0 && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    P.trace[k] = t;
  }
}

// 16-byte asynchronous global -> shared copy; bytes beyond src_bytes are zero-filled (src_bytes in [0, 16])
__device__ __forceinline__ void cp_async16(uint8_t* dst, const void* src, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(tc::smem_u32(dst)), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// MN = 0: operand stored [R][K] (R = M or N rows of this tile, K contiguous);  MN = 1: stored [K][R].
// Issues the copies of chunk [k0, k0 + KC) of rows [r0, r0 + ROWS) into `dst` (zero-filled outside the matrix).
template <int MN, int ROWS>
__device__ __forceinline__ void stage_chunk(uint8_t* dst, const float* __restrict__ src, int ld, int r0, int r_end, int k0,
                                            int k_end) {
  if (MN == 0) {                         // tile rows = R index, 8 chunks of 16 B along K
#pragma unroll
    for (int idx = threadIdx.x; idx < ROWS * (KC / 4); idx += NT) {
      const int r = idx / (KC / 4), c4 = idx % (KC / 4);
      const int gr = r0 + r, gk = k0 + c4 * 4;
      int nb = (gr < r_end) ? (k_end - gk) * 4 : 0;
      nb = nb < 0 ? 0 : (nb > 16 ? 16 : nb);
      cp_async16(dst + km_off16(ROWS, r, c4), nb ? (const void*)(src + int64_t(gr) * ld + gk) : (const void*)src, nb);
    }
  } else {                               // tile rows = K index (KC of them), ROWS/4 chunks of 16 B along R
#pragma unroll
    for (int idx = threadIdx.x; idx < KC * (ROWS / 4); idx += NT) {
      const int k = idx / (ROWS / 4), c4 = idx % (ROWS / 4);
      const int gk = k0 + k, gr = r0 + c4 * 4;
      int nb = (gk < k_end) ? (r_end - gr) * 4 : 0;
      nb = nb < 0 ? 0 : (nb > 16 ? 16 : nb);
      cp_async16(dst + mn_off16(KC, k, c4), nb ? (const void*)(src + int64_t(gk) * ld + gr) : (const void*)src, nb);
    }
  }
}

constexpr int STAGES = 4;

template <int BN, int A_MN, int B_MN>
__global__ void __launch_bounds__(NT) gemm_tf32_kernel(const Params P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr uint32_t A_BYTES = BM * KC * 4, B_BYTES = BN * KC * 4, STAGE_BYTES = A_BYTES + B_BYTES;
  __shared__ uint64_t bar[STAGES];
  __shared__ uint32_t tmem_slot;
  constexpr int TCOLS = BN < 32 ? 32 : BN;
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const unsigned col_tiles = unsigned(P.N + BN - 1) / BN;      // grid x = row tile * col_tiles + column tile
  const int m0 = int(blockIdx.x / col_tiles) * BM, n0 = int(blockIdx.x % col_tiles) * BN;
  const int kbeg = blockIdx.z * P.k_per_split;
  const int kend = min(P.K, kbeg + P.k_per_split);
  const int m_end = P.M, n_end = P.N;
  stamp(P, 0);
  if (t == 0) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) tc::mbar_init(tc::smem_u32(&bar[s]), 1);
    tc::fence_barrier_init();
  }
  if (t < 32) tc::tmem_alloc<TCOLS>(tc::smem_u32(&tmem_slot));
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = tmem_slot;
  stamp(P, 1);                             // TMEM allocated
  constexpr uint32_t idesc = tc::idesc_tf32_f32(BM, BN, A_MN, B_MN);
  const int n_chunks = (kend - kbeg + KC - 1) / KC;
  auto issue = [&](int c) {               // copies of chunk c into stage c % STAGES (an empty group past the end)
    if (c < n_chunks) {
      uint8_t* base = sm + uint32_t(c % STAGES) * STAGE_BYTES;
      stage_chunk<A_MN, BM>(base, P.A, P.lda, m0, m_end, kbeg + c * KC, kend);
      stage_chunk<B_MN, BN>(base + A_BYTES, P.B, P.ldb, n0, n_end, kbeg + c * KC, kend);
    }
    cp_async_commit();
  };
#pragma unroll
  for (int c = 0; c < STAGES - 1; ++c) issue(c);
  uint32_t phase_bits = 0u;               // bit s = parity to wait for on bar[s]
  for (int c = 0; c < n_chunks; ++c) {
    const int sidx = c % STAGES;
    cp_async_wait<STAGES - 2>();          // this thread's copies of chunk c have landed
    tc::fence_proxy_async_smem();
    __syncthreads();                      // ... and everybody's
    tc::fence_after_sync();
    if (c == 0) stamp(P, 2);              // first chunk staged
    if (t == 0) {
      const uint32_t a = tc::smem_u32(sm + uint32_t(sidx) * STAGE_BYTES), bb = a + A_BYTES;
#pragma unroll
      for (int ks = 0; ks < KC / 8; ++ks) {
        const uint64_t ad = A_MN ? tc::smem_desc_sw128_base32(a + uint32_t(ks) * 1024u, KC * 128u, 512)
                                 : tc::smem_desc_sw128_ex(a + uint32_t(ks) * 32u, 16, 1024);
        const uint64_t bd = B_MN ? tc::smem_desc_sw128_base32(bb + uint32_t(ks) * 1024u, KC * 128u, 512)
                                 : tc::smem_desc_sw128_ex(bb + uint32_t(ks) * 32u, 16, 1024);
        tc::mma_tf32_ss(tmem, ad, bd, idesc, (c | ks) != 0 ? 1u : 0u);
      }
      tc::mma_commit(tc::smem_u32(&bar[sidx]));
    }
    // refill the stage chunk c-1 used (chunk c+STAGES-1 maps onto it) once the tensor core has read it
    if (c >= 1 && c + STAGES - 1 < n_chunks) {
      const int ps = (c - 1) % STAGES;
      tc::mbar_wait(tc::smem_u32(&bar[ps]), (phase_bits >> ps) & 1u);
      phase_bits ^= 1u << ps;
    }
    issue(c + STAGES - 1);
  }
  cp_async_wait<0>();
  // drain: every commit whose completion has not been consumed yet (the last min(n_chunks, STAGES) chunks at most)
  for (int c = 0; c < n_chunks; ++c) {
    const bool consumed = (c + STAGES < n_chunks);          // waited for in the loop above (as chunk (c+1) - 1 with refill)
    if (!consumed) { const int ps = c % STAGES; tc::mbar_wait(tc::smem_u32(&bar[ps]), (phase_bits >> ps) & 1u); phase_bits ^= 1u << ps; }
  }
  tc::fence_after_sync();
  __syncthreads();                         // all MMAs done: the stage buffers become the epilogue's staging tile
  stamp(P, 3);                             // products complete
  if (n_chunks > 0) {
    // epilogue: warp w reads lane quadrant (w & 3), column half (w >> 2); rows go through shared memory so that the
    // global stores are whole 16-byte chunks of consecutive columns (row-per-thread scalar stores cost 12 us per tile)
    // (BN = 32: one 32-column read per lane quadrant, warps 4..7 have nothing to read)
    constexpr int HC = BN >= 64 ? BN / 2 : BN, CP = BN + 4;
    float* Cs = reinterpret_cast<float*>(sm);
    const int rl = (warp & 3) * 32 + lane, c0 = BN >= 64 ? (warp >> 2) * HC : 0;
    for (int cc = 0; cc < HC && (BN >= 64 || warp < 4); cc += 32) {
      uint32_t r[32];
      tc::tmem_ld_32x32_issue(tmem + (uint32_t((warp & 3) * 32) << 16) + uint32_t(c0 + cc), r);
      tc::tmem_ld_wait(r);
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        if (cc + j < HC)
          *reinterpret_cast<float4*>(Cs + rl * CP + c0 + cc + j) =
              make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
    }
    __syncthreads();
    stamp(P, 4);                           // accumulators in shared memory
    const bool split = gridDim.z > 1;
    const bool vec = (P.ldc & 3) == 0 && brk_aligned16(P.C);
    for (int idx = t; idx < BM * (BN / 4); idx += NT) {
      const int r = idx / (BN / 4), c4 = idx % (BN / 4);
      const int row = m0 + r, col = n0 + c4 * 4;
      if (row >= P.M || col >= P.N) continue;
      float4 v = *reinterpret_cast<const float4*>(Cs + r * CP + c4 * 4);
      float vv[4] = {P.alpha * v.x, P.alpha * v.y, P.alpha * v.z, P.alpha * v.w};
      float* dst = P.C + int64_t(row) * P.ldc + col;
      const int nv = min(4, P.N - col);
      if (P.bias != nullptr && blockIdx.z == 0)
        for (int q = 0; q < nv; ++q) vv[q] += __ldg(P.bias + col + q);
      if (split) {
        if (vec && nv == 4) red_add_f4(dst, make_float4(vv[0], vv[1], vv[2], vv[3]));
        else for (int q = 0; q < nv; ++q) atomicAdd(dst + q, vv[q]);
      } else if (P.accumulate) {
        for (int q = 0; q < nv; ++q) dst[q] += vv[q];
      } else if (vec && nv == 4) {
        *reinterpret_cast<float4*>(dst) = make_float4(vv[0], vv[1], vv[2], vv[3]);
      } else {
        for (int q = 0; q < nv; ++q) dst[q] = vv[q];
      }
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  stamp(P, 5);                             // stores issued
  if (t < 32) tc::tmem_dealloc<TCOLS>(tmem);
  stamp(P, 6);
}

template <int BN, int A_MN, int B_MN>
int launch(brk_ctx* ctx, const Params& P, int splits, cudaStream_t st) {
  const size_t pipe = size_t(STAGES) * size_t(BM * KC * 4 + BN * KC * 4), stagec = size_t(BM) * (BN + 4) * 4;
  const size_t smem = (pipe > stagec ? pipe : stagec) + 1024;
  // the shared-memory opt-in is per device: set it for the current one on every call
  BRK_CUDA(cudaFuncSetAttribute(gemm_tf32_kernel<BN, A_MN, B_MN>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  // row and column tiles both on x: gridDim.y would cap M at 65535 row tiles
  dim3 grid(unsigned((P.N + BN - 1) / BN) * unsigned((P.M + BM - 1) / BM), 1, splits);
  gemm_tf32_kernel<BN, A_MN, B_MN><<<grid, NT, smem, st>>>(P);
  BRK_LAUNCH_CHECK();
  (void)ctx;
  return 0;
}

}  // namespace gtc

// Same contract as brk_sgemm (trans_a: A stored [K,M]; trans_b: B stored [N,K]); additionally lda / ldb / the
// operand bases must allow 16-byte loads (multiples of 4 floats, 16-byte aligned) and M, N >= 1.  Returns
// BRK_E_ALIGN when they do not -- the caller then takes brk_sgemm.
static int gemm_tf32_run(brk_ctx* ctx, const float* A, const float* B, float* C, const float* bias, int M, int N, int K, int lda,
                         int ldb, int ldc, int trans_a, int trans_b, float alpha, int accumulate, bool allow_split,
                         cudaStream_t st, unsigned long long* trace) {
  if ((lda & 3) || (ldb & 3) || !brk_aligned16(A) || !brk_aligned16(B)) {
    brk_set_error("brk_gemm_tf32: operands must be 16-byte aligned with leading dimensions that are multiples of 4");
    return BRK_E_ALIGN;
  }
  gtc::Params P;
  P.A = A; P.B = B; P.C = C; P.bias = bias; P.M = M; P.N = N; P.K = K; P.lda = lda; P.ldb = ldb; P.ldc = ldc;
  P.alpha = alpha; P.accumulate = accumulate; P.trace = trace;
  // Tile width: the widest of 128 / 64 / 32 that still gives the grid a quarter of a wave of CTAs.  Small products
  // (the two-tower Dense layers at batch 1000: 8 row tiles) are bound by the latency of ONE CTA -- staging, the
  // tcgen05.ld epilogue and the stores of a 128-wide tile -- so narrower tiles on more SMs finish sooner.
  const int row_tiles = (M + gtc::BM - 1) / gtc::BM;
  int BN = 128;
  while (BN > 32 && (BN / 2 >= N || row_tiles * ((N + BN - 1) / BN) < ctx->sm_count / 4)) BN /= 2;
  const int tiles = ((N + BN - 1) / BN) * row_tiles;
  int splits = 1;
  if (allow_split && accumulate) {
    const int want = ctx->sm_count / tiles, max_by_k = (K + 4 * gtc::KC - 1) / (4 * gtc::KC);
    splits = want < 1 ? 1 : (want < max_by_k ? want : max_by_k);
    if (splits > 64) splits = 64;
  }
  int kps = ((K + splits - 1) / splits + gtc::KC - 1) / gtc::KC * gtc::KC;
  splits = (K + kps - 1) / kps;
  P.k_per_split = kps;
  // this library's convention: trans_a = A stored [K, M] (M contiguous -> MN-major view);
  //                            trans_b = 0: B stored [K, N] (N contiguous -> MN-major view), 1: B stored [N, K] (K-major)
  const int a_mn = trans_a ? 1 : 0, b_mn = trans_b ? 0 : 1;
#define BRK_GTC(BN_, AM_, BM_) if (BN == BN_ && a_mn == AM_ && b_mn == BM_) return gtc::launch<BN_, AM_, BM_>(ctx, P, splits, st);
  BRK_GTC(128, 0, 0) BRK_GTC(128, 0, 1) BRK_GTC(128, 1, 0) BRK_GTC(128, 1, 1)
  BRK_GTC(64, 0, 0) BRK_GTC(64, 0, 1) BRK_GTC(64, 1, 0) BRK_GTC(64, 1, 1)
  BRK_GTC(32, 0, 0) BRK_GTC(32, 0, 1) BRK_GTC(32, 1, 0) BRK_GTC(32, 1, 1)
#undef BRK_GTC
  return BRK_E_ARG;
}

int brk_gemm_tf32_impl(brk_ctx* ctx, const float* A, const float* B, float* C, const float* bias, int M, int N, int K, int lda,
                       int ldb, int ldc, int trans_a, int trans_b, float alpha, int accumulate, bool allow_split,
                       cudaStream_t st) {
  return gemm_tf32_run(ctx, A, B, C, bias, M, N, K, lda, ldb, ldc, trans_a, trans_b, alpha, accumulate, allow_split, st, nullptr);
}

extern "C" int brk_gemm_tf32(brk_ctx* ctx, const float* A, const float* B, float* C, const float* bias, int32_t M, int32_t N,
                             int32_t K, int32_t lda, int32_t ldb, int32_t ldc, int32_t trans_a, int32_t trans_b, float alpha,
                             int32_t accumulate, void* stream) {
  BRK_REQUIRE(ctx && A && B && C, BRK_E_ARG, "brk_gemm_tf32: null argument");
  BRK_REQUIRE(M > 0 && N > 0 && K > 0, BRK_E_ARG, "brk_gemm_tf32: M=%d N=%d K=%d", M, N, K);
  BRK_REQUIRE(lda >= (trans_a ? M : K) && ldb >= (trans_b ? K : N) && ldc >= N, BRK_E_ARG,
              "brk_gemm_tf32: lda=%d ldb=%d ldc=%d below the stored row length (M=%d N=%d K=%d trans_a=%d trans_b=%d)", lda,
              ldb, ldc, M, N, K, trans_a, trans_b);
  return brk_gemm_tf32_impl(ctx, A, B, C, bias, M, N, K, lda, ldb, ldc, trans_a, trans_b, alpha, accumulate, true,
                            (cudaStream_t)stream);
}

// Diagnostics: the same product with CTA (0,0,0) writing %globaltimer (ns) into trace[0..6] at: kernel entry, TMEM
// allocated, first K chunk staged, all MMAs complete, accumulators copied to shared memory, stores issued, TMEM freed.
extern "C" int brk_gemm_tf32_trace(brk_ctx* ctx, const float* A, const float* B, float* C, const float* bias, int32_t M,
                                   int32_t N, int32_t K, int32_t lda, int32_t ldb, int32_t ldc, int32_t trans_a,
                                   int32_t trans_b, float alpha, int32_t accumulate, uint64_t* trace, void* stream) {
  BRK_REQUIRE(ctx && A && B && C && trace, BRK_E_ARG, "brk_gemm_tf32_trace: null argument");
  BRK_REQUIRE(M > 0 && N > 0 && K > 0, BRK_E_ARG, "brk_gemm_tf32_trace: M=%d N=%d K=%d", M, N, K);
  BRK_REQUIRE(lda >= (trans_a ? M : K) && ldb >= (trans_b ? K : N) && ldc >= N, BRK_E_ARG,
              "brk_gemm_tf32_trace: lda=%d ldb=%d ldc=%d below the stored row length (M=%d N=%d K=%d trans_a=%d trans_b=%d)", lda,
              ldb, ldc, M, N, K, trans_a, trans_b);
  return gemm_tf32_run(ctx, A, B, C, bias, M, N, K, lda, ldb, ldc, trans_a, trans_b, alpha, accumulate, true,
                       (cudaStream_t)stream, reinterpret_cast<unsigned long long*>(trace));
}
