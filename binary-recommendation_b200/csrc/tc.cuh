// sm_100a building blocks written as inline PTX: mbarrier, TMA (cp.async.bulk.tensor), TMEM
// allocation, tcgen05.mma / commit / ld, and the UMMA shared-memory / instruction descriptors.
// Bit layouts follow the PTX ISA "tcgen05" chapter (the same fields CUTLASS names in
// cute/arch/mma_sm100_desc.hpp); nothing here depends on CUTLASS.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier ---------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "MBAR_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra MBAR_DONE;\n"
      "bra MBAR_WAIT;\n"
      "MBAR_DONE:\n"
      "}\n" ::"r"(bar), "r"(parity) : "memory");
}

// ---- TMA --------------------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tiled load: c0 = innermost (element) coordinate, c1 = row coordinate.
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap* m, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1) : "memory");
}

// ---- TMEM -------------------------------------------------------------------------------------
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_slot) {   // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_slot), "n"(COLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {     // the same warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- descriptors --------------------------------------------------------------------------------
// K-major operand tile stored as rows of 128 bytes with the 128-byte swizzle (what a TMA box of
// 64 bf16 x R rows with CU_TENSOR_MAP_SWIZZLE_128B writes): 8-row groups are 1024 B apart (SBO),
// LBO is unused for this layout (set to 1), descriptor version 1 (sm_100), layout type 2 = SWIZZLE_128B.
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= uint64_t((smem_addr >> 4) & 0x3FFFu);
  d |= uint64_t(1) << 16;            // leading byte offset (16 B units), ignored for swizzled K-major
  d |= uint64_t(1024 >> 4) << 32;    // stride byte offset: 8 rows x 128 B
  d |= uint64_t(1) << 46;            // descriptor version (Blackwell)
  d |= uint64_t(2) << 61;            // SWIZZLE_128B
  return d;
}
// General shared-memory matrix descriptor, SWIZZLE_128B atoms (8 rows x 128 B, 1024-byte aligned):
//   K-major operand  (rows = M/N index, 128 B = the K extent of one K-block): LBO unused, SBO = 1024;
//   MN-major operand (rows = K index, 128 B = 32 fp32 / 64 bf16 along M/N):   LBO = distance between
//     128-byte column blocks along M/N, SBO = distance between 8-row groups along K.
__device__ __forceinline__ uint64_t smem_desc_sw128_ex(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= uint64_t((smem_addr >> 4) & 0x3FFFu);
  d |= uint64_t((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= uint64_t((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= uint64_t(1) << 46;            // descriptor version (Blackwell)
  d |= uint64_t(2) << 61;            // SWIZZLE_128B
  return d;
}
// MN-major TF32 operands only exist in the "128B swizzle, 32-byte base" form (layout type 1): rows = K index,
// 128 B = 32 fp32 along M/N, atoms of 4 rows (512 B), the 32-byte chunk index XORed with (row & 3).
__device__ __forceinline__ uint64_t smem_desc_sw128_base32(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= uint64_t((smem_addr >> 4) & 0x3FFFu);
  d |= uint64_t((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= uint64_t((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= uint64_t(1) << 46;            // descriptor version (Blackwell)
  d |= uint64_t(1) << 61;            // SWIZZLE_128B_BASE32B
  return d;
}
// kind::tf32 instruction descriptor: D = F32, A = B = TF32 (fp32 bits in shared memory, 10-bit mantissa used);
// a_mn / b_mn = 1 selects the MN-major (transposed) view of that operand.
__host__ __device__ constexpr uint32_t idesc_tf32_f32(int M, int N, int a_mn, int b_mn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (uint32_t(a_mn) << 15) | (uint32_t(b_mn) << 16) |
         (uint32_t(N >> 3) << 17) | (uint32_t(M >> 4) << 24);
}
// Generic-proxy shared-memory writes (st.shared) must be made visible to the async proxy that
// tcgen05.mma reads operands through.
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// kind::f16 instruction descriptor: D = F32, A = B = BF16, both K-major, M x N tile.
__host__ __device__ constexpr uint32_t idesc_bf16_f32(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(N >> 3) << 17) | (uint32_t(M >> 4) << 24);
}

// ---- MMA / commit / load -------------------------------------------------------------------------
__device__ __forceinline__ void mma_bf16_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mma_tf32_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// Arrives on the mbarrier when all previously issued tcgen05.mma of this thread have completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 lanes x 32 columns of 32-bit: thread i of the warp receives lane (base+i), columns c..c+31.
// Split into issue + wait so that a second load can be in flight while the first chunk is being
// processed.  The wait names the destination registers as in/out operands: that is what stops the
// compiler from scheduling a use of them above the wait.
__device__ __forceinline__ void tmem_ld_32x32_issue(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
      : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
        "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
        "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
        "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
      :: "memory");
}

// Narrower forms of the same load: 8 or 16 consecutive columns of the thread's lane (issue + wait in one call).
__device__ __forceinline__ void tmem_ld_32x32_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
      "tcgen05.wait::ld.sync.aligned;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
      "tcgen05.wait::ld.sync.aligned;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}

// ---- host: tensor maps through the driver entry point (no link-time libcuda dependency) -----------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// bf16 row-major [rows, cols] matrix, box = 64 columns (128 B, one swizzle span) x box_rows rows.
inline int make_tmap_bf16_sw128(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return -1;
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {cols * 2};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : int(r);
}

}  // namespace tc
