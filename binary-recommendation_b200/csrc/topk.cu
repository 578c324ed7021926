// K7/K8: full-catalog scoring fused with top-K selection.  Stands in for
// tfrs.layers.factorized_top_k.BruteForce(k).index(...) + call
// (/root/reference/trainers/twoTower.py:64-69,60-62,229-230; src/origin_models/svd/SVD.py:424-432),
// bpr_predict (src/models/bpr.py:122-133) and the streaming __topk of trainers/topKmetrics.py:51-72.
//
// scores = Q C^T is a tcgen05 GEMM (bf16 operands staged by TMA with the 128-byte swizzle, fp32
// accumulators in TMEM, M = 128 users x N = 128 items per MMA tile) whose epilogue never writes a
// score to HBM: each epilogue thread owns one user row (= one TMEM lane), pulls 32 scores at a time
// with tcgen05.ld, reduces them with a FMNMX3 max-tree and compares the chunk maximum with the row's
// running k-th best -- branch-free: the four chunk flags of a tile are voted on once per warp -- and
// only flagged chunks are read again for the exact sorted insertion.  Tie rule: strict '>' while items
// stream in ascending id, i.e. equal scores keep the lower item id (tf.math.top_k / the reference's __topk).
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer (one elected
// lane), warps 2-5 = epilogue: warp w reads TMEM lanes 32*(w%4)... of the whole 128-column tile.
// tcgen05.ld is double-buffered against the compare work, two 128-column accumulators double-buffer
// MMA against epilogue, and TWO CTAs share an SM (256 TMEM columns, <= 113 KB of shared memory each):
// the four epilogue warps of a CTA advance in lockstep with their MMA issuer -- the accumulator of
// tile t+2 is only free when the slowest warp has finished tile t -- and with one CTA per SM (round 1:
// 8 epilogue warps on 256-column tiles) they spent 24 % of their time waiting for it (ncu, r02); a
// second CTA fills those gaps: 4.04 -> 3.20 ms on the 65 536 x 250 k x 64 shard, 4.47 -> 3.77 ms at
// d = 128 (profiles/r02_topk_probe.txt).  Algorithmic traffic: 2*dpad B per user + 2*dpad B per item
// per m-tile pass (L2-resident item index) + 8k B of results per user.
#include "common.cuh"
#include "tc.cuh"
#include "topk_select.cuh"
#include <cuda_bf16.h>
#include <limits.h>
#include <math_constants.h>

namespace {

constexpr int kBM = 128;          // users per CTA (TMEM lanes)
constexpr int kBN = 128;          // items per MMA tile (TMEM columns per accumulator)
constexpr int kKBlock = 64;       // bf16 elements per 128-byte swizzle row
constexpr int kThreadsTopk = 192;
constexpr int kEpiWarps = 4;
constexpr int kHalves = 1;        // column parts per tile (epilogue warps per TMEM lane quadrant)
constexpr int kMaxKB = 4;         // dpad <= 256
constexpr uint32_t kABytesPerKB = kBM * 128;   // 16 KB
constexpr uint32_t kBBytes = kBN * 128;        // 32 KB per stage (one k-block of one item tile)

struct TopkParams {
  int64_t U, I;
  int32_t KB;            // k-blocks of 64 (dpad / 64)
  int32_t k;             // requested list length (<= K_CAP)
  int32_t n_tiles;       // item tiles in total
  int32_t tiles_per_split;
  int32_t stages;
  int32_t id_offset;     // added to local item ids (item-range shards)
  float* out_vals;       // [n_splits * kHalves, U, k]
  int32_t* out_ids;
  const int64_t* excl_indptr;   // EXCL only: [U + 1] absolute offsets into excl_ids
  const int32_t* excl_ids;      // EXCL only: excluded global ids, ascending within each row
};

// Exclusion cursor of one epilogue thread (EXCL instantiations): a pointer into its row's list, the entries left from
// there and the id it points at.  Static shared memory, not registers -- the kernel sits at the 168-register cap of two
// CTAs per SM -- touched only on the candidate path.  Budgeted as 4 KB (ptxas places 3 KB).
constexpr size_t kExclCursorBytes = 4096;

// Longest fused lists: 128 entries while dpad <= 128, 64 at dpad 192 and 256, where a 128-entry heap (128 KB) beside
// the 48 / 64 KB query tile leaves no room for two pipeline stages.  hotpath.fused_k_cap states the same caps.
constexpr int kHeapCap = 128;
constexpr int kHeapCapWide = 64;

// Lists longer than 32 (K_CAP = kHeapCap) keep a heap of k entries per row in dynamic shared memory, 128 x k x 8 B, so
// those instantiations run one CTA per SM.
template <int K_CAP, bool EXCL>
__global__ void __launch_bounds__(kThreadsTopk, K_CAP > 32 ? 1 : 2)
score_topk_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_c,
                  const TopkParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // slow-path scratch of the epilogue threads: STATIC shared memory, so that the compiler emits STS / LDS for it (carved
  // out of the dynamic block through a generic pointer it was 32 generic ST.E per spilled chunk)
  __shared__ float scratch_s[kEpiWarps * 32 * 32];
  __shared__ const int32_t* excl_cur_s[EXCL ? kEpiWarps * 32 : 1];
  __shared__ int32_t excl_left_s[EXCL ? kEpiWarps * 32 : 1];
  __shared__ int32_t excl_next_s[EXCL ? kEpiWarps * 32 : 1];
  // 1024-byte alignment for the 128-byte swizzle
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t smem_a = tc::smem_u32(smem);
  const uint32_t smem_b = smem_a + P.KB * kABytesPerKB;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + P.KB * kABytesPerKB + P.stages * kBBytes);
  // barrier map: [0,stages) full, [stages,2*stages) empty, then a_full, tmem_full[2], tmem_empty[2]
  const uint32_t bar0 = tc::smem_u32(bars);
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (P.stages + s); };
  const uint32_t a_full = bar0 + 8u * (2 * P.stages);
  auto tmem_full = [&](int b) { return bar0 + 8u * (2 * P.stages + 1 + b); };
  auto tmem_empty = [&](int b) { return bar0 + 8u * (2 * P.stages + 3 + b); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * P.stages + 5);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tile = blockIdx.x, split = blockIdx.y;
  const int tile_begin = split * P.tiles_per_split;
  const int tile_end = min(P.n_tiles, tile_begin + P.tiles_per_split);
  const int my_tiles = tile_end - tile_begin;

  if (warp == 0 && lane == 0) {
    tc::prefetch_tensormap(&tmap_q);
    tc::prefetch_tensormap(&tmap_c);
    for (int s = 0; s < P.stages; ++s) { tc::mbar_init(full_bar(s), 1); tc::mbar_init(empty_bar(s), 1); }
    tc::mbar_init(a_full, 1);
    for (int b = 0; b < 2; ++b) { tc::mbar_init(tmem_full(b), 1); tc::mbar_init(tmem_empty(b), kEpiWarps); }
    tc::fence_barrier_init();
  }
  if (warp == 1) tc::tmem_alloc<2 * kBN>(tc::smem_u32(tmem_slot));
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      tc::mbar_expect_tx(a_full, P.KB * kABytesPerKB);
      for (int kb = 0; kb < P.KB; ++kb)
        tc::tma_load_2d(smem_a + kb * kABytesPerKB, &tmap_q, kb * kKBlock, m_tile * kBM, a_full);
      int stage = 0; uint32_t phase = 0;
      for (int t = 0; t < my_tiles; ++t) {
        for (int kb = 0; kb < P.KB; ++kb) {
          tc::mbar_wait(empty_bar(stage), phase ^ 1);
          tc::mbar_expect_tx(full_bar(stage), kBBytes);
          tc::tma_load_2d(smem_b + stage * kBBytes, &tmap_c, kb * kKBlock, (tile_begin + t) * kBN, full_bar(stage));
          if (++stage == P.stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      constexpr uint32_t idesc = tc::idesc_bf16_f32(kBM, kBN);
      tc::mbar_wait(a_full, 0);
      int stage = 0; uint32_t phase = 0;
      for (int t = 0; t < my_tiles; ++t) {
        const int buf = t & 1;
        tc::mbar_wait(tmem_empty(buf), ((t >> 1) & 1) ^ 1);
        tc::fence_after_sync();
        const uint32_t d_tmem = tmem_base + buf * kBN;
        for (int kb = 0; kb < P.KB; ++kb) {
          tc::mbar_wait(full_bar(stage), phase);
          tc::fence_after_sync();
          const uint64_t adesc = tc::smem_desc_sw128(smem_a + kb * kABytesPerKB);
          const uint64_t bdesc = tc::smem_desc_sw128(smem_b + stage * kBBytes);
#pragma unroll
          for (int k4 = 0; k4 < kKBlock / 16; ++k4)   // UMMA_K = 16 bf16 = 32 B inside the swizzle row
            tc::mma_bf16_ss(d_tmem, adesc + uint64_t(k4 * 2), bdesc + uint64_t(k4 * 2), idesc, (kb | k4) != 0);
          tc::mma_commit(empty_bar(stage));            // smem slot free once these MMAs retire
          if (++stage == P.stages) { stage = 0; phase ^= 1; }
        }
        tc::mma_commit(tmem_full(buf));                // accumulator ready for the epilogue
      }
    }
  } else {
    // ===== epilogue: threshold filter + exact top-K per user row =====
    const int quad = warp & 3;                          // TMEM lane quadrant this warp may read
    const int half = (warp - 2) >> 2;                   // which 128-column half of each tile
    const int64_t row = int64_t(m_tile) * kBM + quad * 32 + lane;
    // The row's running list.  K_CAP <= 32: K_CAP entries in registers, sorted (topk_insert).  Longer lists: a min-heap
    // of exactly k entries in shared memory behind the barriers (topk_heap_*), so that `thr` is the row's k-th best.
    constexpr bool kHeap = K_CAP > 32;
    float vals[kHeap ? 1 : K_CAP]; int32_t ids[kHeap ? 1 : K_CAP];
    // (addressed from smem_raw, not through `smem`, so that the compiler emits LDS / STS rather than generic loads)
    TopkEntry* heap = reinterpret_cast<TopkEntry*>(smem_raw + (smem - smem_raw) + P.KB * kABytesPerKB + P.stages * kBBytes + 256) +
                      (threadIdx.x - 64);
    if constexpr (kHeap) {
      topk_heap_init(heap, kBM, P.k);
    } else {
#pragma unroll
      for (int j = 0; j < K_CAP; ++j) { vals[j] = -CUDART_INF_F; ids[j] = -1; }
    }
    float thr = -CUDART_INF_F;
    auto insert = [&](float x, int32_t id) {              // precondition: x > thr
      if constexpr (kHeap) {
        thr = topk_heap_replace_root(heap, kBM, P.k, TopkEntry{x, id});
      } else {
        topk_insert<K_CAP>(vals, ids, x, id);
        thr = vals[K_CAP - 1];
      }
    };
    constexpr int kChunks = kBN / kHalves / 32;         // 4 chunks of 32 columns per tile per warp

    // Slow-path scratch: 32 floats per epilogue thread, column-major so that lane i of a warp hits
    // bank i (conflict-free).  Keeps ONE compact copy of the insertion code (a dynamic loop) instead
    // of 32 unrolled copies per call site -- the unrolled form overflowed the instruction cache.
    float* scratch = scratch_s + (threadIdx.x - 64);
    constexpr int kScratchStride = kEpiWarps * 32;

    // Exclusions: the thread meets its row's candidates in ascending global id (tiles, flagged chunks and mask bits
    // all ascend), so one monotone cursor into the row's ascending list answers every membership test.  It starts at
    // the first listed id >= this split's first id; rows >= U (padding of the last m-tile) get an empty list.
    if constexpr (EXCL) {
      const int e = threadIdx.x - 64;
      int64_t pos = 0, end = 0;
      if (row < P.U) {
        pos = P.excl_indptr[row];
        end = P.excl_indptr[row + 1];
        const int64_t first = int64_t(tile_begin) * kBN + P.id_offset;
        int64_t hi = end;
        while (pos < hi) {                                // lower bound of `first`
          const int64_t mid = pos + ((hi - pos) >> 1);
          if (P.excl_ids[mid] < first) pos = mid + 1; else hi = mid;
        }
      }
      const int64_t left = end - pos;                     // a row lists at most I < 2^31 distinct ids
      excl_cur_s[e] = P.excl_ids + pos;
      excl_left_s[e] = int32_t(left < INT_MAX ? left : INT_MAX);
      excl_next_s[e] = pos < end ? P.excl_ids[pos] : INT_MAX;
    }
    // Listed ids of the 32 columns starting at global id `lo`, as a bit mask (EXCL only).  Advances the cursor past
    // lo + 31; chunks must be presented in ascending order.  Applied to a chunk's candidate mask before the insertion
    // loop, so that loop carries no extra register (a per-candidate test there spilled the register list).
    auto excluded_bits = [&](int32_t lo) -> uint32_t {
      const int e = threadIdx.x - 64;
      int32_t next = excl_next_s[e];
      if (next >= lo + 32) return 0u;                    // the launcher keeps lo + 32 <= INT_MAX
      const int32_t* cur = excl_cur_s[e];
      int32_t left = excl_left_s[e];
      uint32_t bits = 0u;
      do {
        if (next >= lo) bits |= 1u << (next - lo);
        next = (--left > 0) ? *++cur : INT_MAX;
      } while (next < lo + 32);
      excl_cur_s[e] = cur;
      excl_left_s[e] = left;
      excl_next_s[e] = next;
      return bits;
    };

#define V(j) __uint_as_float(r[(j)])
    // A chunk of the last item tile, which can be ragged: every column is bounds-checked on its own.
    auto process_ragged = [&](uint32_t (&r)[32], int64_t col0) {
#pragma unroll
      for (int j = 0; j < 32; ++j) scratch[j * kScratchStride] = V(j);
      uint32_t live = 0xffffffffu;                        // EXCL: columns not listed
      if constexpr (EXCL) live = ~excluded_bits(int32_t(col0) + P.id_offset);
#pragma unroll 1
      for (int j = 0; j < 32; ++j) {
        const float x = scratch[j * kScratchStride];
        if (col0 + j < P.I && x > thr) {
          if constexpr (EXCL) {
            if (!((live >> j) & 1u)) continue;
          }
          insert(x, int32_t(col0 + j) + P.id_offset);
        }
      }
    };

    // A flagged chunk of a full tile.  The scores are used straight out of the registers tcgen05.ld filled: copying them
    // into a float array cost 32 moves per 32 scores, more than the max-tree itself.
    auto process_flagged = [&](uint32_t (&r)[32], int64_t col0) {
      // 4 independent FMNMX3 chains, one per group of 8 columns
      float gm[4];
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float m = fmaxf(fmaxf(V(8 * g), V(8 * g + 1)), V(8 * g + 2));
        m = fmaxf(fmaxf(m, V(8 * g + 3)), V(8 * g + 4));
        m = fmaxf(fmaxf(m, V(8 * g + 5)), V(8 * g + 6));
        gm[g] = fmaxf(m, V(8 * g + 7));
      }
      const float cmax = fmaxf(fmaxf(fmaxf(gm[0], gm[1]), gm[2]), gm[3]);
      if (cmax > thr) {
        // candidates = bitmask of columns beating the threshold; only groups whose max beats it are
        // examined and spilled.  The loop below then runs once per candidate (usually once).
        uint32_t mask = 0u;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          if (gm[g] > thr) {
#pragma unroll
            for (int j = 8 * g; j < 8 * g + 8; ++j) {
              scratch[j * kScratchStride] = V(j);
              mask |= (V(j) > thr) ? (1u << j) : 0u;
            }
          }
        }
        if constexpr (EXCL) mask &= ~excluded_bits(int32_t(col0) + P.id_offset);
#pragma unroll 1
        while (mask) {                                  // ascending column = ascending item id
          const int j = __ffs(mask) - 1;
          mask &= mask - 1;
          const float x = scratch[j * kScratchStride];
          if (x > thr) {
            insert(x, int32_t(col0 + j) + P.id_offset);
          }
        }
      }
    };
#undef V

    // max of a 32-score chunk: 4 independent FMNMX3 chains (one per group of 8 columns), no branch
    auto chunk_max = [&](const uint32_t (&r)[32]) -> float {
#define V(j) __uint_as_float(r[(j)])
      float gm[4];
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float m = fmaxf(fmaxf(V(8 * g), V(8 * g + 1)), V(8 * g + 2));
        m = fmaxf(fmaxf(m, V(8 * g + 3)), V(8 * g + 4));
        m = fmaxf(fmaxf(m, V(8 * g + 5)), V(8 * g + 6));
        gm[g] = fmaxf(m, V(8 * g + 7));
      }
#undef V
      return fmaxf(fmaxf(fmaxf(gm[0], gm[1]), gm[2]), gm[3]);
    };

    for (int t = 0; t < my_tiles; ++t) {
      const int buf = t & 1;
      tc::mbar_wait(tmem_full(buf), (t >> 1) & 1);
      tc::fence_after_sync();
      const int64_t col_half = int64_t(tile_begin + t) * kBN + half * (kBN / kHalves);
      const bool ragged = col_half + kBN / kHalves > P.I;   // only in the last item tile
      const uint32_t taddr = tmem_base + (uint32_t(quad * 32) << 16) + buf * kBN + half * (kBN / kHalves);
      uint32_t ra[32], rb[32];
      if (ragged) {                                       // last item tile: chunk by chunk
        tc::tmem_ld_32x32_issue(taddr, ra);
        tc::tmem_ld_wait(ra);
#pragma unroll 1
        for (int c = 0; c < kChunks; c += 2) {
          tc::tmem_ld_32x32_issue(taddr + (c + 1) * 32, rb);     // in flight while chunk c is processed
          process_ragged(ra, col_half + c * 32);
          tc::tmem_ld_wait(rb);
          if (c + 2 < kChunks) tc::tmem_ld_32x32_issue(taddr + (c + 2) * 32, ra);
          process_ragged(rb, col_half + (c + 1) * 32);
          if (c + 2 < kChunks) tc::tmem_ld_wait(ra);
        }
      } else {
        // The common case has NO branch per chunk: the four chunk maxima are compared with the row's k-th best (as it
        // stood at the start of the tile: it only rises, so this flags a superset) into a 4-bit mask, and ONE warp-wide
        // vote per tile decides whether anything has to be looked at again.  (With a compare-and-branch and two uniform
        // checks per chunk the epilogue ran at 15-17 scores/clk/SM against 29 for the bare TMEM drain: the ~5 branches per
        // chunk, not the max-tree, were the cost, and one extra uniform branch per chunk alone cost 11 % --
        // profiles/r02_topk_probe.txt.)
        static_assert(kChunks == 4, "the tile epilogue is written out for four 32-column chunks per warp");
        uint32_t flagged = 0u;
        tc::tmem_ld_32x32_issue(taddr, ra);
        tc::tmem_ld_wait(ra);
        tc::tmem_ld_32x32_issue(taddr + 32, rb);
        flagged |= chunk_max(ra) > thr ? 1u : 0u;
        tc::tmem_ld_wait(rb);
        tc::tmem_ld_32x32_issue(taddr + 64, ra);
        flagged |= chunk_max(rb) > thr ? 2u : 0u;
        tc::tmem_ld_wait(ra);
        tc::tmem_ld_32x32_issue(taddr + 96, rb);
        flagged |= chunk_max(ra) > thr ? 4u : 0u;
        tc::tmem_ld_wait(rb);
        flagged |= chunk_max(rb) > thr ? 8u : 0u;
        // chunks some lane of the warp has to look at again.  They are read out of TMEM a second time (the accumulator is
        // still ours): keeping all four chunks in registers and inlining the candidate path four times measured slower
        // (instruction cache: 4.34 vs 4.04 ms on the 65 536 x 250 k shard)
        uint32_t todo = __reduce_or_sync(0xffffffffu, flagged);
#pragma unroll 1
        while (todo) {                                    // ascending chunk = ascending item id
          const int c = __ffs(todo) - 1;
          todo &= todo - 1;
          tc::tmem_ld_32x32_issue(taddr + c * 32, ra);
          tc::tmem_ld_wait(ra);
          process_flagged(ra, col_half + c * 32);
        }
      }
      tc::fence_before_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(tmem_empty(buf));
    }
    if (row < P.U) {
      const int64_t part = int64_t(split) * kHalves + half;
      float* ov = P.out_vals + (part * P.U + row) * P.k;
      int32_t* oi = P.out_ids + (part * P.U + row) * P.k;
      if constexpr (kHeap) {
        topk_heap_sort(heap, kBM, P.k);
#pragma unroll 1
        for (int j = 0; j < P.k; ++j) { const TopkEntry e = heap[j * kBM]; ov[j] = e.v; oi[j] = e.id; }
      } else {
#pragma unroll
        for (int j = 0; j < K_CAP; ++j)
          if (j < P.k) { ov[j] = vals[j]; oi[j] = ids[j]; }
      }
    }
  }

  tc::fence_before_sync();
  __syncthreads();
  if (warp == 1) tc::tmem_dealloc<2 * kBN>(tmem_base);
}

// Merge S sorted partial lists per user into one: score descending, id ascending on ties --
// identical to an unsharded scan (used for item splits inside a GPU and for item-range shards
// across GPUs).  One thread per user; S*k is small.
__global__ void __launch_bounds__(256)
topk_merge_kernel(const float* __restrict__ pv, const int32_t* __restrict__ pi, int S, int64_t U, int k,
                  float* __restrict__ ov, int32_t* __restrict__ oi) {
  const int64_t u = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (u >= U) return;
  int head[64];
  for (int s = 0; s < S; ++s) head[s] = 0;
  for (int j = 0; j < k; ++j) {
    int best = -1; float bv = 0.f; int32_t bi = 0;
    for (int s = 0; s < S; ++s) {
      if (head[s] >= k) continue;
      const int64_t o = (int64_t(s) * U + u) * k + head[s];
      const int32_t id = pi[o];
      if (id < 0) { head[s] = k; continue; }           // exhausted list (fewer than k candidates)
      const float v = pv[o];
      if (best < 0 || v > bv || (v == bv && id < bi)) { best = s; bv = v; bi = id; }
    }
    if (best < 0) { ov[u * k + j] = -CUDART_INF_F; oi[u * k + j] = -1; }
    else { ov[u * k + j] = bv; oi[u * k + j] = bi; ++head[best]; }
  }
}

// The same merge for the long lists of the heap form (k > 32, S <= 32 item splits): one warp per user, lane s holding
// the head of list s.  Each output entry is one warp arg-max (score desc, id asc; ids are distinct across splits) and
// the winning lane steps its list.  topk_merge_kernel's thread per user walks S*k entries one dependent load after the
// other: 2.09 ms at S = 32, k = 128 for 128 users, against 0.048 ms here (B200 at 1000 W, profiles/r08_topk_long.json).
__global__ void __launch_bounds__(256)
topk_merge_warp_kernel(const float* __restrict__ pv, const int32_t* __restrict__ pi, int S, int64_t U, int k,
                       float* __restrict__ ov, int32_t* __restrict__ oi) {
  const int lane = threadIdx.x & 31;
  const int64_t u = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (u >= U) return;
  const int64_t base = (int64_t(lane) * U + u) * k;   // list `lane` of user u (lane < S)
  int h = 0;
  float v = -CUDART_INF_F; int32_t id = -1;           // the lane's head; id < 0: no list or exhausted
  auto load = [&]() {
    id = (lane < S && h < k) ? pi[base + h] : -1;
    v = id >= 0 ? pv[base + h] : -CUDART_INF_F;
  };
  load();
  for (int j = 0; j < k; ++j) {
    float bv = v; int32_t bi = id;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float v2 = __shfl_xor_sync(0xffffffffu, bv, o);
      const int32_t i2 = __shfl_xor_sync(0xffffffffu, bi, o);
      if (i2 >= 0 && (bi < 0 || v2 > bv || (v2 == bv && i2 < bi))) { bv = v2; bi = i2; }
    }
    if (lane == 0) { ov[u * k + j] = bi < 0 ? -CUDART_INF_F : bv; oi[u * k + j] = bi; }
    if (bi >= 0 && id == bi) { ++h; load(); }
  }
}

// The merge of item-range lists that live in other GPUs' memory (brk_topk_merge_peer).  A peer's list is read in bulk:
// each CTA copies the [users, k] rows of its block of kMergeUsers users from every part into shared memory with 16-byte
// loads (one contiguous span per part and array), then one warp per user merges on chip, lane s holding the head of
// part s.  Each output entry scans the heads in part order with topk_merge_kernel's comparison, so the result equals
// that kernel's for any input, duplicate ids and equal scores across parts included.  Before anything is written every
// CTA checks each part's header {seq, U, k} against part 0's seq and the caller's U and k; on a mismatch it returns,
// and CTA 0 reports it in *err.
constexpr int kMergeUsers = 8;                         // users (= warps) per CTA

__device__ __forceinline__ void stage_span(void* dst, const void* src, int64_t n_words) {
  const int t = threadIdx.x, nt = blockDim.x;
  uint32_t* d = static_cast<uint32_t*>(dst);
  const uint32_t* s = static_cast<const uint32_t*>(src);
  int64_t head = 0;
  if ((reinterpret_cast<uintptr_t>(s) & 15) == 0 && (reinterpret_cast<uintptr_t>(d) & 15) == 0) {
    const int64_t n4 = n_words >> 2;
    for (int64_t q = t; q < n4; q += nt) reinterpret_cast<uint4*>(d)[q] = reinterpret_cast<const uint4*>(s)[q];
    head = n4 << 2;
  }
  for (int64_t q = head + t; q < n_words; q += nt) d[q] = s[q];
}

__global__ void __launch_bounds__(kMergeUsers * 32)
topk_merge_peer_kernel(const float* const* __restrict__ part_vals, const int32_t* const* __restrict__ part_ids,
                       const int32_t* const* __restrict__ part_hdr, int S, int64_t U, int k, float* __restrict__ ov,
                       int32_t* __restrict__ oi, int32_t* __restrict__ err) {
  extern __shared__ __align__(16) unsigned char merge_smem[];
  __shared__ int bad;
  if (threadIdx.x == 0) {
    bad = 0;
    const int32_t seq = part_hdr[0][0];
    for (int s = 0; s < S; ++s) {
      const int32_t* h = part_hdr[s];
      if (!bad && (h[0] != seq || int64_t(h[1]) != U || h[2] != k)) bad = 1 + s;
    }
    if (bad && blockIdx.x == 0) *err = bad;
  }
  __syncthreads();
  if (bad) return;

  const int64_t u0 = int64_t(blockIdx.x) * kMergeUsers;
  const int nb = int(U - u0 < kMergeUsers ? U - u0 : kMergeUsers);
  const int span = nb * k;                             // entries of one part for this block
  const int stride = kMergeUsers * k;                  // shared-memory stride between parts (a multiple of 8 entries)
  float* sv = reinterpret_cast<float*>(merge_smem);
  int32_t* si = reinterpret_cast<int32_t*>(sv + int64_t(S) * stride);
  for (int s = 0; s < S; ++s) {
    stage_span(sv + s * stride, part_vals[s] + u0 * k, span);
    stage_span(si + s * stride, part_ids[s] + u0 * k, span);
  }
  __syncthreads();

  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (w >= nb) return;
  const float* lv = sv + lane * stride + w * k;        // lane < S: part `lane`'s list of user u0 + w
  const int32_t* li = si + lane * stride + w * k;
  int h = 0;
  float v = -CUDART_INF_F; int32_t id = -1;            // the lane's head; id < 0: no part or exhausted
  if (lane < S) { id = li[0]; v = lv[0]; }
  const int64_t o = (u0 + w) * k;
  for (int j = 0; j < k; ++j) {
    int best = -1; float bv = 0.f; int32_t bi = 0;
    for (int s = 0; s < S; ++s) {
      const float v2 = __shfl_sync(0xffffffffu, v, s);
      const int32_t i2 = __shfl_sync(0xffffffffu, id, s);
      if (i2 < 0) continue;
      if (best < 0 || v2 > bv || (v2 == bv && i2 < bi)) { best = s; bv = v2; bi = i2; }
    }
    if (lane == 0) {
      if (best < 0) { ov[o + j] = -CUDART_INF_F; oi[o + j] = -1; }
      else { ov[o + j] = bv; oi[o + j] = bi; }
    }
    if (lane == best) {
      ++h;
      if (h < k) { id = li[h]; v = lv[h]; } else id = -1;
      if (id < 0) v = -CUDART_INF_F;
    }
  }
}

__global__ void __launch_bounds__(256)
rows_to_bf16_kernel(const float* __restrict__ src, int64_t rows, int d, __nv_bfloat16* __restrict__ dst, int dpad) {
  const int64_t n = rows * dpad;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t r = i / dpad; const int c = int(i - r * dpad);
    dst[i] = __float2bfloat16_rn(c < d ? __ldg(src + r * d + c) : 0.f);
  }
}

// Warp-level top-K over rows of a materialised score matrix (models without a factorised scorer,
// e.g. NeuMF: /root/reference/trainers/topKmetrics.py:29-33 + __topk :51-72).  One warp per row: each
// lane keeps a sorted register list over its strided columns, then k rounds of a shuffle arg-max
// (score desc, column asc) pop the winners.  4 B read per score.
template <int K_CAP>
__global__ void __launch_bounds__(256)
topk_rows_kernel(const float* __restrict__ scores, int64_t R, int64_t I, int k, float* __restrict__ ov,
                 int32_t* __restrict__ oi) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (row >= R) return;
  float vals[K_CAP]; int32_t ids[K_CAP];
#pragma unroll
  for (int j = 0; j < K_CAP; ++j) { vals[j] = -CUDART_INF_F; ids[j] = 0x7fffffff; }
  const float* sr = scores + row * I;
  for (int64_t c = lane; c < I; c += 32) {
    const float v = __ldg(sr + c);
    if (v > vals[K_CAP - 1]) topk_insert<K_CAP>(vals, ids, v, int32_t(c));
  }
  for (int j = 0; j < k; ++j) {
    float bv = vals[0]; int32_t bi = ids[0];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov2 = __shfl_xor_sync(0xffffffffu, bv, o);
      const int32_t oi2 = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov2 > bv || (ov2 == bv && oi2 < bi)) { bv = ov2; bi = oi2; }
    }
    if (lane == 0) { ov[row * k + j] = bv; oi[row * k + j] = bi == 0x7fffffff ? -1 : bi; }
    if (ids[0] == bi && vals[0] == bv) {                 // the winning lane pops its head
#pragma unroll
      for (int q = 0; q < K_CAP - 1; ++q) { vals[q] = vals[q + 1]; ids[q] = ids[q + 1]; }
      vals[K_CAP - 1] = -CUDART_INF_F; ids[K_CAP - 1] = 0x7fffffff;
    }
  }
}

// Excluded items of materialised score rows: scores[r, id - col_offset] = -inf for every id of row r's list inside
// [col_offset, col_offset + I).  One warp per row, lanes striding the list.  topk_rows_kernel never inserts -inf, so
// masking followed by it selects among the remaining columns and pads with -1 like the fused path.
__global__ void __launch_bounds__(256)
mask_excluded_kernel(float* __restrict__ scores, int64_t R, int64_t I, int32_t col_offset,
                     const int64_t* __restrict__ indptr, const int32_t* __restrict__ ids) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (row >= R) return;
  const int64_t end = indptr[row + 1];
  for (int64_t p = indptr[row] + lane; p < end; p += 32) {
    const int64_t c = int64_t(__ldg(ids + p)) - col_offset;
    if (c >= 0 && c < I) scores[row * I + c] = -CUDART_INF_F;
  }
}

template <int K_CAP, bool EXCL>
int launch_topk(const CUtensorMap& tq, const CUtensorMap& tcm, const TopkParams& P, dim3 grid, size_t smem,
                cudaStream_t st) {
  BRK_CUDA(cudaFuncSetAttribute(score_topk_kernel<K_CAP, EXCL>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  if constexpr (K_CAP > 32) {                         // the heap form is planned for one resident CTA per SM
    int per_sm = 0;
    BRK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, score_topk_kernel<K_CAP, EXCL>, kThreadsTopk, smem));
    BRK_REQUIRE(per_sm >= 1, BRK_E_STATE, "brk_score_topk_bf16: %zu bytes of shared memory do not fit an SM", smem);
  }
  score_topk_kernel<K_CAP, EXCL><<<grid, kThreadsTopk, smem, st>>>(tq, tcm, P);
  BRK_LAUNCH_CHECK();
  return 0;
}

// Item splits for small user counts: enough CTAs for every slot (`slots` = SMs x CTAs per SM at this row width)
int plan_splits(int slots, int64_t U, int64_t I, int* n_splits, int* tiles_per_split) {
  const int64_t m_tiles = (U + kBM - 1) / kBM;
  const int n_tiles = int((I + kBN - 1) / kBN);
  int S = 1;
  if (m_tiles < slots) S = int((slots + m_tiles - 1) / m_tiles);
  if (S > n_tiles) S = n_tiles;
  if (S > 32) S = 32;
  if (S < 1) S = 1;
  const int tps = (n_tiles + S - 1) / S;
  *tiles_per_split = tps;
  *n_splits = (n_tiles + tps - 1) / tps;
  return n_tiles;
}

}  // namespace

extern "C" int32_t brk_bf16_padded_dim(int32_t d) { return (d + kKBlock - 1) / kKBlock * kKBlock; }

extern "C" int brk_rows_to_bf16(brk_ctx* ctx, const float* src, int64_t rows, int32_t d, uint16_t* dst,
                                int32_t dpad, void* stream) {
  BRK_REQUIRE(ctx && (rows == 0 || (src && dst)), BRK_E_ARG, "brk_rows_to_bf16: null argument");
  BRK_REQUIRE(rows >= 0 && d > 0 && dpad >= d, BRK_E_ARG, "brk_rows_to_bf16: rows=%lld d=%d dpad=%d",
              (long long)rows, d, dpad);
  if (rows == 0) return 0;
  const int64_t n = rows * dpad;
  int64_t need = (n + 255) / 256;
  const int64_t cap = int64_t(ctx->sm_count) * 8;
  rows_to_bf16_kernel<<<int(need < cap ? need : cap), 256, 0, (cudaStream_t)stream>>>(
      src, rows, d, reinterpret_cast<__nv_bfloat16*>(dst), dpad);
  BRK_LAUNCH_CHECK();
  return 0;
}

extern "C" int64_t brk_score_topk_workspace_bytes(brk_ctx* ctx, int64_t U, int64_t I, int32_t k) {
  if (!ctx || U <= 0 || I <= 0 || k <= 0) return 0;
  int S, tps;
  plan_splits(2 * ctx->sm_count, U, I, &S, &tps);      // the most any row width asks for
  return int64_t(S) * kHalves * U * k * 8;
}

namespace {

// brk_score_topk_bf16 (excl_indptr == nullptr: the EXCL = false kernels) and brk_score_topk_bf16_excl
int score_topk(brk_ctx* ctx, const uint16_t* q_bf16, int64_t U, const uint16_t* c_bf16, int64_t I, int32_t dpad,
               int32_t k, int32_t id_offset, const int64_t* excl_indptr, const int32_t* excl_ids, float* out_vals,
               int32_t* out_ids, void* workspace, int64_t workspace_bytes, void* stream) {
  BRK_REQUIRE(ctx && q_bf16 && c_bf16 && out_vals && out_ids, BRK_E_ARG, "brk_score_topk_bf16: null argument");
  const bool excl = excl_indptr != nullptr;
  BRK_REQUIRE(U > 0 && I > 0 && U < (int64_t(1) << 31) && I < (int64_t(1) << 31), BRK_E_ARG,
              "brk_score_topk_bf16: U=%lld I=%lld", (long long)U, (long long)I);
  BRK_REQUIRE(dpad > 0 && dpad % kKBlock == 0 && dpad / kKBlock <= kMaxKB, BRK_E_ARG,
              "brk_score_topk_bf16: dpad=%d must be a multiple of %d and <= %d", dpad, kKBlock, kKBlock * kMaxKB);
  BRK_REQUIRE(k >= 1 && k <= kHeapCap, BRK_E_ARG, "brk_score_topk_bf16: k=%d (1..%d)", k, kHeapCap);
  BRK_REQUIRE(dpad <= 128 || k <= kHeapCapWide, BRK_E_ARG, "brk_score_topk_bf16: k=%d at dpad=%d (k <= %d above dpad 128)",
              k, dpad, kHeapCapWide);
  BRK_REQUIRE(brk_aligned16(q_bf16) && brk_aligned16(c_bf16), BRK_E_ALIGN, "brk_score_topk_bf16: operands must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;

  TopkParams P;
  P.U = U; P.I = I; P.KB = dpad / kKBlock; P.k = k; P.id_offset = id_offset;
  P.excl_indptr = excl_indptr; P.excl_ids = excl_ids;
  const bool heap = k > 32;
  const size_t a_bytes = size_t(P.KB) * kABytesPerKB;
  const size_t heap_bytes = heap ? size_t(kBM) * k * sizeof(TopkEntry) : 0;
  constexpr size_t kScratchBytes = size_t(kEpiWarps) * 32 * 32 * sizeof(float);   // 16 KB
  // two CTAs per SM (each with its own pair of TMEM accumulators) when the query tile and the lists leave room: while one
  // CTA's epilogue warps wait for their next accumulator the other's keep the SM busy
  const bool two_ctas = a_bytes <= 32 * 1024 && !heap;
  int S, tps;
  P.n_tiles = plan_splits(ctx->sm_count * (two_ctas ? 2 : 1), U, I, &S, &tps);
  P.tiles_per_split = tps;
  const int64_t budget = two_ctas ? int64_t(113) * 1024 : int64_t(227) * 1024;
  int stages = int((budget - 1024 - 256 - int64_t(kScratchBytes) - (excl ? int64_t(kExclCursorBytes) : 0) - int64_t(a_bytes) -
                    int64_t(heap_bytes)) / int64_t(kBBytes));
  if (stages > 6) stages = 6;
  BRK_REQUIRE(stages >= 2, BRK_E_ARG, "brk_score_topk_bf16: no room for a 2-stage pipeline at dpad=%d k=%d", dpad, k);
  P.stages = stages;
  // + kScratchBytes (+ kExclCursorBytes) of static shared memory; the heaps follow the 256 bytes of barriers
  const size_t smem = 1024 + a_bytes + size_t(stages) * kBBytes + 256 + heap_bytes;

  const int parts = S * kHalves;                       // partial lists per user row
  const int64_t need = int64_t(parts) * U * k * 8;
  BRK_REQUIRE(workspace && workspace_bytes >= need, BRK_E_ARG,
              "brk_score_topk_bf16: workspace of %lld bytes needed, %lld given", (long long)need,
              (long long)workspace_bytes);
  float* pv = reinterpret_cast<float*>(workspace);
  int32_t* pi = reinterpret_cast<int32_t*>(pv + int64_t(parts) * U * k);
  // a heap-form launch without item splits writes the final lists: merging one list is a copy, 1.05 ms of a 28.8 ms call
  // at 65 536 x 250 000, k = 128 on a B200
  const bool direct = heap && parts == 1;
  P.out_vals = direct ? out_vals : pv; P.out_ids = direct ? out_ids : pi;

  CUtensorMap tq, tcm;
  BRK_REQUIRE(tc::make_tmap_bf16_sw128(&tq, q_bf16, uint64_t(U), uint64_t(dpad), kBM) == 0, BRK_E_STATE,
              "brk_score_topk_bf16: cuTensorMapEncodeTiled failed for the query matrix");
  BRK_REQUIRE(tc::make_tmap_bf16_sw128(&tcm, c_bf16, uint64_t(I), uint64_t(dpad), kBN) == 0, BRK_E_STATE,
              "brk_score_topk_bf16: cuTensorMapEncodeTiled failed for the candidate matrix");

  const dim3 grid(unsigned((U + kBM - 1) / kBM), unsigned(S));
  int rc;
  if (k <= 10) rc = excl ? launch_topk<10, true>(tq, tcm, P, grid, smem, st) : launch_topk<10, false>(tq, tcm, P, grid, smem, st);
  else if (k <= 16) rc = excl ? launch_topk<16, true>(tq, tcm, P, grid, smem, st) : launch_topk<16, false>(tq, tcm, P, grid, smem, st);
  else if (k <= 32) rc = excl ? launch_topk<32, true>(tq, tcm, P, grid, smem, st) : launch_topk<32, false>(tq, tcm, P, grid, smem, st);
  else rc = excl ? launch_topk<kHeapCap, true>(tq, tcm, P, grid, smem, st) : launch_topk<kHeapCap, false>(tq, tcm, P, grid, smem, st);
  if (rc || direct) return rc;
  if (heap)
    topk_merge_warp_kernel<<<unsigned((U * 32 + 255) / 256), 256, 0, st>>>(pv, pi, parts, U, k, out_vals, out_ids);
  else
    topk_merge_kernel<<<unsigned((U + 255) / 256), 256, 0, st>>>(pv, pi, parts, U, k, out_vals, out_ids);
  BRK_LAUNCH_CHECK();
  return 0;
}

}  // namespace

extern "C" int brk_score_topk_bf16(brk_ctx* ctx, const uint16_t* q_bf16, int64_t U, const uint16_t* c_bf16,
                                   int64_t I, int32_t dpad, int32_t k, int32_t id_offset, float* out_vals,
                                   int32_t* out_ids, void* workspace, int64_t workspace_bytes, void* stream) {
  return score_topk(ctx, q_bf16, U, c_bf16, I, dpad, k, id_offset, nullptr, nullptr, out_vals, out_ids, workspace,
                    workspace_bytes, stream);
}

extern "C" int brk_score_topk_bf16_excl(brk_ctx* ctx, const uint16_t* q_bf16, int64_t U, const uint16_t* c_bf16,
                                        int64_t I, int32_t dpad, int32_t k, int32_t id_offset,
                                        const int64_t* excl_indptr, const int32_t* excl_ids, float* out_vals,
                                        int32_t* out_ids, void* workspace, int64_t workspace_bytes, void* stream) {
  BRK_REQUIRE(excl_indptr && excl_ids, BRK_E_ARG, "brk_score_topk_bf16_excl: null exclusion list");
  // the kernel's exclusion cursor ends on INT_MAX and looks 32 ids past a chunk's first: every chunk of every item tile
  // must stay below it
  BRK_REQUIRE(int64_t(id_offset) + (I + kBN - 1) / kBN * kBN < int64_t(INT_MAX), BRK_E_ARG,
              "brk_score_topk_bf16_excl: id_offset=%d + I=%lld reaches INT_MAX", id_offset, (long long)I);
  return score_topk(ctx, q_bf16, U, c_bf16, I, dpad, k, id_offset, excl_indptr, excl_ids, out_vals, out_ids, workspace,
                    workspace_bytes, stream);
}

extern "C" int brk_mask_excluded(brk_ctx* ctx, float* scores, int64_t R, int64_t I, int32_t col_offset,
                                 const int64_t* excl_indptr, const int32_t* excl_ids, void* stream) {
  BRK_REQUIRE(ctx && scores && excl_indptr && excl_ids, BRK_E_ARG, "brk_mask_excluded: null argument");
  BRK_REQUIRE(R >= 0 && I > 0, BRK_E_ARG, "brk_mask_excluded: R=%lld I=%lld", (long long)R, (long long)I);
  if (R == 0) return 0;
  mask_excluded_kernel<<<unsigned((R * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(scores, R, I, col_offset,
                                                                                         excl_indptr, excl_ids);
  BRK_LAUNCH_CHECK();
  return 0;
}

extern "C" int brk_topk_merge(brk_ctx* ctx, const float* part_vals, const int32_t* part_ids, int32_t n_parts,
                              int64_t U, int32_t k, float* out_vals, int32_t* out_ids, void* stream) {
  BRK_REQUIRE(ctx && part_vals && part_ids && out_vals && out_ids, BRK_E_ARG, "brk_topk_merge: null argument");
  BRK_REQUIRE(n_parts >= 1 && n_parts <= 64 && U > 0 && k >= 1, BRK_E_ARG, "brk_topk_merge: n_parts=%d U=%lld k=%d",
              n_parts, (long long)U, k);
  topk_merge_kernel<<<unsigned((U + 255) / 256), 256, 0, (cudaStream_t)stream>>>(part_vals, part_ids, n_parts, U, k,
                                                                               out_vals, out_ids);
  BRK_LAUNCH_CHECK();
  return 0;
}

extern "C" int brk_topk_merge_peer(brk_ctx* ctx, const float* const* part_vals, const int32_t* const* part_ids,
                                   const int32_t* const* part_hdr, int32_t n_parts, int64_t U, int32_t k, float* out_vals,
                                   int32_t* out_ids, int32_t* err, void* stream) {
  BRK_REQUIRE(ctx && part_vals && part_ids && part_hdr && out_vals && out_ids && err, BRK_E_ARG,
              "brk_topk_merge_peer: null argument");
  BRK_REQUIRE(n_parts >= 1 && n_parts <= BRK_MAX_PEERS && k >= 1 && k <= kHeapCap && U >= 0 &&
                  (U + kMergeUsers - 1) / kMergeUsers <= INT_MAX,
              BRK_E_ARG, "brk_topk_merge_peer: n_parts=%d (1..%d) U=%lld k=%d (1..%d)", n_parts, BRK_MAX_PEERS,
              (long long)U, k, kHeapCap);
  if (U == 0) return 0;
  const size_t smem = size_t(n_parts) * kMergeUsers * k * 8;
  BRK_CUDA(cudaFuncSetAttribute(topk_merge_peer_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  topk_merge_peer_kernel<<<unsigned((U + kMergeUsers - 1) / kMergeUsers), kMergeUsers * 32, smem, (cudaStream_t)stream>>>(
      part_vals, part_ids, part_hdr, n_parts, U, k, out_vals, out_ids, err);
  BRK_LAUNCH_CHECK();
  return 0;
}

extern "C" int brk_topk_rows(brk_ctx* ctx, const float* scores, int64_t R, int64_t I, int32_t k, float* out_vals,
                             int32_t* out_ids, void* stream) {
  BRK_REQUIRE(ctx && scores && out_vals && out_ids, BRK_E_ARG, "brk_topk_rows: null argument");
  BRK_REQUIRE(R > 0 && I > 0 && I < (int64_t(1) << 31) && k >= 1 && k <= 32, BRK_E_ARG,
              "brk_topk_rows: R=%lld I=%lld k=%d", (long long)R, (long long)I, k);
  const unsigned grid = unsigned((R * 32 + 255) / 256);
  cudaStream_t st = (cudaStream_t)stream;
  if (k <= 10) topk_rows_kernel<10><<<grid, 256, 0, st>>>(scores, R, I, k, out_vals, out_ids);
  else if (k <= 16) topk_rows_kernel<16><<<grid, 256, 0, st>>>(scores, R, I, k, out_vals, out_ids);
  else topk_rows_kernel<32><<<grid, 256, 0, st>>>(scores, R, I, k, out_vals, out_ids);
  BRK_LAUNCH_CHECK();
  return 0;
}
