// Per-thread running top-K list of the fused selection epilogues (topk.cu score_topk_kernel / topk_rows_kernel,
// neumf_topk.cu): vals sorted descending, ids beside them.
#pragma once
#include <stdint.h>
#include <math_constants.h>

template <int K>
__device__ __forceinline__ void topk_insert(float (&vals)[K], int32_t (&ids)[K], float v, int32_t id) {
  // precondition: v > vals[K-1].  vals sorted descending; strict '>' keeps earlier (lower id) on ties.
#pragma unroll
  for (int j = K - 1; j > 0; --j) {
    const bool up = v > vals[j - 1];
    const bool here = v > vals[j];
    ids[j] = up ? ids[j - 1] : (here ? id : ids[j]);
    vals[j] = up ? vals[j - 1] : fmaxf(v, vals[j]);
  }
  if (v > vals[0]) { vals[0] = v; ids[0] = id; }
}

// Lists too long for registers (topk.cu, k > 32): one row's list as a bounded min-heap of n entries in shared memory.
// Entry j of the row sits at h[j * stride]; with one row per thread and stride = the block's row count, lane i of a
// warp always reads bank i (8-byte entries: one wavefront per half-warp), whatever heap index each lane is at.  Key
// order: score ascending, then id descending, so the root is the row's worst entry and its score is the insertion
// threshold.  Candidates that arrive in ascending id and are inserted only when they beat the root's score (strict
// '>') give the tie rule of topk_insert: equal scores keep the lower id.  O(log n) shared-memory steps per insertion
// against O(K) register moves for topk_insert.
struct __align__(8) TopkEntry {
  float v;
  int32_t id;
};

__device__ __forceinline__ bool topk_worse(TopkEntry a, TopkEntry b) { return a.v < b.v || (a.v == b.v && a.id > b.id); }

// n sentinels (-inf, -1): a row with fewer than n candidates comes out padded with them
__device__ __forceinline__ void topk_heap_init(TopkEntry* h, int stride, int n) {
#pragma unroll 1
  for (int j = 0; j < n; ++j) h[j * stride] = TopkEntry{-CUDART_INF_F, -1};
}

// Puts x in the root's place of an n-entry heap and sifts it down; returns the new root's score.  As an insertion, x
// must beat the root.
__device__ __forceinline__ float topk_heap_replace_root(TopkEntry* h, int stride, int n, TopkEntry x) {
  int i = 0;
#pragma unroll 1
  for (int c = 1; c < n; c = 2 * i + 1) {
    TopkEntry e = h[c * stride];
    if (c + 1 < n) {
      const TopkEntry f = h[(c + 1) * stride];
      if (topk_worse(f, e)) { e = f; ++c; }
    }
    if (!topk_worse(e, x)) break;                      // x is no better than its worse child: it stays at i
    h[i * stride] = e;
    i = c;
  }
  h[i * stride] = x;
  return h[0].v;
}

// Sorts the heap in place into h[0 .. n): score descending, ties -> lower id (the order of topk_insert's lists)
__device__ __forceinline__ void topk_heap_sort(TopkEntry* h, int stride, int n) {
#pragma unroll 1
  for (int end = n - 1; end > 0; --end) {
    const TopkEntry last = h[end * stride];
    h[end * stride] = h[0];                            // the worst of h[0 .. end] goes behind them
    topk_heap_replace_root(h, stride, end, last);
  }
}
