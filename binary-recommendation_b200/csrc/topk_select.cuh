// Per-thread running top-K list of the fused selection epilogues (topk.cu score_topk_kernel / topk_rows_kernel,
// neumf_topk.cu): vals sorted descending, ids beside them.
#pragma once
#include <stdint.h>

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
