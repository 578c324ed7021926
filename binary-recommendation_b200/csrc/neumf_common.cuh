// Shared by the NeuMF kernels (neumf.cu, neumf2.cu, neumf_tc.cu, neumf_fused.cu, neumf_generic.cu): parameter
// layout, accumulator layout, sharded-table addressing, kernel arguments, activations, dropout bits.
#pragma once
#include "common.cuh"
#include <math_constants.h>

namespace v2 {

constexpr float kBnEps = 1e-3f, kBnMomentum = 0.99f;
constexpr uint32_t kDropThreshold = 51;
constexpr float kDropScale = 256.0f / 205.0f;

template <int E, int H1, int H2, int H3>
struct Layout {   // offsets (floats) inside the flat dense parameter block -- mirrored in hotpath.py
  static constexpr int W1 = 0, b1 = W1 + 2 * E * H1, g1 = b1 + H1, be1 = g1 + H1;
  static constexpr int W2 = be1 + H1, b2 = W2 + H1 * H2, g2 = b2 + H2, be2 = g2 + H2;
  static constexpr int W3 = be2 + H2, b3 = W3 + H2 * H3, W4 = b3 + H3;   // b4 = W4 + H3 + 1
};
// accumulator block (doubles): forward sums, backward sums, loss
template <int H1, int H2>
struct Acc {
  static constexpr int s1 = 0, q1 = s1 + H1, s2 = q1 + H1, q2 = s2 + H2;        // sum h, sum h^2
  static constexpr int d2 = q2 + H2, e2 = d2 + H2, d1 = e2 + H2, e1 = d1 + H1;  // sum dy, sum dy*xhat
  static constexpr int loss = e1 + H1, total = loss + 1;
};

// A table as the kernels address it: one shard per rank, row r on rank r % world at local row r / world
// (world == 1: the table itself).  Shard pointers of other ranks are NVLink peer mappings: rows are read
// with ordinary loads and gradients leave as REDs straight into the owner's accumulator -- the row
// "all-to-all" of a sharded lookup and of its gradient happen inside the gather / scatter instructions.
struct TabRef {
  const float* w[BRK_MAX_PEERS];
  float* g[BRK_MAX_PEERS];
  uint32_t* t[BRK_MAX_PEERS];
  int32_t world;
};
struct RowRef { const float* w; float* g; uint32_t* t; int64_t lrow; };
template <int E>
__device__ __forceinline__ RowRef locate(const TabRef& T, int64_t row) {
  int o = 0; int64_t l = row;
  if (T.world > 1) { o = int(row % T.world); l = row / T.world; }
  RowRef r; r.w = T.w[o] + l * E; r.g = T.g[o] ? T.g[o] + l * E : nullptr; r.t = T.t[o]; r.lrow = l;
  return r;
}
// Touched bit of a row: one fire-and-forget RED.OR.  (Round 1 peeked at the word first with a volatile load to skip
// redundant REDs; at configs[3] table sizes every peek is a dependent HBM round trip, volatile loads do not overlap, and
// tc_head issued 16 of them in a row per tile: ncu put most of that kernel's samples on the instruction consuming them.)
__device__ __forceinline__ void mark_row(const RowRef& r) {
  if (r.t) {
    const uint32_t bit = 1u << (r.lrow & 31);
    asm volatile("red.global.or.b32 [%0], %1;" ::"l"(r.t + (r.lrow >> 5)), "r"(bit) : "memory");
  }
}

struct Args {
  TabRef uMLP, iMLP, uMF, iMF;
  brk_table dense;
  const int32_t* u; const int32_t* i; const float* y;
  int64_t B, first_index, global_B;
  float *h1, *h2, *dy1, *dy2, *out;
  double* acc;
  float* bn_moving;
  float* loss_out;
  uint32_t drop_seed, drop_epoch;
  int32_t dropout, loss_kind, training;
};

template <int ACT> __device__ __forceinline__ float act_f(float x) {
  return ACT == 0 ? fmaxf(x, 0.f) : 1.0f / (1.0f + expf(-x));
}
template <int ACT> __device__ __forceinline__ float act_grad(float h) {
  return ACT == 0 ? (h > 0.f ? 1.f : 0.f) : h * (1.f - h);
}

// 16 dropout factors (features 16c .. 16c+15 of `layer`) of sample idx: keep iff its Philox byte >= 51
__device__ __forceinline__ void drop16(uint64_t idx, int c, int layer, uint32_t seed, uint32_t epoch, float (&m)[16]) {
  const uint4 w = philox4x32_10(make_uint4(uint32_t(idx), uint32_t(idx >> 32), uint32_t(c), 0xD0u + layer), seed, epoch);
  const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
  for (int q = 0; q < 4; ++q)
#pragma unroll
    for (int b = 0; b < 4; ++b) m[q * 4 + b] = ((ww[q] >> (8 * b)) & 0xFFu) >= kDropThreshold ? kDropScale : 0.f;
}
// the same 16 decisions as a bitmask (bit j set = feature 16c + j kept)
__device__ __forceinline__ uint32_t drop16_bits(uint64_t idx, int c, int layer, uint32_t seed, uint32_t epoch) {
  const uint4 w = philox4x32_10(make_uint4(uint32_t(idx), uint32_t(idx >> 32), uint32_t(c), 0xD0u + layer), seed, epoch);
  const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
  uint32_t bits = 0;
#pragma unroll
  for (int q = 0; q < 4; ++q)
#pragma unroll
    for (int b = 0; b < 4; ++b) bits |= (((ww[q] >> (8 * b)) & 0xFFu) >= kDropThreshold ? 1u : 0u) << (q * 4 + b);
  return bits;
}

}  // namespace v2
