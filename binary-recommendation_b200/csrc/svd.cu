// Biased-SVD SGD (SURVEY.md section 8 row f4): the reference's rating-by-rating pass
// (/root/reference/src/origin_models/svd/SVD.py:187-221) run on the device with EXACTLY the sequential
// semantics, in float64 like the NumPy original.
//
// The sequential pass only orders ratings that share a user or an item: rating k reads and writes row P[u_k],
// row Q[i_k], bu[u_k], bi[i_k] and nothing else.  brk_svd_schedule gives every rating two tickets,
//   tu[k] = number of earlier ratings of the same user,  ti[k] = number of earlier ratings of the same item,
// and every word of a parameter row carries the version of the row (self-validating rows, below).  A warp owns
// rating k, polls its user's and its item's rows until they carry versions tu[k] and ti[k] (every earlier rating
// touching either row has been applied), applies the update and writes the new rows with versions tu[k] + 1 and
// ti[k] + 1.  Ratings are dealt to the resident warps round-robin in file order, so the oldest unfinished rating is
// always held by a running warp whose tickets are already satisfied: no deadlock (the launch is cooperative, which
// guarantees co-residency), no global barrier, and the result equals the sequential pass up to the summation order
// inside the 'np.dot' (a 5-step butterfly over the lanes here; the element-wise updates are not contracted into FMAs,
// like NumPy).
//
// Bound: not HBM, not the tensor pipe -- the longest dependency chain (>= the rating count of the most popular
// item) times one L2 hand-over of a row between two SMs.  DESIGN.md section 4.5.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include "common.cuh"

namespace {

constexpr int kSvdThreads = 256;
constexpr int kSvdWarps = kSvdThreads / 32;

__device__ __forceinline__ uint32_t ld_relaxed_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_u32(uint32_t* p, uint32_t v) {
  asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ double warp_sum_f64(double x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x = __dadd_rn(x, __shfl_xor_sync(0xffffffffu, x, o));
  return x;
}

// w + lr * (e * other - reg * w), every operation rounded on its own (no FMA contraction), SVD.py:203-206.
__device__ __forceinline__ double svd_rule(double w, double other, double e, double lr, double reg) {
  return __dadd_rn(w, __dmul_rn(lr, __dsub_rn(__dmul_rn(e, other), __dmul_rn(reg, w))));
}

// Self-validating rows.  Every 8-byte word of a row carries its own version: a float64 element is two words
// {low half | version << 32} {high half | version << 32} written by one st.v2.b64 (two 8-byte accesses, each
// single-copy atomic).  The consumer polls the row itself and accepts a word when its version equals the ticket;
// version t of a row is written once (by the rating with ticket t - 1), read by exactly one warp (the rating with
// ticket t) and then overwritten by that same warp -- no fence, no separate flag, no reader that could see a torn row.
// A separate version counter per row costs, per hand-over of a row from one warp to the next, row stores -> fence ->
// flag store, then on the other side flag poll -> row loads (about 3.5 L2 round trips): it measured half the speed of
// this form (profiles/r01m_svd_sweep.txt).  Parameters are packed into this form at the start of the epoch and
// unpacked at its end (two streaming passes over the tables).
struct SvdLL {
  const int4* sched;          // [n] (user, item, user ticket, item ticket)
  const double* ratings;      // [n]
  int64_t n;
  ulonglong2 *P, *Q, *bu, *bi;
  uint32_t* abort;            // set when a wait exceeds kSvdSpinLimit polls (inconsistent schedule): every warp leaves
  double mu, lr, ereg, breg;
  int32_t d;
};
__device__ __forceinline__ ulonglong2 ld_ll(const ulonglong2* p) {
  ulonglong2 v;
  asm volatile("ld.relaxed.gpu.global.v2.b64 {%0,%1}, [%2];" : "=l"(v.x), "=l"(v.y) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ ulonglong2 ll_pack(double x, uint32_t ver) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(x), v = (unsigned long long)ver << 32;
  return make_ulonglong2(v | (b & 0xffffffffull), v | (b >> 32));
}
__device__ __forceinline__ void st_ll(ulonglong2* p, double x, uint32_t ver) {
  const ulonglong2 w = ll_pack(x, ver);
  asm volatile("st.relaxed.gpu.global.v2.b64 [%0], {%1,%2};" :: "l"(p), "l"(w.x), "l"(w.y) : "memory");
}
__device__ __forceinline__ bool ll_valid(const ulonglong2& v, uint32_t ver) {
  return uint32_t(v.x >> 32) == ver && uint32_t(v.y >> 32) == ver;
}
__device__ __forceinline__ double ll_value(const ulonglong2& v) {
  return __longlong_as_double((long long)((v.y << 32) | (v.x & 0xffffffffull)));
}

// A wait is bounded: a schedule that does not belong to the rating arrays would otherwise spin for ever.
constexpr uint32_t kSvdSpinLimit = 1u << 25;

// EPL = row elements per lane (d <= 32 * EPL).
template <int EPL>
__global__ void __launch_bounds__(kSvdThreads) svd_epoch_ll_kernel(SvdLL a) {
  const int lane = threadIdx.x & 31;
  const int64_t W = int64_t(gridDim.x) * kSvdWarps;
  int64_t k = int64_t(threadIdx.x >> 5) * gridDim.x + blockIdx.x;
  if (k >= a.n) return;
  int4 s = __ldg(a.sched + k);
  double r = __ldg(a.ratings + k);
  uint32_t live = 0;                                   // bit e: element lane + 32 e exists
#pragma unroll
  for (int e = 0; e < EPL; ++e) live |= (lane + 32 * e < a.d) ? (1u << e) : 0u;
  while (true) {
    const int64_t kn = k + W;
    int4 sn = s;
    double rn = r;
    if (kn < a.n) { sn = __ldg(a.sched + kn); rn = __ldg(a.ratings + kn); }

    const uint32_t tu = uint32_t(s.z), ti = uint32_t(s.w);
    ulonglong2* prow = a.P + int64_t(s.x) * a.d + lane;
    ulonglong2* qrow = a.Q + int64_t(s.y) * a.d + lane;
    ulonglong2* brow = lane == 0 ? a.bu + s.x : a.bi + s.y;       // lane 0: user bias, lane 1: item bias
    const uint32_t tb = lane == 0 ? tu : ti;
    ulonglong2 pv[EPL], qv[EPL], bv = make_ulonglong2(0, 0);
    uint32_t pend_p = live, pend_q = live;
    bool pend_b = lane < 2;
    uint32_t spins = 0;
    while (true) {
#pragma unroll
      for (int e = 0; e < EPL; ++e) {
        if (pend_p >> e & 1u) pv[e] = ld_ll(prow + 32 * e);
        if (pend_q >> e & 1u) qv[e] = ld_ll(qrow + 32 * e);
      }
      if (pend_b) bv = ld_ll(brow);
#pragma unroll
      for (int e = 0; e < EPL; ++e) {
        if ((pend_p >> e & 1u) && ll_valid(pv[e], tu)) pend_p &= ~(1u << e);
        if ((pend_q >> e & 1u) && ll_valid(qv[e], ti)) pend_q &= ~(1u << e);
      }
      if (pend_b && ll_valid(bv, tb)) pend_b = false;
      if (__all_sync(0xffffffffu, (pend_p | pend_q) == 0u && !pend_b)) break;
      if ((++spins & 1023u) == 0) {
        if (spins >= kSvdSpinLimit) st_relaxed_u32(a.abort, 1u);
        if (ld_relaxed_u32(a.abort) != 0u) return;
      }
    }
    double p[EPL], q[EPL];
    double dot = 0.0;
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
      p[e] = (live >> e & 1u) ? ll_value(pv[e]) : 0.0;
      q[e] = (live >> e & 1u) ? ll_value(qv[e]) : 0.0;
      dot = __dadd_rn(dot, __dmul_rn(q[e], p[e]));
    }
    dot = warp_sum_f64(dot);
    const double b_mine = ll_value(bv);
    const double b_u = __shfl_sync(0xffffffffu, b_mine, 0), b_i = __shfl_sync(0xffffffffu, b_mine, 1);
    const double err = __dsub_rn(r, __dadd_rn(__dadd_rn(__dadd_rn(b_u, b_i), a.mu), dot));
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
      if (live >> e & 1u) {
        const double qn = svd_rule(q[e], p[e], err, a.lr, a.ereg);
        const double pn = svd_rule(p[e], qn, err, a.lr, a.ereg);
        st_ll(qrow + 32 * e, qn, ti + 1u);
        st_ll(prow + 32 * e, pn, tu + 1u);
      }
    }
    if (lane < 2) st_ll(brow, svd_rule(b_mine, b_mine, err, a.lr, a.breg), tb + 1u);
    if (kn >= a.n) break;
    k = kn; s = sn; r = rn;
  }
}

// plain float64 tables <-> self-validating form (version 0), all four tables in one launch each way
struct SvdTables { double* plain[4]; ulonglong2* ll[4]; int64_t end[4]; };   // end: running element counts
__global__ void svd_pack_kernel(SvdTables t, int unpack) {
  for (int64_t x = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; x < t.end[3]; x += int64_t(gridDim.x) * blockDim.x) {
    const int a = x < t.end[0] ? 0 : x < t.end[1] ? 1 : x < t.end[2] ? 2 : 3;
    const int64_t j = x - (a ? t.end[a - 1] : 0);
    if (unpack) t.plain[a][j] = ll_value(t.ll[a][j]);
    else t.ll[a][j] = ll_pack(t.plain[a][j], 0u);
  }
}

// ---- schedule ---------------------------------------------------------------------------------------------
__global__ void svd_hist_kernel(const int32_t* __restrict__ keys, int64_t n, int32_t rows, uint32_t* cnt,
                                int32_t* iota, int32_t* bad) {
  for (int64_t k = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; k < n; k += int64_t(gridDim.x) * blockDim.x) {
    const int32_t key = keys[k];
    if (iota) iota[k] = int32_t(k);
    if (key < 0 || key >= rows) { atomicExch(bad, 1); continue; }
    atomicAdd(cnt + key, 1u);
  }
}
// after the stable sort by key: position s holds rating idx[s]; its ticket is s - start[key]
__global__ void svd_ticket_kernel(const int32_t* __restrict__ sorted_keys, const int32_t* __restrict__ idx,
                                  const uint32_t* __restrict__ start, int64_t n, int32_t rows, int32_t* sched,
                                  int field) {
  for (int64_t s = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; s < n; s += int64_t(gridDim.x) * blockDim.x) {
    const int32_t key = sorted_keys[s];
    const int64_t k = idx[s];
    if (key < 0 || key >= rows) continue;                          // reported through bad_id by the histogram pass
    sched[4 * k + field] = key;
    sched[4 * k + 2 + field] = int32_t(uint32_t(s) - start[key]);
  }
}

// ---- predict / errors / mean --------------------------------------------------------------------------------
// One lane group of 8 per rating; prediction = bu + bi + mu + <q, p> (SVD.py:179-185).
__device__ __forceinline__ double svd_predict_one(const double* __restrict__ P, const double* __restrict__ Q,
                                                  const double* __restrict__ bu, const double* __restrict__ bi,
                                                  int32_t u, int32_t i, int32_t d, double mu, int sub) {
  const double* p = P + int64_t(u) * d;
  const double* q = Q + int64_t(i) * d;
  double dot = 0.0;
  for (int c = sub; c < d; c += 8) dot = __dadd_rn(dot, __dmul_rn(q[c], p[c]));
#pragma unroll
  for (int o = 4; o > 0; o >>= 1) dot = __dadd_rn(dot, __shfl_xor_sync(0xffffffffu, dot, o));
  return __dadd_rn(__dadd_rn(__dadd_rn(bu[u], bi[i]), mu), dot);
}

__global__ void svd_predict_kernel(const int32_t* __restrict__ users, const int32_t* __restrict__ items, int64_t n,
                                   const double* P, const double* Q, const double* bu, const double* bi, int32_t d,
                                   double mu, double* out) {
  const int sub = threadIdx.x & 7;
  const int64_t groups = (int64_t(gridDim.x) * blockDim.x) >> 3;
  const int64_t n_pad = (n + 3) & ~int64_t(3);                      // whole warps stay converged for the shuffles
  for (int64_t k = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 3; k < n_pad; k += groups) {
    const bool live = k < n;
    const double y = svd_predict_one(P, Q, bu, bi, live ? users[k] : 0, live ? items[k] : 0, d, mu, sub);
    if (live && sub == 0) out[k] = y;
  }
}

// mode 0: partial sums of (e^2, |e|) with e = rating - prediction; mode 1: partial sums of (x, 0) (the global mean).
// Partials are combined in a fixed order by svd_finish_kernel: the result does not depend on the launch.
__global__ void __launch_bounds__(256) svd_partial_kernel(const int32_t* __restrict__ users,
                                                          const int32_t* __restrict__ items,
                                                          const double* __restrict__ x, int64_t n, const double* P,
                                                          const double* Q, const double* bu, const double* bi, int32_t d,
                                                          double mu, int mode, double* partial) {
  __shared__ double sm[64];
  double s0 = 0.0, s1 = 0.0;
  if (mode == 0) {
    const int sub = threadIdx.x & 7;
    const int64_t groups = (int64_t(gridDim.x) * blockDim.x) >> 3;
    const int64_t n_pad = (n + 3) & ~int64_t(3);
    for (int64_t k = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 3; k < n_pad; k += groups) {
      const bool live = k < n;
      const double y = svd_predict_one(P, Q, bu, bi, live ? users[k] : 0, live ? items[k] : 0, d, mu, sub);
      if (live && sub == 0) { const double e = x[k] - y; s0 += e * e; s1 += fabs(e); }
    }
  } else {
    for (int64_t k = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; k < n; k += int64_t(gridDim.x) * blockDim.x) s0 += x[k];
  }
  s0 = block_sum_double(s0, sm);
  __syncthreads();
  s1 = block_sum_double(s1, sm + 32);
  if (threadIdx.x == 0) { partial[2 * blockIdx.x] = s0; partial[2 * blockIdx.x + 1] = s1; }
}
__global__ void svd_finish_kernel(const double* partial, int blocks, int64_t n, double* out) {
  __shared__ double sm[64];
  double s0 = 0.0, s1 = 0.0;
  for (int b = threadIdx.x; b < blocks; b += blockDim.x) { s0 += partial[2 * b]; s1 += partial[2 * b + 1]; }
  s0 = block_sum_double(s0, sm);
  __syncthreads();
  s1 = block_sum_double(s1, sm + 32);
  if (threadIdx.x == 0) { out[0] = s0 / double(n); out[1] = s1 / double(n); }
}

// ---- get_rating without a rating column (SVD.py:255-270) -------------------------------------------------------
struct SvdQuintiles { double tc[3], qs[3], tc_scale, qs_scale; };
__device__ __forceinline__ double svd_quintile(double v, const double* q) {
  return v > q[2] ? 4.0 : v > q[1] ? 3.0 : v > q[0] ? 2.0 : 1.0;
}
__global__ void svd_quintile_kernel(const double* __restrict__ tc, const double* __restrict__ qs, int64_t n,
                                    SvdQuintiles h, double* out) {
  for (int64_t k = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; k < n; k += int64_t(gridDim.x) * blockDim.x)
    out[k] = h.tc_scale * svd_quintile(tc[k], h.tc) + h.qs_scale * svd_quintile(qs[k], h.qs);
}

// ---- recommend (SVD.py:286-299): the k best items of a user by plain <p_u, q_i> in float64 ----------------------
// scores[j, i] = <P[users[j]], Q[i]>, one warp per (user, item).
__global__ void svd_scores_kernel(const double* __restrict__ P, const int32_t* __restrict__ users, int32_t nu,
                                  const double* __restrict__ Q, int64_t I, int32_t d, double* scores) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t(gridDim.x) * blockDim.x) >> 5;
  for (int64_t w = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5; w < int64_t(nu) * I; w += warps) {
    const int64_t j = w / I, i = w - j * I;
    const double* p = P + int64_t(users[j]) * d;
    const double* q = Q + i * d;
    double dot = 0.0;
    for (int c = lane; c < d; c += 32) dot = __dadd_rn(dot, __dmul_rn(p[c], q[c]));
    dot = warp_sum_f64(dot);
    if (lane == 0) scores[w] = dot;
  }
}
// One CTA per user: k rounds of "best remaining" = (score desc, index asc), the rule of the reference's strict '>'
// replacement (an equal later score never displaces an earlier one).  NaN scores are never selected.
__global__ void __launch_bounds__(256) svd_select_kernel(const double* __restrict__ scores, int64_t I, int32_t k,
                                                         double* out_vals, int32_t* out_ids) {
  __shared__ double sv[8];
  __shared__ int64_t si[8];
  __shared__ double last_v;
  __shared__ int64_t last_i;
  const double* s = scores + int64_t(blockIdx.x) * I;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int r = 0; r < k; ++r) {
    double bv = -INFINITY; int64_t bi = -1;
    const double lv = r ? last_v : INFINITY;
    const int64_t li = r ? last_i : -1;
    for (int64_t i = threadIdx.x; i < I && !(r && li < 0); i += blockDim.x) {   // li < 0: nothing left to pick
      const double v = s[i];
      const bool after_last = v < lv || (v == lv && i > li);     // strictly behind the previous pick
      if (after_last && (bi < 0 || v > bv)) { bv = v; bi = i; }  // ascending i per thread: ties keep the lower index
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int64_t oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
    }
    if (lane == 0) { sv[w] = bv; si[w] = bi; }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int j = 1; j < 8; ++j)
        if (si[j] >= 0 && (si[0] < 0 || sv[j] > sv[0] || (sv[j] == sv[0] && si[j] < si[0]))) { sv[0] = sv[j]; si[0] = si[j]; }
      last_v = sv[0]; last_i = si[0];
      out_vals[int64_t(blockIdx.x) * k + r] = si[0] >= 0 ? sv[0] : -INFINITY;
      out_ids[int64_t(blockIdx.x) * k + r] = int32_t(si[0]);
    }
    __syncthreads();
  }
}

inline int grid_for(int64_t work_threads, int sm_count, int threads) {
  int64_t g = (work_threads + threads - 1) / threads;
  const int64_t cap = int64_t(sm_count) * 8;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return int(g);
}
inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

struct SchedLayout { size_t cnt, flag, iota, keys_out, idx_out, cub, total; size_t cub_bytes; };
SchedLayout sched_layout(int64_t n, int64_t rows_max) {
  SchedLayout L;
  size_t sort_bytes = 0, scan_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const int32_t*)nullptr, (int32_t*)nullptr,
                                  (const int32_t*)nullptr, (int32_t*)nullptr, int(n), 0, 32);
  cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (uint32_t*)nullptr, (uint32_t*)nullptr, int(rows_max));
  L.cub_bytes = sort_bytes > scan_bytes ? sort_bytes : scan_bytes;
  size_t off = 0;
  L.cnt = off;      off += align256(size_t(rows_max) * 4);
  L.flag = off;     off += 256;
  L.iota = off;     off += align256(size_t(n) * 4);
  L.keys_out = off; off += align256(size_t(n) * 4);
  L.idx_out = off;  off += align256(size_t(n) * 4);
  L.cub = off;      off += align256(L.cub_bytes);
  L.total = off;
  return L;
}

}  // namespace

extern "C" int64_t brk_svd_schedule_workspace_bytes(int64_t n, int64_t num_users, int64_t num_items) {
  if (n < 0 || num_users < 1 || num_items < 1 || n >= (int64_t(1) << 31)) return BRK_E_ARG;
  return int64_t(sched_layout(n > 0 ? n : 1, num_users > num_items ? num_users : num_items).total);
}

extern "C" int brk_svd_schedule(brk_ctx* ctx, const int32_t* users, const int32_t* items, int64_t n,
                                int64_t num_users, int64_t num_items, int32_t* sched, int32_t* bad_id,
                                void* workspace, int64_t workspace_bytes, void* stream) {
  BRK_REQUIRE(ctx && sched && workspace && bad_id, BRK_E_ARG, "brk_svd_schedule: null argument");
  BRK_REQUIRE(n >= 0 && n < (int64_t(1) << 31) && num_users >= 1 && num_items >= 1 &&
              num_users < (int64_t(1) << 31) && num_items < (int64_t(1) << 31), BRK_E_ARG,
              "brk_svd_schedule: n=%lld users=%lld items=%lld", (long long)n, (long long)num_users, (long long)num_items);
  BRK_REQUIRE(brk_aligned16(sched) && brk_aligned16(workspace), BRK_E_ALIGN, "brk_svd_schedule: sched / workspace not 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  BRK_CUDA(cudaMemsetAsync(bad_id, 0, sizeof(int32_t), st));
  if (n == 0) return 0;
  BRK_REQUIRE(users && items, BRK_E_ARG, "brk_svd_schedule: null id arrays");
  const SchedLayout L = sched_layout(n, num_users > num_items ? num_users : num_items);
  BRK_REQUIRE(workspace_bytes >= int64_t(L.total), BRK_E_ARG, "brk_svd_schedule: workspace %lld < %lld bytes",
              (long long)workspace_bytes, (long long)L.total);
  char* ws = reinterpret_cast<char*>(workspace);
  uint32_t* cnt = reinterpret_cast<uint32_t*>(ws + L.cnt);
  int32_t* iota = reinterpret_cast<int32_t*>(ws + L.iota);
  int32_t* keys_out = reinterpret_cast<int32_t*>(ws + L.keys_out);
  int32_t* idx_out = reinterpret_cast<int32_t*>(ws + L.idx_out);
  const int grid = grid_for(n, ctx->sm_count, 256);
  for (int field = 0; field < 2; ++field) {
    const int32_t* keys = field == 0 ? users : items;
    const int64_t rows = field == 0 ? num_users : num_items;
    int bits = 1;
    while ((int64_t(1) << bits) < rows) ++bits;
    BRK_CUDA(cudaMemsetAsync(cnt, 0, size_t(rows) * 4, st));
    svd_hist_kernel<<<grid, 256, 0, st>>>(keys, n, int32_t(rows), cnt, field == 0 ? iota : nullptr, bad_id);
    BRK_LAUNCH_CHECK();
    size_t cb = L.cub_bytes;
    BRK_CUDA(cub::DeviceScan::ExclusiveSum(ws + L.cub, cb, cnt, cnt, int(rows), st));
    cb = L.cub_bytes;
    // out-of-range keys (reported through bad_id) are masked to the sorted bits and land in some bucket: harmless,
    // the caller must not use a schedule whose bad_id flag is set
    BRK_CUDA(cub::DeviceRadixSort::SortPairs(ws + L.cub, cb, keys, keys_out, iota, idx_out, int(n), 0, bits, st));
    svd_ticket_kernel<<<grid, 256, 0, st>>>(keys_out, idx_out, cnt, n, int32_t(rows), sched, field);
    BRK_LAUNCH_CHECK();
  }
  return 0;
}

template <int EPL>
static int svd_launch_epoch(brk_ctx* ctx, SvdLL& a, int warps_per_sm, cudaStream_t st) {
  int occ = 0;
  BRK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, svd_epoch_ll_kernel<EPL>, kSvdThreads, 0));
  BRK_REQUIRE(occ >= 1, BRK_E_STATE, "brk_svd_fit_epoch: kernel does not fit an SM");
  int per_sm = occ;
  if (warps_per_sm > 0) {
    per_sm = (warps_per_sm + kSvdWarps - 1) / kSvdWarps;
    if (per_sm > occ) per_sm = occ;
  }
  int64_t grid = int64_t(ctx->sm_count) * per_sm;
  const int64_t need = (a.n + kSvdWarps - 1) / kSvdWarps;
  if (grid > need) grid = need;
  void* args[] = {&a};
  BRK_CUDA(cudaLaunchCooperativeKernel((const void*)svd_epoch_ll_kernel<EPL>, dim3((unsigned)grid), dim3(kSvdThreads),
                                       args, 0, st));
  return 0;
}

// workspace: [abort flag, 256 B] [P, Q, bu, bi in self-validating form, 16 B per element]
static int64_t svd_fit_ws_bytes(int64_t U, int64_t I, int64_t d) {
  return 256 + int64_t(align256(size_t((U + I) * (d + 1)) * 16));
}
extern "C" int64_t brk_svd_fit_workspace_bytes(int64_t num_users, int64_t num_items, int32_t d) {
  if (num_users < 1 || num_items < 1 || d < 1 || d > 512) return BRK_E_ARG;
  return svd_fit_ws_bytes(num_users, num_items, d);
}

extern "C" int brk_svd_fit_epoch(brk_ctx* ctx, const int32_t* sched, const double* ratings, int64_t n, double* P,
                                 double* Q, double* bu, double* bi, int64_t num_users, int64_t num_items, int32_t d,
                                 double mu, double lr, double emb_reg, double bias_reg, void* workspace,
                                 int64_t workspace_bytes, int32_t warps_per_sm, void* stream) {
  BRK_REQUIRE(ctx && P && Q && bu && bi && workspace, BRK_E_ARG, "brk_svd_fit_epoch: null argument");
  BRK_REQUIRE(n >= 0 && num_users >= 1 && num_items >= 1 && d >= 1 && d <= 512, BRK_E_ARG,
              "brk_svd_fit_epoch: n=%lld d=%d (1..512)", (long long)n, d);
  BRK_REQUIRE(brk_aligned16(workspace) && workspace_bytes >= svd_fit_ws_bytes(num_users, num_items, d), BRK_E_ARG,
              "brk_svd_fit_epoch: workspace %lld < %lld bytes or not 16-byte aligned", (long long)workspace_bytes,
              (long long)svd_fit_ws_bytes(num_users, num_items, d));
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = reinterpret_cast<char*>(workspace);
  BRK_CUDA(cudaMemsetAsync(ws, 0, 256, st));
  if (n == 0) return 0;
  BRK_REQUIRE(sched && ratings, BRK_E_ARG, "brk_svd_fit_epoch: null schedule / ratings");
  BRK_REQUIRE(brk_aligned16(sched), BRK_E_ALIGN, "brk_svd_fit_epoch: sched not 16-byte aligned");
  SvdLL a;
  a.sched = reinterpret_cast<const int4*>(sched); a.ratings = ratings; a.n = n;
  a.P = reinterpret_cast<ulonglong2*>(ws + 256); a.Q = a.P + num_users * int64_t(d); a.bu = a.Q + num_items * int64_t(d);
  a.bi = a.bu + num_users;
  a.abort = reinterpret_cast<uint32_t*>(ws); a.mu = mu; a.lr = lr; a.ereg = emb_reg; a.breg = bias_reg; a.d = d;
  SvdTables t;
  t.plain[0] = P; t.plain[1] = Q; t.plain[2] = bu; t.plain[3] = bi;
  t.ll[0] = a.P; t.ll[1] = a.Q; t.ll[2] = a.bu; t.ll[3] = a.bi;
  t.end[0] = num_users * int64_t(d); t.end[1] = t.end[0] + num_items * int64_t(d);
  t.end[2] = t.end[1] + num_users; t.end[3] = t.end[2] + num_items;
  const int pack_grid = grid_for(t.end[3], ctx->sm_count, 256);
  svd_pack_kernel<<<pack_grid, 256, 0, st>>>(t, 0);
  BRK_LAUNCH_CHECK();
  int rc;
  if (d <= 32) rc = svd_launch_epoch<1>(ctx, a, warps_per_sm, st);
  else if (d <= 64) rc = svd_launch_epoch<2>(ctx, a, warps_per_sm, st);
  else if (d <= 128) rc = svd_launch_epoch<4>(ctx, a, warps_per_sm, st);
  else if (d <= 256) rc = svd_launch_epoch<8>(ctx, a, warps_per_sm, st);
  else rc = svd_launch_epoch<16>(ctx, a, warps_per_sm, st);
  if (rc) return rc;
  svd_pack_kernel<<<pack_grid, 256, 0, st>>>(t, 1);
  BRK_LAUNCH_CHECK();
  return 0;
}

extern "C" int brk_svd_predict(brk_ctx* ctx, const int32_t* users, const int32_t* items, int64_t n, const double* P,
                               const double* Q, const double* bu, const double* bi, int32_t d, double mu, double* out,
                               void* stream) {
  BRK_REQUIRE(ctx && P && Q && bu && bi, BRK_E_ARG, "brk_svd_predict: null argument");
  BRK_REQUIRE(n >= 0 && d >= 1, BRK_E_ARG, "brk_svd_predict: n=%lld d=%d", (long long)n, d);
  if (n == 0) return 0;
  BRK_REQUIRE(users && items && out, BRK_E_ARG, "brk_svd_predict: null ids / out");
  svd_predict_kernel<<<grid_for(n * 8, ctx->sm_count, 256), 256, 0, (cudaStream_t)stream>>>(users, items, n, P, Q, bu, bi, d, mu, out);
  BRK_LAUNCH_CHECK();
  return 0;
}

extern "C" int64_t brk_svd_reduce_workspace_bytes(const brk_ctx* ctx) {
  return ctx ? int64_t(ctx->sm_count) * 8 * 2 * int64_t(sizeof(double)) : int64_t(BRK_E_ARG);
}

extern "C" int brk_svd_errors(brk_ctx* ctx, const int32_t* users, const int32_t* items, const double* ratings,
                              int64_t n, const double* P, const double* Q, const double* bu, const double* bi,
                              int32_t d, double mu, double* out_mse_mae, void* workspace, void* stream) {
  BRK_REQUIRE(ctx && users && items && ratings && P && Q && bu && bi && out_mse_mae && workspace, BRK_E_ARG,
              "brk_svd_errors: null argument");
  BRK_REQUIRE(n >= 1 && d >= 1, BRK_E_ARG, "brk_svd_errors: n=%lld d=%d (the reference divides by the count: n >= 1)", (long long)n, d);
  const int grid = grid_for(n * 8, ctx->sm_count, 256);
  cudaStream_t st = (cudaStream_t)stream;
  svd_partial_kernel<<<grid, 256, 0, st>>>(users, items, ratings, n, P, Q, bu, bi, d, mu, 0, reinterpret_cast<double*>(workspace));
  BRK_LAUNCH_CHECK();
  svd_finish_kernel<<<1, 256, 0, st>>>(reinterpret_cast<const double*>(workspace), grid, n, out_mse_mae);
  BRK_LAUNCH_CHECK();
  return 0;
}

extern "C" int brk_svd_mean(brk_ctx* ctx, const double* x, int64_t n, double* out2, void* workspace, void* stream) {
  BRK_REQUIRE(ctx && x && out2 && workspace, BRK_E_ARG, "brk_svd_mean: null argument");
  BRK_REQUIRE(n >= 1, BRK_E_ARG, "brk_svd_mean: n=%lld", (long long)n);
  const int grid = grid_for(n, ctx->sm_count, 256);
  cudaStream_t st = (cudaStream_t)stream;
  svd_partial_kernel<<<grid, 256, 0, st>>>(nullptr, nullptr, x, n, nullptr, nullptr, nullptr, nullptr, 0, 0.0, 1, reinterpret_cast<double*>(workspace));
  BRK_LAUNCH_CHECK();
  svd_finish_kernel<<<1, 256, 0, st>>>(reinterpret_cast<const double*>(workspace), grid, n, out2);
  BRK_LAUNCH_CHECK();
  return 0;
}

extern "C" int brk_svd_quintile_ratings(brk_ctx* ctx, const double* transaction_count, const double* quantity_sum,
                                        int64_t n, double tc_scale, double qs_scale, const double* tc_quintiles_host,
                                        const double* qs_quintiles_host, double* out, void* stream) {
  BRK_REQUIRE(ctx && tc_quintiles_host && qs_quintiles_host, BRK_E_ARG, "brk_svd_quintile_ratings: null argument");
  BRK_REQUIRE(n >= 0, BRK_E_ARG, "brk_svd_quintile_ratings: n=%lld", (long long)n);
  if (n == 0) return 0;
  BRK_REQUIRE(transaction_count && quantity_sum && out, BRK_E_ARG, "brk_svd_quintile_ratings: null column");
  SvdQuintiles h;
  for (int j = 0; j < 3; ++j) { h.tc[j] = tc_quintiles_host[j]; h.qs[j] = qs_quintiles_host[j]; }
  h.tc_scale = tc_scale; h.qs_scale = qs_scale;
  svd_quintile_kernel<<<grid_for(n, ctx->sm_count, 256), 256, 0, (cudaStream_t)stream>>>(transaction_count, quantity_sum, n, h, out);
  BRK_LAUNCH_CHECK();
  return 0;
}

extern "C" int brk_svd_recommend(brk_ctx* ctx, const double* P, const int32_t* users, int32_t n_users, const double* Q,
                                 int64_t num_items, int32_t d, int32_t k, double* scores, double* out_vals,
                                 int32_t* out_ids, void* stream) {
  BRK_REQUIRE(ctx && P && Q, BRK_E_ARG, "brk_svd_recommend: null argument");
  BRK_REQUIRE(n_users >= 0 && num_items >= 1 && num_items < (int64_t(1) << 31) && d >= 1 && k >= 1, BRK_E_ARG,
              "brk_svd_recommend: users=%d items=%lld d=%d k=%d", n_users, (long long)num_items, d, k);
  if (n_users == 0) return 0;
  BRK_REQUIRE(users && scores && out_vals && out_ids, BRK_E_ARG, "brk_svd_recommend: null ids / outputs");
  cudaStream_t st = (cudaStream_t)stream;
  svd_scores_kernel<<<grid_for(int64_t(n_users) * num_items * 32, ctx->sm_count, 256), 256, 0, st>>>(P, users, n_users, Q, num_items, d, scores);
  BRK_LAUNCH_CHECK();
  svd_select_kernel<<<n_users, 256, 0, st>>>(scores, num_items, k, out_vals, out_ids);
  BRK_LAUNCH_CHECK();
  return 0;
}
