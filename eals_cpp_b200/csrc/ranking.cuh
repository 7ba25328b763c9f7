// ranking.cuh — ranking metrics on a held-out test matrix, device part (host side: retrieval.cuh, DESIGN.md §3.7).
//
// For a test entry (u, g) the rank is g's position in recommend([u], k, exclude_seen) (recommend.cuh), or -1:
//
//     rank(u, g) = #{ eligible i != g : s_i > s_g, or s_i == s_g and i < g }   if that count is < k, else -1
//
// with s_i = predict(u, i) (seq_dot, bit for bit) and, with exclude_seen, the items of u's train row not eligible
// (a test item that is also in the train row is -1).  One filter slot per test entry: its row is U[u], its
// threshold the exact s_g.  The kernels here are the pieces around the tcgen05 filter of eval_tc.cuh:
//   rm_entry_kernel        test entry -> (user, item)
//   rm_train_score_kernel  the exact score of every train nonzero of the users that have test entries, once
//   rm_train_count_kernel  c_R = train items ahead of g (they are ahead in the full order but not in the list), the
//                          "g is in the train row" verdict, and the per-slot limit k + c_R of the certain count
//                          (the working set keeps a slot while its certain count is below it: below_limit_flags_kernel)
//   rm_rescore_kernel      exact tie-aware count over the MODE 2 candidates of the survivors
//   rm_rank_kernel         rank = exact count - c_R, or -1
//   rm_lookup_kernel       exact engine: positions of the test items in recommend's exact lists
//   rm_metrics_kernel      per user: hit rate, precision, recall, NDCG, MAP and MRR at k
#pragma once

#include "common.cuh"
#include "eval.cuh"
#include "eval_tc.cuh"
#include "recommend.cuh"

namespace eals {
namespace rk {

constexpr int kMetrics = 6;   // hit rate, precision, recall, NDCG, MAP, MRR

// the row r in [lo, hi) with ptr[r] <= e < ptr[r + 1] (ptr ascending, e inside the rows' range)
__device__ __forceinline__ int row_of(const int64_t* __restrict__ ptr, int lo, int hi, int64_t e) {
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (ptr[mid] <= e) lo = mid; else hi = mid;
  }
  return lo;
}

// Entries e0 .. e0 + n of the owned test rows [r0, r1) (tptr / tidx: the validated test CSR, row 0 = user ub):
// user[s] = global user id, item[s] = test item of entry e0 + s.
__global__ void rm_entry_kernel(const int64_t* __restrict__ tptr, const int32_t* __restrict__ tidx, int r0, int r1, int ub,
                                int64_t e0, int n, int32_t* __restrict__ user, int32_t* __restrict__ item) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  const int64_t e = e0 + s;
  user[s] = ub + row_of(tptr, r0, r1, e);
  item[s] = tidx[e];
}

// score[t] = seq_dot(U[u], V[ridx[z0 + t]]) for the train nonzeros z0 .. z0 + nz of the owned rows [r0, r1), u the
// nonzero's user; nonzeros of users without test entries are skipped.  128 threads per block, whole warps.
__global__ void __launch_bounds__(128)
rm_train_score_kernel(const double* __restrict__ U, const double* __restrict__ V, int K, int LD, const int64_t* __restrict__ rptr,
                      const int32_t* __restrict__ ridx, const int64_t* __restrict__ tptr, int r0, int r1, int ub, int64_t z0,
                      long long nz, double* __restrict__ score) {
  __shared__ double sm[4][2 * 32 * 17];
  const long long n_round = (nz + 31) & ~31ll;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n_round; t += (long long)gridDim.x * blockDim.x) {
    const double *a = nullptr, *b = nullptr;
    if (t < nz) {
      const int64_t z = z0 + t;
      const int r = row_of(rptr, r0, r1, z);
      if (tptr[r + 1] > tptr[r]) {
        a = U + (size_t)(ub + r) * LD;
        b = V + (size_t)ridx[z] * LD;
      }
    }
    const double acc = seq_dot_warp32(a, b, K, sm[threadIdx.x >> 5]);
    if (a) score[t] = acc;
  }
}

// One warp per slot s (test entry of user[s], item[s], exact score gts[s]).  rptr == nullptr (no exclusion): c_r = 0,
// lim = k.  Otherwise the walk over the user's train row (scores from rm_train_score_kernel, score[z - z0]):
// c_r[s] = train items ahead of g under the list's order, and lim[s] = k + c_r[s], or 0 when g itself is in the
// train row (rank -1, the slot never enters the filter).  A slot whose certain count reaches k + c_R has at least k
// eligible items ahead of it (at most c_R of the certainly larger ones are train items).
__global__ void rm_train_count_kernel(const int64_t* __restrict__ rptr, const int32_t* __restrict__ ridx, const double* __restrict__ score,
                                      int64_t z0, int ub, const int32_t* __restrict__ user, const int32_t* __restrict__ item,
                                      const double* __restrict__ gts, int n, int k, int32_t* __restrict__ c_r, int32_t* __restrict__ lim) {
  const int s = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (s >= n) return;
  int cnt = 0;
  bool seen = false;
  if (rptr) {
    const int r = user[s] - ub;
    const int32_t g = item[s];
    const double sg = gts[s];
    for (int64_t z = rptr[r] + lane; z < rptr[r + 1]; z += 32) {
      const int32_t i = ridx[z];
      seen |= i == g;
      cnt += rec::better(score[z - z0], i, sg, g) ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(kFullMask, cnt, o);
    seen = __any_sync(kFullMask, seen);
  }
  if (lane == 0) {
    c_r[s] = cnt;
    lim[s] = seen ? 0 : k + cnt;
  }
}

// One thread per candidate pair of the MODE 2 emission (every item with acc >= g^ - E, so every item that is not
// certainly below s_g): its exact score, and cnt_exact[slot] += 1 when the item is ahead of g (score larger, or equal
// with a smaller id).
__global__ void __launch_bounds__(128)
rm_rescore_kernel(const double* __restrict__ U, const double* __restrict__ V, int K, int LD, const int32_t* __restrict__ user,
                  const int32_t* __restrict__ item, const double* __restrict__ gts, const tc::EvalPair* __restrict__ pairs,
                  unsigned long long n, int32_t* __restrict__ cnt_exact) {
  __shared__ double sm[4][2 * 32 * 17];
  const unsigned long long n_round = (n + 31ull) & ~31ull;
  for (unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; t < n_round; t += (unsigned long long)gridDim.x * blockDim.x) {
    const bool live = t < n;
    tc::EvalPair pr{0, 0, 0, 0};
    const double *a = nullptr, *b = nullptr;
    if (live) {
      pr = pairs[t];
      a = U + (size_t)user[pr.slot] * LD;
      b = V + (size_t)pr.item * LD;
    }
    const double acc = seq_dot_warp32(a, b, K, sm[threadIdx.x >> 5]);
    if (live && rec::better(acc, pr.item, gts[pr.slot], item[pr.slot])) atomicAdd(cnt_exact + pr.slot, 1);
  }
}

// ranks[s] for the slots of a filtered chunk: survivors of the certain count (cnt_hi < lim) get the exact count of
// eligible items ahead, if it is below k; every other slot -1.
__global__ void rm_rank_kernel(int n, const int32_t* __restrict__ cnt_hi, const int32_t* __restrict__ lim, const int32_t* __restrict__ cnt_exact,
                               const int32_t* __restrict__ c_r, int k, int32_t* __restrict__ ranks) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  int r = -1;
  if (cnt_hi[s] < lim[s]) {
    const int ahead = cnt_exact[s] - c_r[s];
    if (ahead < k) r = ahead;
  }
  ranks[s] = r;
}

// Exact engine: slot d answers user users[d] (recommend's list top_i[d][0 .. k)); every listed item that is in the
// user's test row (owned row users[d] - ub of tptr / tidx) gives that entry its rank: its position in the list.
// ranks is indexed by test entry and holds -1 for every entry no list reaches.
__global__ void rm_lookup_kernel(const int32_t* __restrict__ top_i, int k, int n, const int32_t* __restrict__ users, int ub,
                                 const int64_t* __restrict__ tptr, const int32_t* __restrict__ tidx, int32_t* __restrict__ ranks) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n * k) return;
  const int d = (int)(t / k), p = (int)(t % k);
  const int32_t it = top_i[t];
  if (it == rec::kNoItem || it < 0) return;
  const int r = users[d] - ub;
  int64_t lo = tptr[r], hi = tptr[r + 1];
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    const int32_t v = tidx[mid];
    if (v == it) { ranks[mid] = p; return; }
    if (v < it) lo = mid + 1; else hi = mid;
  }
}

// One warp per owned row r with n_u test entries: the hit ranks H (ranks >= 0, distinct since a row's items are)
// as a k-bit map, then lane 0 walks it in ascending order.  out[r][*] = hit rate, |H| / k, |H| / n_u,
// sum gain[h] / idcg[min(k, n_u)], (1 / min(k, n_u)) sum_{h in H} #{h' <= h} / (h + 1) and 1 / (min H + 1); all
// zero for n_u = 0.  gain[j] = ln 2 / ln(j + 2) and idcg[j] = gain[0] + .. + gain[j - 1] in that order (host
// tables, metric_ndcg).  128 threads per block.
__global__ void __launch_bounds__(128)
rm_metrics_kernel(const int64_t* __restrict__ tptr, int n_rows, const int32_t* __restrict__ ranks, int k, const double* __restrict__ gain,
                  const double* __restrict__ idcg, double* __restrict__ out) {
  __shared__ uint32_t bits[4][32];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (r >= n_rows) return;
  uint32_t* bm = bits[w];
  bm[lane] = 0u;
  __syncwarp();
  const int64_t b = tptr[r], e = tptr[r + 1];
  for (int64_t t = b + lane; t < e; t += 32) {
    const int h = ranks[t];
    if (h >= 0) atomicOr(&bm[h >> 5], 1u << (h & 31));
  }
  __syncwarp();
  if (lane != 0) return;
  double* o = out + (size_t)r * kMetrics;
  const long long n_u = e - b;
  if (n_u == 0) {
    for (int j = 0; j < kMetrics; j++) o[j] = 0.0;
    return;
  }
  int hits = 0, first = -1;
  double dcg = 0.0, ap = 0.0;
  for (int word = 0; word < (k + 31) / 32; word++) {
    uint32_t x = bm[word];
    while (x) {
      const int h = word * 32 + __ffs(x) - 1;
      x &= x - 1;
      if (first < 0) first = h;
      hits++;
      dcg = __dadd_rn(dcg, gain[h]);
      ap = __dadd_rn(ap, __ddiv_rn((double)hits, (double)(h + 1)));
    }
  }
  const int cap = (int)min((long long)k, n_u);
  o[0] = hits > 0 ? 1.0 : 0.0;
  o[1] = __ddiv_rn((double)hits, (double)k);
  o[2] = __ddiv_rn((double)hits, (double)n_u);
  o[3] = __ddiv_rn(dcg, idcg[cap]);
  o[4] = __ddiv_rn(ap, (double)cap);
  o[5] = hits > 0 ? __ddiv_rn(1.0, (double)(first + 1)) : 0.0;
}

}  // namespace rk
}  // namespace eals
