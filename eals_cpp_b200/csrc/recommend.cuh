// recommend.cuh — top-k retrieval: for each user the k unseen items of highest score.
//
// score(u, i) is predict(u, i): the sequential-k fp64 sum of separately rounded products (eval.cuh seq_dot).
// Order: score descending, ties by item id ascending — a total order, so the result does not depend on the
// engine, the scan order or the GPU count.  A user's list lives in global memory as k (score, item) entries in
// that order; an empty slot is (-inf, kNoItem), which every real item beats.
//
// Two sources feed the same per-user merge (one CTA per user, bitonic sort in shared memory):
//   SRC_EXACT  items [r0, r1) of an order (perm, nullable: identity), every score computed here in fp64 —
//              the exact engine, and the seed of the tensor-core engine (the highest-norm items);
//   SRC_PAIRS  candidate pairs emitted by the tcgen05 filter (eval_tc.cuh, MODE 2) and re-scored exactly by
//              rec_rescore_kernel, sorted by slot: only close calls, a sliver of the catalogue.
// Every entry that reaches a list was compared in fp64 under the total order; the fp16 filter only ever
// discards items it has proven to score strictly below the user's current k-th score.
#pragma once

#include "common.cuh"
#include "eval.cuh"

namespace eals {
namespace rec {

constexpr int kMaxK = 1024;
constexpr int kThreads = 256;
constexpr int kSort = 2048;             // entries sorted at once: the list (k) + up to kSort - k candidates
constexpr int32_t kNoItem = 0x7fffffff;
constexpr int kMaxFactors = 256;        // SRC_EXACT keeps the user row in shared memory

enum { SRC_EXACT = 0, SRC_PAIRS = 1 };

__device__ __forceinline__ bool better(double s1, int32_t i1, double s2, int32_t i2) {
  return s1 > s2 || (s1 == s2 && i1 < i2);
}

// item in the sorted CSR row [b, e) of idx
__device__ __forceinline__ bool row_has(const int32_t* __restrict__ idx, int64_t b, int64_t e, int32_t item) {
  while (b < e) {
    const int64_t mid = (b + e) >> 1;
    const int32_t v = idx[mid];
    if (v == item) return true;
    if (v < item) b = mid + 1; else e = mid;
  }
  return false;
}

struct MergeArgs {
  const double* U; const double* V; int K, LD;   // U: the query rows (the model's U, or query vectors)
  const int32_t* users;                 // slot -> row of U (nullable: the slot itself)
  int k;
  double* top_s; int32_t* top_i;        // [n][k] per slot
  double* thr;                          // [n] per slot: score of the k-th entry (-inf while the list is not full)
  // excluded items: CSR with a row per row of U (row = U row - row_base); ptr == nullptr: no exclusion
  const int64_t* ptr; const int32_t* idx; int row_base;
  // SRC_EXACT: list of slots (nullable: block b = slot b) and the items order[r0 .. r1) (order nullable: identity)
  const int32_t* list; const int32_t* order; int r0, r1;
  // SRC_PAIRS: block b merges run b: slot run_slot[b], sorted positions run_off[b] .. + run_cnt[b]
  const int32_t* run_slot; const int32_t* run_off; const int32_t* run_cnt;
  const int32_t* pos_pair;              // sorted position -> pair index
  const int32_t* pair_item; int pair_stride;   // item of pair t at pair_item[t * pair_stride]
  const double* pair_score;
};

// One CTA per user.  The list and a buffer of candidates that beat the current k-th entry share P = pow2 >= k + 256
// shared-memory entries; a full buffer is merged by one bitonic sort of all P.
template <int SRC>
__global__ void __launch_bounds__(kThreads)
rec_merge_kernel(MergeArgs a) {
  __shared__ double ss[kSort];
  __shared__ int32_t si[kSort];
  __shared__ double urow[kMaxFactors];
  __shared__ double sv[kThreads][9];      // SRC_EXACT: 8 factors of the round's 256 item rows
  __shared__ int32_t sitem[kThreads];
  __shared__ int fill;
  const int tid = threadIdx.x, k = a.k;
  int P = 512;
  while (P < k + kThreads) P <<= 1;
  const int cap = P - k;
  int slot, c0 = 0, c_n;
  if (SRC == SRC_EXACT) {
    slot = a.list ? a.list[blockIdx.x] : blockIdx.x;
    c_n = a.r1 - a.r0;
  } else {
    slot = a.run_slot[blockIdx.x];
    c0 = a.run_off[blockIdx.x];
    c_n = a.run_cnt[blockIdx.x];
  }
  const int u = a.users ? a.users[slot] : slot;
  double* ts = a.top_s + (size_t)slot * k;
  int32_t* ti = a.top_i + (size_t)slot * k;
  for (int t = tid; t < P; t += kThreads) {
    ss[t] = t < k ? ts[t] : -INFINITY;
    si[t] = t < k ? ti[t] : kNoItem;
  }
  if (SRC == SRC_EXACT)
    for (int t = tid; t < a.K; t += kThreads) urow[t] = a.U[(size_t)u * a.LD + t];
  if (tid == 0) fill = 0;
  int64_t rb = 0, re = 0;
  if (a.ptr) { rb = a.ptr[u - a.row_base]; re = a.ptr[u - a.row_base + 1]; }
  __syncthreads();

  auto sort_all = [&]() {       // bitonic, best first; entries past the list + fill hold (-inf, kNoItem)
    for (int size = 2; size <= P; size <<= 1)
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int t = tid; t < P / 2; t += kThreads) {
          const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
          const bool up = (lo & size) == 0;
          if (better(ss[hi], si[hi], ss[lo], si[lo]) == up) {
            const double s = ss[lo]; ss[lo] = ss[hi]; ss[hi] = s;
            const int32_t i = si[lo]; si[lo] = si[hi]; si[hi] = i;
          }
        }
        __syncthreads();
      }
    for (int t = k + tid; t < P; t += kThreads) { ss[t] = -INFINITY; si[t] = kNoItem; }
    if (tid == 0) fill = 0;
    __syncthreads();
  };

  for (int b0 = 0; b0 < c_n; b0 += kThreads) {
    // every thread must take the same branch into sort_all (it is full of barriers): read `fill` once, and let
    // no thread of this round append (atomicAdd below) before all have read it
    const int fill_now = fill;
    __syncthreads();
    if (fill_now > cap - kThreads) sort_all();
    const double ks = ss[k - 1];
    const int32_t ki = si[k - 1];
    const int c = b0 + tid;
    const bool live = c < c_n;
    double s = 0.0;
    int32_t item = 0;
    if (SRC == SRC_EXACT) {
      // seq_dot of the user row with 256 item rows, the rows staged 8 factors at a time (coalesced 64-byte pieces)
      item = live ? (a.order ? a.order[a.r0 + c] : a.r0 + c) : -1;
      sitem[tid] = item;
      __syncthreads();
      double acc = 0.0;
      for (int k0 = 0; k0 < a.K; k0 += 8) {
        for (int e = tid; e < kThreads * 4; e += kThreads) {
          const int row = e >> 2, col = (e & 3) * 2;
          const int it = sitem[row];
          double2 v = make_double2(0.0, 0.0);
          if (it >= 0 && k0 + col < a.K) v = ldg2(a.V + (size_t)it * a.LD + k0 + col);   // rows padded to LD
          sv[row][col] = v.x; sv[row][col + 1] = v.y;
        }
        __syncthreads();
        const int kend = min(8, a.K - k0);
        for (int q = 0; q < kend; q++) acc = __dadd_rn(acc, __dmul_rn(urow[k0 + q], sv[tid][q]));
        __syncthreads();
      }
      s = acc;
    } else if (live) {
      const int p = a.pos_pair[c0 + c];
      item = a.pair_item[(size_t)p * a.pair_stride];
      s = a.pair_score[p];
    }
    bool take = live && better(s, item, ks, ki);
    if (take && a.ptr) take = !row_has(a.idx, rb, re, item);
    if (take && SRC == SRC_PAIRS) {
      // already listed (a seed extension covered this item): the same (score, item) is in the list
      int lo = 0, hi = k;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (better(ss[mid], si[mid], s, item)) lo = mid + 1; else hi = mid;
      }
      take = !(lo < k && si[lo] == item);
    }
    if (take) {
      const int at = atomicAdd(&fill, 1);
      ss[k + at] = s;
      si[k + at] = item;
    }
    __syncthreads();
  }
  if (fill > 0) sort_all();
  for (int t = tid; t < k; t += kThreads) { ts[t] = ss[t]; ti[t] = si[t]; }
  if (tid == 0) a.thr[slot] = si[k - 1] == kNoItem ? -INFINITY : ss[k - 1];
}

__global__ void rec_init_kernel(double* __restrict__ top_s, int32_t* __restrict__ top_i, size_t n, double* __restrict__ thr, int n_slots) {
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (size_t)gridDim.x * blockDim.x) {
    top_s[t] = -INFINITY;
    top_i[t] = kNoItem;
    if (t < (size_t)n_slots) thr[t] = -INFINITY;
  }
}

// Every factor of the query rows X[0 .. n) finite (the filter's error bound assumes it); bad[0] = 1 + first
// offending row otherwise.
__global__ void rec_check_finite_kernel(const double* __restrict__ X, int n, int K, int LD, int* __restrict__ bad) {
  const size_t total = (size_t)n * K;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const size_t r = t / K;
    if (!isfinite(X[r * LD + t % K])) atomicMin(bad, (int)r + 1);
  }
}

// users[s] in [lo, hi) for every s; bad[0] = 1 + first offending position otherwise
__global__ void rec_check_users_kernel(const int32_t* __restrict__ users, int n, int lo, int hi, int* __restrict__ bad) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < n && (users[s] < lo || users[s] >= hi)) atomicMin(bad, s + 1);
}

// Final lists: empty slots become item -1 (score stays -inf).
__global__ void rec_finish_kernel(int32_t* __restrict__ top_i, size_t n) {
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (size_t)gridDim.x * blockDim.x)
    if (top_i[t] == kNoItem) top_i[t] = -1;
}

// Exact scores of the filter's candidate pairs (seq_dot, bit-identical to predict) and the slot sort keys.  users:
// slot -> row of U (nullable: the slot itself).
template <typename Pair>
__global__ void __launch_bounds__(128)
rec_rescore_kernel(const double* __restrict__ U, const double* __restrict__ V, int K, int LD, const int32_t* __restrict__ users,
                   const Pair* __restrict__ pairs, unsigned long long n, double* __restrict__ score,
                   uint32_t* __restrict__ key, int32_t* __restrict__ val) {
  __shared__ double sm[4][2 * 32 * 17];
  const unsigned long long n_round = (n + 31ull) & ~31ull;
  for (unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; t < n_round; t += (unsigned long long)gridDim.x * blockDim.x) {
    const bool live = t < n;
    const double *pa = nullptr, *pb = nullptr;
    int32_t slot = 0;
    if (live) {
      const Pair pr = pairs[t];
      slot = pr.slot;
      pa = U + (size_t)(users ? users[pr.slot] : pr.slot) * LD;
      pb = V + (size_t)pr.item * LD;
    }
    const double acc = seq_dot_warp32(pa, pb, K, sm[threadIdx.x >> 5]);
    if (live) {
      score[t] = acc;
      key[t] = (uint32_t)slot;
      val[t] = (int32_t)t;
    }
  }
}

// Early-out: the slot at list position p stays in the working set while some item of rank >= the next block
// may still beat its k-th score.  With items in decreasing-norm order, |score| <= |u| * max |v| over the rest
// (Cauchy-Schwarz), in the filter's scaled domain: un_hat = |u^| and rem = max (|vh| + |dv|) >= |v^| over the
// remaining tiles, both rounded up with a relative margin (1e-9) far above the fp64 rounding of seq_dot
// (K * 2^-53 < 3e-14 for K <= 256).  bound < t^ (rounded down) means every remaining score is STRICTLY below
// the k-th: none can enter, ties by item id included.
__global__ void rec_keep_flags_kernel(const int32_t* __restrict__ list, const int32_t* __restrict__ n_list, int n_max,
                                      const float* __restrict__ un_hat, const float4* __restrict__ sp0, const double* __restrict__ thr,
                                      float rem, uint8_t* __restrict__ flags) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_max) return;
  const int n = n_list ? *n_list : n_max;
  uint8_t f = 0;
  if (p < n) {
    const int s = list ? list[p] : p;
    const float bound = __fmul_ru(un_hat[s], rem);
    f = thr[s] != -INFINITY && !(bound < sp0[s].y);
  }
  flags[p] = f;
}

// Cosine catalogue of similar(): out[r] = Y[r] / |Y[r]| for the rows [0, rows) of Y [rows][LD], with
// |y| = __dsqrt_rn(seq_dot(y, y)) and one __ddiv_rn per factor, so the normalised rows are defined bit for bit.  A row
// of norm 0 stays zero; the padding columns [K, LD) are written as zeros.  One warp per row: the row is read as
// coalesced 256-byte pieces (LD <= kMaxFactors, so at most 8 per lane stay in registers) and its squares are added
// in factor order through shuffles, every lane holding the same sum.
__global__ void sim_normalize_kernel(const double* __restrict__ Y, int rows, int K, int LD, double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < rows; r += warps) {
    const double* y = Y + (size_t)r * LD;
    double v[kMaxFactors / 32];
    double acc = 0.0;
#pragma unroll
    for (int c = 0; c < kMaxFactors / 32; c++) {
      const int k0 = c * 32;
      v[c] = 0.0;
      if (k0 < K) {
        if (k0 + lane < K) v[c] = y[k0 + lane];
        const double p = __dmul_rn(v[c], v[c]);
        const int kend = min(32, K - k0);
        for (int j = 0; j < kend; j++) acc = __dadd_rn(acc, __shfl_sync(kFullMask, p, j));
      }
    }
    const double norm = __dsqrt_rn(acc);
    double* o = out + (size_t)r * LD;
#pragma unroll
    for (int c = 0; c < kMaxFactors / 32; c++) {
      const int k = c * 32 + lane;
      if (k < LD) o[k] = k < K && norm != 0.0 ? __ddiv_rn(v[c], norm) : 0.0;
    }
  }
}

// The query rows of similar() and their self-exclusion CSR: qx[s] = Yhat[ids[s]] ([n][LD]) and ex_ptr[s] = s for
// s <= n, so that row s of the CSR over the index array `ids` is the query's own id and nothing else.
__global__ void sim_queries_kernel(const double* __restrict__ Yhat, int LD, const int32_t* __restrict__ ids, int n,
                                   double* __restrict__ qx, int64_t* __restrict__ ex_ptr) {
  const size_t total = (size_t)n * LD;   // >= n + 1 (LD >= 16, n >= 1)
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const size_t s = t / LD;
    qx[t] = Yhat[(size_t)ids[s] * LD + t % LD];
    if (t <= (size_t)n) ex_ptr[t] = (int64_t)t;
  }
}

// flags[p] = 1 when slot p's list is not full yet (the seed has to be extended for it)
__global__ void rec_unfilled_flags_kernel(const int32_t* __restrict__ list, const int32_t* __restrict__ n_list, int n_max,
                                          const double* __restrict__ thr, uint8_t* __restrict__ flags) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_max) return;
  const int n = n_list ? *n_list : n_max;
  uint8_t f = 0;
  if (p < n) f = thr[list ? list[p] : p] == -INFINITY;
  flags[p] = f;
}

}  // namespace rec
}  // namespace eals
