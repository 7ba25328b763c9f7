// eals_b200.cu — libeals_b200.so: the C ABI of include/eals_b200.h over the sm_100a kernels in this
// directory.  Host-side logic here is limited to what the reference's constructor does once
// (popularity weights, factor initialisation — both on the host with the SAME libm / libstdc++
// calls as the reference, so they are bit-identical by construction), row bucketing by length,
// launch sequencing, and the replay of the reference's int-truncating partial_sort_copy for the
// few users that survive the count-larger filter in evaluation.
//
// There is no CPU compute fallback: every entry point that does work needs a CUDA device.

#include "../../include/eals_b200.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstring>
#include <limits>
#include <new>
#include <random>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include <cuda.h>
#include <cuda_fp16.h>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_run_length_encode.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "cd_block.cuh"
#include "cd_sweep.cuh"
#include "common.cuh"
#include "eval.cuh"
#include "eval_tc.cuh"
#include "gram.cuh"
#include "loss.cuh"
#include "ranking.cuh"
#include "recommend.cuh"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CU(call)                                                                                 \
  do {                                                                                           \
    cudaError_t e_ = (call);                                                                     \
    if (e_ != cudaSuccess)                                                                       \
      return fail(e_ == cudaErrorMemoryAllocation ? EALS_ERR_ALLOC : EALS_ERR_CUDA,              \
                  "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));          \
  } while (0)

#define OK(call)                 \
  do {                           \
    int r_ = (call);             \
    if (r_ != EALS_OK) return r_; \
  } while (0)

// EALS_VERBOSE=1: wall-clock of the setup stages on stderr.
struct StageTimer {
  bool on;
  std::chrono::steady_clock::time_point t;
  StageTimer() : on(getenv("EALS_VERBOSE") && getenv("EALS_VERBOSE")[0] == '1'), t(std::chrono::steady_clock::now()) {}
  void lap(const char* what) {
    if (!on) return;
    cudaDeviceSynchronize();
    const auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[eals] %-28s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(now - t).count());
    t = now;
  }
};

// Host-side helper: fn(thread, begin, end) over [0, n) in contiguous chunks on up to 16 threads.
template <typename F>
void parallel_chunks(int64_t n, int* n_threads_out, F fn, int64_t min_per_thread = 65536) {
  unsigned hw = std::thread::hardware_concurrency();
  int T = (int)std::min<int64_t>(std::max(1u, std::min(hw, 16u)), std::max<int64_t>(1, n / min_per_thread));
  if (n_threads_out) *n_threads_out = T;
  if (T <= 1) { fn(0, (int64_t)0, n); return; }
  std::vector<std::thread> th;
  const int64_t per = (n + T - 1) / T;
  for (int t = 0; t < T; t++) th.emplace_back(fn, t, std::min(n, t * per), std::min(n, (t + 1) * per));
  for (auto& x : th) x.join();
}
constexpr int kMaxHostThreads = 16;

template <typename T>
int dev_alloc(T** p, size_t n) {
  *p = nullptr;
  if (n == 0) n = 1;
  CU(cudaMalloc((void**)p, n * sizeof(T)));
  return EALS_OK;
}

// Grow-only device buffer: reallocated only when the request exceeds the capacity, so that replacing
// the train matrix by one of the same shape (setTrain) does not free and re-allocate gigabytes.
template <typename T>
int dev_reserve(T** p, size_t* cap, size_t n) {
  if (n == 0) n = 1;
  if (*p && n <= *cap) return EALS_OK;
  cudaFree(*p);
  *p = nullptr;
  *cap = 0;
  CU(cudaMalloc((void**)p, n * sizeof(T)));
  *cap = n;
  return EALS_OK;
}

// Where the receive area of the copy-engine exchange starts inside a prediction-cache allocation of n values.
inline size_t recv_offset(int64_t n) { return ((size_t)n + 15) & ~(size_t)15; }

// Buckets of owned rows by length.  Bucket 0 = empty rows (skipped: MF_fastALS.cpp:249,344).
// 1..4: one warp per row (1/2/3/4 nonzeros per lane); 5..7: one CTA per row (4 warps x 2, 4 x 3,
// 8 x 2 nonzeros per thread); 8: heavy rows, split into slabs.  The finer the buckets, the closer a
// row's shared-memory tile is to its real length and the more rows an SM holds in flight.
// Measured on c4: rows of 513..1024 nonzeros run faster through the slab pipeline than as one CTA.
constexpr int kNumBuckets = 9;
constexpr int kBucketMax[kNumBuckets] = {0, 32, 64, 96, 128, 256, 384, 512, 0x7fffffff};
constexpr int kMidBucket = 5;     // first one-CTA-per-row bucket
constexpr int kHeavyBucket = 8;
// Heavy rows per launch group.  Measured on c4 (profiles/README.md r01b): launch granularity matters
// more than keeping one factor block of the batch L2-resident (384k nnz: 363 ms, 24M nnz: 204 ms).
// Since the slabs of a batch are launched in neighbour order (HeavyUnits::launch) the bigger the batch
// the more slabs share a gathered line while it is in L2, so by default ALL heavy rows of a side form
// one batch (the limit only bounds the partials scratch: 6.5 bytes per nonzero).
constexpr int64_t kDefaultBatchNnz = 4LL * 1024 * 1024 * 1024;

struct HeavyBatch { int h0, h1, u0, u1; };

struct Side {
  int rows = 0;       // owned rows
  int row_base = 0;   // global id of owned row 0
  int64_t nnz = 0;    // nonzeros of the owned rows
  int64_t* ptr = nullptr;
  int32_t* idx = nullptr;
  double* val = nullptr;
  int32_t* order = nullptr;           // owned-row ids grouped by bucket, ascending id inside
  int first[kNumBuckets + 1] = {0};   // bucket b = order[first[b] .. first[b+1])
  // heavy rows (bucket kHeavyBucket): row h = order[first[kHeavyBucket] + h], longest first
  int n_hrows = 0, n_units = 0, max_batch_units = 0;
  int64_t heavy_nnz = 0;
  eals::UnitDesc* units_canon = nullptr;    // slab descriptors, canonical order (row by row)
  eals::UnitDesc* units_launch = nullptr;   // the same, every canonical batch in neighbour order
  int slab = eals::kMaxSlab;                // nonzeros per slab (= threads of a heavy_step CTA)
  int32_t *hrow_id = nullptr, *hrow_unit0 = nullptr, *hrow_units = nullptr;
  int32_t *hrow_grp0 = nullptr, *hrow_grps = nullptr, *grp_unit0 = nullptr, *grp_cnt = nullptr;
  int64_t* hrow_poff = nullptr;       // offset of heavy row h in the compact prediction cache
  size_t cap_hrow_poff = 0;
  int32_t* unit_launch = nullptr;     // scratch: sorted canonical unit ids of a batch
  uint32_t *sort_keys = nullptr, *sort_keys_out = nullptr;   // scratch of build_launch_order, kept across setTrain
  int32_t* sort_vals = nullptr;
  unsigned char* sort_tmp = nullptr;
  size_t cap_sort_keys = 0, cap_sort_keys_out = 0, cap_sort_vals = 0, cap_sort_tmp = 0;
  int n_groups = 0;
  std::vector<int32_t> h_hrow_grp0, h_hrow_grps;
  std::vector<int32_t> h_hrow_unit0, h_hrow_units;
  std::vector<int32_t> h_row_to_hrow;  // owned row -> heavy index or -1 (only filled when heavy rows exist)
  std::vector<HeavyBatch> batches;
  double* pred = nullptr;             // prediction cache of the heavy rows (compact)
  double* delta = nullptr;            // [n_hrows][16] factor changes of the current block
  // capacities (elements) of the device arrays above, see dev_reserve
  size_t cap_ptr = 0, cap_idx = 0, cap_val = 0, cap_order = 0, cap_units_canon = 0, cap_units_launch = 0, cap_hrow_id = 0, cap_hrow_unit0 = 0, cap_hrow_units = 0, cap_pred = 0,
         cap_delta = 0, cap_hrow_grp0 = 0, cap_hrow_grps = 0, cap_grp_unit0 = 0, cap_grp_cnt = 0, cap_unit_launch = 0;
  std::vector<int64_t> h_ptr;         // host copy of ptr (rebased to 0)
};

enum { T_USER_SWEEP, T_USER_GRAM, T_ITEM_SWEEP, T_ITEM_GRAM, T_LOSS, T_EVAL,
       // sub-phases of the sweeps (eals_timings_detail): heavy slab pipeline, one-CTA rows, warp rows
       T_U_HEAVY, T_U_MID, T_U_WARP, T_I_HEAVY, T_I_MID, T_I_WARP, T_COUNT };
constexpr int kPublicTimers = 6;

// What the last evaluate / recommend did (eals_eval_stats, eals_recommend_stats).  engine: 0 exact fp64, 1 tcgen05
// filter + exact re-score.  blk0: the first filtered item block's users, items and device time, zero unless that
// block ran as one launch.
struct BlockTiming { long long users = 0, items = 0; double ms = 0; };
struct EvalStats { int engine = 0; long long candidates = 0, pairs = 0; BlockTiming blk0; };
struct RecStats { int engine = 0; long long seed = 0, pairs = 0, left1 = 0; BlockTiming blk0; };   // left1: users left after block 1

}  // namespace

struct eals_model {
  eals_params p;
  cudaStream_t own_stream = nullptr;
  int K = 0, LD = 0;
  int M = 0, N = 0;
  int ub = 0, ue = 0, ib = 0, ie = 0;
  cudaStream_t stream = nullptr;
  double *U = nullptr, *V = nullptr, *SU = nullptr, *SV = nullptr, *Wi = nullptr;
  double* terms = nullptr;      // [4] loss terms
  double* partials = nullptr;   // scratch for deterministic two-stage reductions
  size_t partials_len = 0;
  Side users, items;
  int sm_count = 148;
  int64_t launches = 0;
  double last_ms[T_COUNT] = {0};
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending[T_COUNT];  // not yet folded into acc_ms
  std::vector<cudaEvent_t> pool;
  double acc_ms[T_COUNT] = {0};
  int64_t acc_calls[T_COUNT] = {0};
  bool factors_set = false;
  struct eals_eval_ws* eval = nullptr;   // evaluation workspace (grow-only)
  EvalStats eval_stats;
  RecStats rec_stats;
  double init_stream_s = 0;              // host seconds of the last factor-stream generation
  bool su_fresh = true;          // SU describes the current U (false after single-row user updates without a Gram)
  double* S_tmp = nullptr;       // [LD][LD] scratch Gram for loss() while SU is stale
  int* flags = nullptr;          // [8] device scratch for validation kernels (no malloc/free per call)
  eals::PeerSet peersU = {}, peersV = {};   // IPC mappings of the other ranks' U / V replicas
  // symmetric prediction cache (single-rank models only)
  double* pc_u = nullptr;        // predictions of the owned user rows' nonzeros (CSR order)
  double* pc_i = nullptr;        // predictions of the owned item columns' nonzeros (CSC order)
  uint32_t* map_u = nullptr;     // owned CSR nonzero -> global CSC position of the same nonzero
  uint32_t* map_i = nullptr;     // owned CSC nonzero -> global CSR position
  size_t cap_pc_u = 0, cap_pc_i = 0, cap_map_u = 0, cap_map_i = 0;
  // multi-rank: staged routing of the final predictions (see CdSide::pc_stage)
  double *pc_stage_u = nullptr, *pc_stage_i = nullptr;
  uint32_t *route_src_u = nullptr, *route_dst_u = nullptr, *route_src_i = nullptr, *route_dst_i = nullptr;
  size_t cap_stage_u = 0, cap_stage_i = 0, cap_rsrc_u = 0, cap_rdst_u = 0, cap_rsrc_i = 0, cap_rdst_i = 0;
  bool routed = false;
  // Copy-engine exchange of the staged predictions (multi-rank): pair_cnt[su][ri] = nonzeros whose user belongs to
  // rank su and whose item to rank ri (every rank computes the whole table from the full index arrays).  A sender's
  // staging array is already in destination order, i.e. segmented by destination rank; each segment is copied
  // (cudaMemcpyAsync, peer-to-peer: no SM involved, runs under the Gram) into the receiver's RECEIVE area — the
  // second half of the allocation that holds the receiver's prediction cache, so no extra mapping is needed — at the
  // offset that belongs to this sender; before its next sweep the receiver unpacks the area into the cache through
  // recv_idx (a stable partition of its nonzeros by source rank: the order every sender's segment arrives in).
  long long pair_cnt[8][8] = {{0}};
  uint32_t *recv_idx_u = nullptr, *recv_idx_i = nullptr;
  size_t cap_recv_idx_u = 0, cap_recv_idx_i = 0;
  bool copy_route = false;
  bool unpack_u_pending = false, unpack_i_pending = false;
  // multi-rank: a prediction cache that had to grow is not freed while peers may still map it (CUDA IPC):
  // the old buffer waits here until eals_ipc_gc; ipc_gen counts such reallocations
  std::vector<void*> graveyard;
  int ipc_gen = 0;
  // multi-rank, host input: device copies of the FULL offset / index arrays for the position maps, and the
  // sort scratch of the routes — kept across setTrain (cudaMalloc / cudaFree per call cost 0.5 s at c4)
  int64_t *full_rp = nullptr, *full_cp = nullptr;
  int32_t *full_ci = nullptr, *full_ri = nullptr;
  unsigned char* route_tmp = nullptr;
  size_t cap_full_rp = 0, cap_full_cp = 0, cap_full_ci = 0, cap_full_ri = 0, cap_route_tmp = 0;
  eals::PcOut out_to_items = {}, out_to_users = {};   // where the other side's caches live (all ranks)
  int n_ranks = 1, rank = 0;
  cudaStream_t side_stream = nullptr;   // routing of the final predictions runs here, under the Gram
  cudaEvent_t ev_swept = nullptr, ev_routed = nullptr;
  // two more streams for the peer-to-peer copies: several copy engines work at once (one stream serialises the
  // 7 copies of an 8-GPU exchange; each is too small to fill NVLink on its own)
  cudaStream_t copy_stream[2] = {nullptr, nullptr};
  cudaEvent_t ev_copied[2] = {nullptr, nullptr};
  bool route_pending = false;
  // whole epochs as one CUDA graph (eals_run_epochs): the launch-bound configurations (yelp-sized matrices:
  // ~170 launches of a few microseconds each per epoch) replay a captured epoch instead of re-issuing it
  cudaGraphExec_t epoch_graph = nullptr;
  long long graph_key = -1, config_gen = 0;
  long long graph_launches_per_epoch = 0;
  bool capturing = false;
  int route_todo = 0;            // 1 / 2: the user / item sweep's staged predictions still have to be routed
  bool local_peers = false;      // peers are plain pointers of models in this process (eals_group), not CUDA IPC mappings
  bool pc_attached = false;      // caches usable: single rank, or both peers' cache sets mapped
  bool pc_users_attached = false, pc_items_attached = false;
  bool pcache_on = false;        // structures built for the current matrix
  bool pc_u_valid = false, pc_i_valid = false;
  int sweeps_since_fresh = 0;
  int pred_refresh_every = 0;    // EALS_PRED_REFRESH_EVERY: recompute the cache from scratch every n sweeps (0 = never)
};

namespace {

using eals::CdSide;

int sync_if_debug(eals_model* m) {
  if (m->p.flags & EALS_FLAG_SYNC_EACH_CALL) {
    CU(cudaStreamSynchronize(m->stream));
    CU(cudaGetLastError());
  }
  return EALS_OK;
}

int check_launch(eals_model* m) {
  m->launches++;
  CU(cudaGetLastError());
  return EALS_OK;
}

void free_side(Side& s) {
  cudaFree(s.ptr); cudaFree(s.idx); cudaFree(s.val); cudaFree(s.order);
  cudaFree(s.pred); cudaFree(s.delta);
  cudaFree(s.units_canon); cudaFree(s.units_launch);
  cudaFree(s.hrow_id); cudaFree(s.hrow_unit0); cudaFree(s.hrow_units);
  cudaFree(s.hrow_poff);
  cudaFree(s.hrow_grp0); cudaFree(s.hrow_grps); cudaFree(s.grp_unit0); cudaFree(s.grp_cnt); cudaFree(s.unit_launch);
  cudaFree(s.sort_keys); cudaFree(s.sort_keys_out); cudaFree(s.sort_vals); cudaFree(s.sort_tmp);
  s = Side();
}

// Copy `n` elements from a host or device source to a device destination.
template <typename T>
int copy_in(T* dst, const T* src, size_t n, int space, cudaStream_t st) {
  if (n == 0) return EALS_OK;
  CU(cudaMemcpyAsync(dst, src, n * sizeof(T),
                     space == EALS_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
  return EALS_OK;
}

// One warp per row (grid-stride): every index in range and strictly larger than its predecessor.
// Indices in range and strictly ascending inside every row, flat over the nonzeros so that a column with
// millions of entries costs no more than its share (one warp per row took 26 ms on c4's item side):
// `descents` counts the positions whose index does not exceed its predecessor's; each of them is legal
// only as the first nonzero of a row, which check_row_starts_kernel counts — equal counts <=> sorted.
__global__ void check_indices_kernel(const int32_t* __restrict__ idx, int64_t nnz, int limit,
                                     int* __restrict__ bad, unsigned long long* __restrict__ descents) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool oob = false, desc = false;
  if (q < nnz) {
    const int c = idx[q];
    oob = c < 0 || c >= limit;
    desc = q > 0 && idx[q - 1] >= c;
  }
  if (__syncthreads_or(oob) && threadIdx.x == 0) atomicExch(bad, 1);
  const int nd = __syncthreads_count(desc);
  if (nd && threadIdx.x == 0) atomicAdd(descents, (unsigned long long)nd);
}
__global__ void check_row_starts_kernel(const int64_t* __restrict__ ptr, const int32_t* __restrict__ idx, int rows,
                                        unsigned long long* __restrict__ starts) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  bool hit = false;
  if (r < rows) {
    const int64_t q = ptr[r];
    hit = q > 0 && ptr[r + 1] > q && idx[q - 1] >= idx[q];
  }
  const int n = __syncthreads_count(hit);
  if (n && threadIdx.x == 0) atomicAdd(starts, (unsigned long long)n);
}

int ensure_partials(eals_model* m, size_t n);

// Both position maps in one pass over the FULL CSC arrays, one thread per nonzero q: its column i
// (search in the offsets; neighbouring threads walk the same path), its user u = row_idx[q] and the
// CSR position p of (u, i) — a search inside the SHORT row u instead of inside a column that may
// hold millions of entries.  map_i[q] = p for the owned items, map_u[p] = q for the owned users.
struct RankBounds {
  int32_t user[9], item[9];
  int n;                                    // ranks (<= 1: no table)
};

__global__ void build_maps_kernel(const int64_t* __restrict__ cp, const int32_t* __restrict__ ri, int N,
                                  const int64_t* __restrict__ rp, const int32_t* __restrict__ ci, int64_t nnz,
                                  int ub, int ue, int64_t rp_ub, uint32_t* __restrict__ map_u,
                                  int ib, int ie, int64_t cp_ib, uint32_t* __restrict__ map_i, int* __restrict__ bad,
                                  RankBounds rb, unsigned long long* __restrict__ pair_cnt) {
  __shared__ unsigned int hist[64];
  if (rb.n > 1) {
    if (threadIdx.x < 64) hist[threadIdx.x] = 0;
    __syncthreads();
  }
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int i = 0, u = 0;
  bool own_u = false, own_i = false;
  if (q < nnz) {
    int lo = 0, hi = N;                     // largest i with cp[i] <= q
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (cp[mid] <= q) lo = mid; else hi = mid;
    }
    i = lo; u = ri[q];
    own_u = u >= ub && u < ue; own_i = i >= ib && i < ie;
    if (rb.n > 1) {                         // (owner of the user, owner of the item) of this nonzero
      int su = 0, si = 0;
#pragma unroll
      for (int t = 1; t < 8; t++) { su += (t < rb.n && u >= rb.user[t]) ? 1 : 0; si += (t < rb.n && i >= rb.item[t]) ? 1 : 0; }
      atomicAdd(&hist[su * 8 + si], 1u);
    }
  }
  if (rb.n > 1) {
    __syncthreads();
    if (threadIdx.x < 64 && hist[threadIdx.x]) atomicAdd(pair_cnt + threadIdx.x, (unsigned long long)hist[threadIdx.x]);
  }
  if (q >= nnz) return;
  if (!own_u && !own_i) return;
  int64_t a = rp[u], b = rp[u + 1];
  while (b - a > 1) {
    const int64_t mid = (a + b) >> 1;
    if (ci[mid] <= i) a = mid; else b = mid;
  }
  if (!(b > a && ci[a] == i)) { atomicExch(bad, 1); return; }
  if (own_i) map_i[q - cp_ib] = (uint32_t)a;
  if (own_u) map_u[a - rp_ub] = (uint32_t)q;
}

// key[t] = rank that owns idx[t] (bounds[0..n]); val[t] = t
__global__ void source_rank_kernel(const int32_t* __restrict__ idx, int64_t n, RankBounds rb, bool by_user,
                                   uint32_t* __restrict__ key, uint32_t* __restrict__ val) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int x = idx[t];
  int r = 0;
#pragma unroll
  for (int k = 1; k < 8; k++) r += (k < rb.n && x >= (by_user ? rb.user[k] : rb.item[k])) ? 1 : 0;
  key[t] = (uint32_t)r;
  val[t] = (uint32_t)t;
}

// cache[recv_idx[k]] = recv[k]: the receive area (segments in source-rank order) into the prediction cache
// Slots [local_lo, local_hi) — the segment this rank sent to itself — are read straight from the sender-side
// staging array instead (no copy for them: a same-device cudaMemcpyAsync is an SM kernel, and an SM kernel queues
// behind the Gram's CTAs, which fill the register file).
__global__ void __launch_bounds__(256)
pc_unpack_kernel(const double* __restrict__ recv, const uint32_t* __restrict__ recv_idx, int64_t n, double* __restrict__ cache,
                 const double* __restrict__ local_src, int64_t local_lo, int64_t local_hi) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride)
    cache[recv_idx[k]] = (k >= local_lo && k < local_hi) ? local_src[k - local_lo] : recv[k];
}

__global__ void check_perm_kernel(const uint32_t* __restrict__ perm, int64_t nnz, int* __restrict__ bad) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q < nnz && perm[q] == 0xffffffffu) atomicExch(bad, 1);
}

__global__ void iota_kernel(uint32_t* __restrict__ v, int64_t n) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) v[t] = (uint32_t)t;
}

// Destination order of one side's nonzeros (cub radix sort, once per matrix): route_dst = the map values
// ascending; rsrc ends up holding, per LOCAL nonzero, its slot in that order — the index the sweep kernels
// scatter their final predictions through (CdSide::pc_map in staged mode).
int build_routes(eals_model* m, const uint32_t* map, int64_t n, double** stage, size_t* cap_stage,
                 uint32_t** rsrc, size_t* cap_rsrc, uint32_t** rdst, size_t* cap_rdst) {
  OK(dev_reserve(stage, cap_stage, (size_t)n));
  OK(dev_reserve(rsrc, cap_rsrc, (size_t)n));
  OK(dev_reserve(rdst, cap_rdst, (size_t)n));
  if (n == 0) return EALS_OK;
  if (n >= 0x7fffffffLL) return fail(EALS_ERR_UNSUPPORTED, "too many nonzeros per rank for the routed prediction cache");
  uint32_t* iota = reinterpret_cast<uint32_t*>(*stage);   // scratch: the staging buffer is not live yet
  iota_kernel<<<(unsigned)((n + 255) / 256), 256, 0, m->stream>>>(iota, n);
  OK(check_launch(m));
  size_t tmp_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, map, *rdst, iota, *rsrc, (int)n, 0, 32, m->stream);
  OK(dev_reserve(&m->route_tmp, &m->cap_route_tmp, std::max<size_t>(tmp_bytes, 16)));
  const cudaError_t e = cub::DeviceRadixSort::SortPairs(m->route_tmp, tmp_bytes, map, *rdst, iota, *rsrc, (int)n, 0, 32, m->stream);
  if (e != cudaSuccess) return fail(EALS_ERR_CUDA, "route sort -> %s", cudaGetErrorString(e));
  // the kernels scatter into the staging array through the INVERSE permutation (local nonzero -> slot in
  // destination order); rsrc is replaced by it (the staging buffer, not live yet, is the scratch)
  eals::invert_perm_kernel<<<(unsigned)((n + 255) / 256), 256, 0, m->stream>>>(*rsrc, n, iota);
  OK(check_launch(m));
  CU(cudaMemcpyAsync(*rsrc, iota, sizeof(uint32_t) * (size_t)n, cudaMemcpyDeviceToDevice, m->stream));
  CU(cudaStreamSynchronize(m->stream));
  return EALS_OK;
}

// Unmap the other ranks' prediction caches (multi-rank models).
void close_pc_peers(eals_model* m, eals::PcOut& out, bool& attached_flag) {
  for (int r = 0; r < out.n; r++)
    if (r != m->rank && out.base[r]) {
      if (!m->local_peers) cudaIpcCloseMemHandle(out.base[r]);
      out.base[r] = nullptr;
    }
  attached_flag = false;
}

// (Re)build the symmetric prediction cache structures after the matrix changed.  Needs the FULL
// offsets and index arrays of both orientations (the arguments of eals_create / eals_set_train).
int build_pred_cache(eals_model* m, int space, const int64_t* row_ptr, const int32_t* col_idx,
                     const int64_t* col_ptr, const int32_t* row_idx) {
  StageTimer tm;
  m->pc_u_valid = m->pc_i_valid = false;
  m->pcache_on = false;
  const bool was_attached = m->pc_attached;
  m->pc_attached = false;
  const bool single = m->ub == 0 && m->ue == m->M && m->ib == 0 && m->ie == m->N;
  const bool multi = !single && m->n_ranks > 1;
  const char* off = getenv("EALS_NO_PRED_CACHE");
  if ((!single && !multi) || m->users.nnz == 0 || m->items.nnz == 0 || (off && off[0] == '1')) return EALS_OK;
  // total nonzeros must fit the 32-bit positions of the maps
  std::vector<int64_t> rp((size_t)m->n_ranks + 1), cp((size_t)m->n_ranks + 1);
  auto fetch = [&](const int64_t* src, int64_t at, int64_t* dst) -> int {
    if (space == EALS_DEVICE) CU(cudaMemcpy(dst, src + at, sizeof(int64_t), cudaMemcpyDeviceToHost));
    else *dst = src[at];
    return EALS_OK;
  };
  int64_t nnz_total = 0;
  OK(fetch(row_ptr, m->M, &nnz_total));
  if (nnz_total >= 0xffffffffLL) return EALS_OK;
  for (int r = 0; r <= m->n_ranks; r++) {
    OK(fetch(row_ptr, single ? (r ? m->M : 0) : m->p.user_bounds[r], &rp[r]));
    OK(fetch(col_ptr, single ? (r ? m->N : 0) : m->p.item_bounds[r], &cp[r]));
  }
  // full arrays of the OTHER orientation on the device (temporary copies when the input is on the host
  // and this model holds only a slice)
  const int64_t* d_rp = nullptr; const int32_t* d_ci = nullptr; const int64_t* d_cp = nullptr; const int32_t* d_ri = nullptr;
  if (single) {
    d_rp = m->users.ptr; d_ci = m->users.idx; d_cp = m->items.ptr; d_ri = m->items.idx;
  } else if (space == EALS_DEVICE) {
    d_rp = row_ptr; d_ci = col_idx; d_cp = col_ptr; d_ri = row_idx;
  } else {
    OK(dev_reserve(&m->full_rp, &m->cap_full_rp, (size_t)m->M + 1)); OK(dev_reserve(&m->full_cp, &m->cap_full_cp, (size_t)m->N + 1));
    OK(dev_reserve(&m->full_ci, &m->cap_full_ci, (size_t)nnz_total)); OK(dev_reserve(&m->full_ri, &m->cap_full_ri, (size_t)nnz_total));
    CU(cudaMemcpyAsync(m->full_rp, row_ptr, sizeof(int64_t) * (m->M + 1), cudaMemcpyHostToDevice, m->stream));
    CU(cudaMemcpyAsync(m->full_cp, col_ptr, sizeof(int64_t) * (m->N + 1), cudaMemcpyHostToDevice, m->stream));
    CU(cudaMemcpyAsync(m->full_ci, col_idx, sizeof(int32_t) * nnz_total, cudaMemcpyHostToDevice, m->stream));
    CU(cudaMemcpyAsync(m->full_ri, row_idx, sizeof(int32_t) * nnz_total, cudaMemcpyHostToDevice, m->stream));
    d_rp = m->full_rp; d_ci = m->full_ci; d_cp = m->full_cp; d_ri = m->full_ri;
  }
  const int64_t nu = m->users.nnz, ni = m->items.nnz;
  {   // the caches themselves: growing one while peers map it (multi-rank) must not free it under them
    auto reserve_shared = [&](double** p, size_t* cap, size_t n) -> int {
      if (*p && n <= *cap) return EALS_OK;
      if (*p && m->n_ranks > 1) { m->graveyard.push_back(*p); *p = nullptr; *cap = 0; }
      m->ipc_gen++;
      // a little headroom: matrices of similar size keep the buffers.  Several ranks: the allocation is the
      // cache followed by the receive area of the copy-engine exchange (recv_offset() doubles further on)
      const size_t want = n + n / 16;
      if (!multi) return dev_reserve(p, cap, want);
      cudaFree(*p);
      *p = nullptr; *cap = 0;
      CU(cudaMalloc((void**)p, sizeof(double) * (2 * (want + 16) + 16)));
      *cap = want;
      return EALS_OK;
    };
    OK(reserve_shared(&m->pc_u, &m->cap_pc_u, (size_t)nu));
    OK(reserve_shared(&m->pc_i, &m->cap_pc_i, (size_t)ni));
  }
  OK(dev_reserve(&m->map_u, &m->cap_map_u, (size_t)nu));
  OK(dev_reserve(&m->map_i, &m->cap_map_i, (size_t)ni));
  int* bad = m->flags + 14;
  CU(cudaMemsetAsync(bad, 0, sizeof(int), m->stream));
  CU(cudaMemsetAsync(m->map_u, 0xff, sizeof(uint32_t) * (size_t)nu, m->stream));   // unreached CSR entries stay invalid
  RankBounds rb;
  rb.n = multi ? m->n_ranks : 1;
  for (int r = 0; r <= 8; r++) {
    rb.user[r] = multi && r <= m->n_ranks ? m->p.user_bounds[r] : 0;
    rb.item[r] = multi && r <= m->n_ranks ? m->p.item_bounds[r] : 0;
  }
  OK(ensure_partials(m, 64));
  unsigned long long* d_pairs = reinterpret_cast<unsigned long long*>(m->partials);
  CU(cudaMemsetAsync(d_pairs, 0, 64 * sizeof(unsigned long long), m->stream));
  {
    const int me_ = single ? 0 : m->rank;
    build_maps_kernel<<<(unsigned)((nnz_total + 255) / 256), 256, 0, m->stream>>>(
        d_cp, d_ri, m->N, d_rp, d_ci, nnz_total, m->ub, m->ue, rp[me_], m->map_u, m->ib, m->ie, cp[me_], m->map_i, bad, rb, d_pairs);
    OK(check_launch(m));
  }
  unsigned long long h_pairs[64];
  CU(cudaMemcpyAsync(h_pairs, d_pairs, sizeof(h_pairs), cudaMemcpyDeviceToHost, m->stream));
  check_perm_kernel<<<(unsigned)((nu + 255) / 256), 256, 0, m->stream>>>(m->map_u, nu, bad);
  OK(check_launch(m));
  int h_bad = 0;
  CU(cudaMemcpyAsync(&h_bad, bad, sizeof(int), cudaMemcpyDeviceToHost, m->stream));
  CU(cudaStreamSynchronize(m->stream));
  if (h_bad) return fail(EALS_ERR_ARG, "the CSR and CSC arrays do not describe the same matrix");
  for (int a = 0; a < 8; a++)
    for (int b = 0; b < 8; b++) m->pair_cnt[a][b] = (long long)h_pairs[a * 8 + b];
  // destination tables; the own rank's entries are filled now, the peers' by eals_ipc_attach
  const int nr = single ? 1 : m->n_ranks, me = single ? 0 : m->rank;
  {   // the peers' mappings stay (their buffers only move when THEY report a new ipc generation)
    const eals::PcOut old_items = m->out_to_items, old_users = m->out_to_users;
    m->out_to_items = eals::PcOut{}; m->out_to_users = eals::PcOut{};
    if (multi && was_attached)
      for (int r = 0; r < nr; r++) { m->out_to_items.base[r] = old_items.base[r]; m->out_to_users.base[r] = old_users.base[r]; }
  }
  m->out_to_items.n = m->out_to_users.n = nr;
  for (int r = 0; r <= nr; r++) {
    m->out_to_items.bound[r] = (uint32_t)cp[r];   // user sweeps write CSC-ordered caches
    m->out_to_users.bound[r] = (uint32_t)rp[r];   // item sweeps write CSR-ordered caches
  }
  m->out_to_items.base[me] = m->pc_i;
  m->out_to_users.base[me] = m->pc_u;
  m->pc_attached = single || (multi && was_attached);
  tm.lap("pred cache: position maps");
  m->routed = false;
  if (multi && !(getenv("EALS_PC_ROUTE") && getenv("EALS_PC_ROUTE")[0] == '0')) {
    OK(build_routes(m, m->map_u, nu, &m->pc_stage_u, &m->cap_stage_u, &m->route_src_u, &m->cap_rsrc_u, &m->route_dst_u, &m->cap_rdst_u));
    OK(build_routes(m, m->map_i, ni, &m->pc_stage_i, &m->cap_stage_i, &m->route_src_i, &m->cap_rsrc_i, &m->route_dst_i, &m->cap_rdst_i));
    m->routed = true;
    // receiver side of the copy-engine exchange: the order the senders' segments arrive in = this rank's nonzeros
    // stably partitioned by the rank that owns the OTHER index (users of an item column ascend and a rank's
    // users are one contiguous range, so every sender's values arrive in ascending position)
    m->copy_route = !(getenv("EALS_ROUTE_COPY") && getenv("EALS_ROUTE_COPY")[0] == '0');
    m->unpack_u_pending = m->unpack_i_pending = false;
    if (m->copy_route) {
      auto build_recv = [&](const Side& sd, bool by_user, uint32_t** out, size_t* cap, double* scratch_a, double* scratch_b) -> int {
        const int64_t n = sd.nnz;
        OK(dev_reserve(out, cap, (size_t)std::max<int64_t>(n, 1)));
        if (n == 0) return EALS_OK;
        uint32_t* key = reinterpret_cast<uint32_t*>(scratch_a);            // staging arrays are not live yet:
        uint32_t* key_out = key + n;                                         // 8 n bytes each
        uint32_t* val = reinterpret_cast<uint32_t*>(scratch_b);
        source_rank_kernel<<<(unsigned)((n + 255) / 256), 256, 0, m->stream>>>(sd.idx, n, rb, by_user, key, val);
        OK(check_launch(m));
        size_t tmp = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, tmp, key, key_out, val, *out, (int)n, 0, 3, m->stream);
        OK(dev_reserve(&m->route_tmp, &m->cap_route_tmp, std::max<size_t>(tmp, 16)));
        if (cub::DeviceRadixSort::SortPairs(m->route_tmp, tmp, key, key_out, val, *out, (int)n, 0, 3, m->stream) != cudaSuccess)
          return fail(EALS_ERR_CUDA, "receive-order sort");
        CU(cudaStreamSynchronize(m->stream));
        return EALS_OK;
      };
      // item columns hold USER ids (source = owner of the user); user rows hold ITEM ids
      OK(build_recv(m->items, true, &m->recv_idx_i, &m->cap_recv_idx_i, m->pc_stage_i, m->pc_i + recv_offset(ni)));
      OK(build_recv(m->users, false, &m->recv_idx_u, &m->cap_recv_idx_u, m->pc_stage_u, m->pc_u + recv_offset(nu)));
    }
    tm.lap("pred cache: routes");
  }
  m->pcache_on = true;
  if (const char* e = getenv("EALS_PRED_REFRESH_EVERY")) m->pred_refresh_every = atoi(e);
  return EALS_OK;
}

// Slab descriptors in canonical order, one thread per slab (the host only keeps per-ROW tables).
__global__ void unit_fill_kernel(const int64_t* __restrict__ ptr, const int32_t* __restrict__ hrow_id,
                                 const int32_t* __restrict__ hrow_unit0, const int64_t* __restrict__ hrow_poff,
                                 int n_hrows, int n_units, int slab, eals::UnitDesc* __restrict__ out) {
  const int u = blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= n_units) return;
  int lo = 0, hi = n_hrows;                 // largest h with hrow_unit0[h] <= u
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (hrow_unit0[mid] <= u) lo = mid; else hi = mid;
  }
  const int h = lo, r = hrow_id[h];
  const int64_t k = (int64_t)(u - hrow_unit0[h]) * slab;
  const int64_t p0 = ptr[r], n = ptr[r + 1] - p0;
  eals::UnitDesc d;
  d.off = p0 + k; d.poff = hrow_poff[h] + k;
  d.cnt = (int)(n - k < slab ? n - k : slab);
  d.row = r; d.hrow = h; d.slot = u;
  out[u] = d;
}

__global__ void unit_key_kernel(const int32_t* __restrict__ idx, const eals::UnitDesc* __restrict__ canon, int u0, int n,
                                uint32_t* __restrict__ keys, int32_t* __restrict__ vals) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  keys[t] = (uint32_t)idx[canon[u0 + t].off];
  vals[t] = u0 + t;
}

__global__ void unit_gather_kernel(const eals::UnitDesc* __restrict__ canon, const int32_t* __restrict__ sorted_ids, int n,
                                   eals::UnitDesc* __restrict__ out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) out[t] = canon[sorted_ids[t]];
}

// Launch order of every canonical batch: its slabs sorted by the id of their first neighbour.
int build_launch_order(eals_model* m, Side& s) {
  OK(dev_reserve(&s.unit_launch, &s.cap_unit_launch, (size_t)std::max(s.n_units, 1)));
  OK(dev_reserve(&s.units_launch, &s.cap_units_launch, (size_t)std::max(s.n_units, 1)));
  if (s.n_units == 0) return EALS_OK;
  OK(dev_reserve(&s.sort_keys, &s.cap_sort_keys, (size_t)s.max_batch_units));
  OK(dev_reserve(&s.sort_keys_out, &s.cap_sort_keys_out, (size_t)s.max_batch_units));
  OK(dev_reserve(&s.sort_vals, &s.cap_sort_vals, (size_t)s.max_batch_units));
  uint32_t *keys = s.sort_keys, *keys_out = s.sort_keys_out;
  int32_t* vals = s.sort_vals;
  size_t tmp_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys, keys_out, vals, s.unit_launch, s.max_batch_units, 0, 32, m->stream);
  OK(dev_reserve(&s.sort_tmp, &s.cap_sort_tmp, std::max<size_t>(tmp_bytes, 16)));
  void* tmp = s.sort_tmp;
  auto done = [&](int code) { return code; };
  for (const HeavyBatch& b : s.batches) {
    const int n = b.u1 - b.u0;
    unit_key_kernel<<<(n + 255) / 256, 256, 0, m->stream>>>(s.idx, s.units_canon, b.u0, n, keys, vals);
    if (cudaGetLastError() != cudaSuccess) return done(fail(EALS_ERR_CUDA, "unit_key_kernel launch"));
    if (cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, keys, keys_out, vals, s.unit_launch + b.u0, n, 0, 32, m->stream) != cudaSuccess)
      return done(fail(EALS_ERR_CUDA, "slab sort"));
    unit_gather_kernel<<<(n + 255) / 256, 256, 0, m->stream>>>(s.units_canon, s.unit_launch + b.u0, n, s.units_launch + b.u0);
    if (cudaGetLastError() != cudaSuccess) return done(fail(EALS_ERR_CUDA, "unit_gather_kernel launch"));
  }
  if (cudaStreamSynchronize(m->stream) != cudaSuccess) return done(fail(EALS_ERR_CUDA, "slab sort sync"));
  return done(EALS_OK);
}

// Upload the owned slice [begin, end) of one orientation of the matrix and bucket its rows.  `check` is 6 ints of
// device scratch that belong to this side alone (the validation's read-back overlaps the host bucketing).
int build_side(eals_model* m, Side& s, int begin, int end, int other_dim, int space,
               const int64_t* ptr_full, const int32_t* idx_full, const double* val_full, int* check) {
  StageTimer tm;
  s.rows = end - begin;
  s.row_base = begin;
  s.h_ptr.resize((size_t)s.rows + 1);
  if (s.rows == 0) s.h_ptr[0] = 0;
  int64_t base = 0;   // offset of the slice's first nonzero in the full index arrays
  if (s.rows > 0) {
    std::vector<int64_t> raw;
    if (space == EALS_DEVICE) {
      raw.resize((size_t)s.rows + 1);
      CU(cudaMemcpy(raw.data(), ptr_full + begin, sizeof(int64_t) * (s.rows + 1), cudaMemcpyDeviceToHost));
    }
    const int64_t* src = space == EALS_DEVICE ? raw.data() : ptr_full + begin;
    base = src[0];
    int bad_row[kMaxHostThreads];
    for (int& b : bad_row) b = -1;
    int64_t* dst = s.h_ptr.data();
    // copy + rebase + check, chunked over host threads (10M offsets: 30 ms -> a few ms)
    parallel_chunks((int64_t)s.rows + 1, nullptr, [&](int t, int64_t b0, int64_t b1) {
      for (int64_t r = b0; r < b1; r++) {
        if (r < s.rows) {
          const int64_t len = src[r + 1] - src[r];
          if ((len < 0 || len > other_dim) && bad_row[t] < 0) bad_row[t] = (int)r;
        }
        dst[r] = src[r] - base;
      }
    });
    for (int b : bad_row)
      if (b >= 0) return fail(EALS_ERR_ARG, "offsets not monotone / row longer than the other dimension at row %d", begin + b);
  }
  s.nnz = s.h_ptr[s.rows];
  tm.lap("side: offsets to host+check");

  OK(dev_reserve(&s.ptr, &s.cap_ptr, (size_t)s.rows + 1));
  OK(dev_reserve(&s.idx, &s.cap_idx, (size_t)s.nnz));
  CU(cudaMemcpyAsync(s.ptr, s.h_ptr.data(), sizeof(int64_t) * (s.rows + 1), cudaMemcpyHostToDevice, m->stream));
  OK(copy_in(s.idx, idx_full + base, (size_t)s.nnz, space, m->stream));
  if (val_full) {
    OK(dev_reserve(&s.val, &s.cap_val, (size_t)s.nnz));
    OK(copy_in(s.val, val_full + base, (size_t)s.nnz, space, m->stream));
  } else if (s.val) {
    cudaFree(s.val);
    s.val = nullptr;
    s.cap_val = 0;
  }

  tm.lap("side: alloc + copy indices");
  // indices must ascend strictly inside a row and stay in range (main.cpp:198-205 order)
  int* sorted_flag = nullptr;
  if (s.rows > 0) {
    int* bad = check;                                          // 6 ints: bad, pad, descents (u64), row-start descents (u64)
    unsigned long long* counts = reinterpret_cast<unsigned long long*>(bad + 2);
    CU(cudaMemsetAsync(bad, 0, 6 * sizeof(int), m->stream));
    if (s.nnz > 0) {
      check_indices_kernel<<<(unsigned)((s.nnz + 255) / 256), 256, 0, m->stream>>>(s.idx, s.nnz, other_dim, bad, counts);
      OK(check_launch(m));
    }
    check_row_starts_kernel<<<(s.rows + 255) / 256, 256, 0, m->stream>>>(s.ptr, s.idx, s.rows, counts + 1);
    OK(check_launch(m));
    sorted_flag = bad;   // read back after the host-side bucketing below (overlaps the upload)
  }

  tm.lap("side: validate sorted (enqueued)");
  // counting sort of the rows into length buckets
  std::vector<int32_t> order((size_t)std::max(s.rows, 1));
  int count[kNumBuckets] = {0};
  constexpr int kLut = kBucketMax[kHeavyBucket - 1] + 2;        // lengths 0..512 by table, longer = heavy
  uint8_t lut[kLut];
  for (int n = 0, b = 0; n < kLut; n++) {
    while (n > kBucketMax[b]) b++;
    lut[n] = (uint8_t)b;
  }
  // EALS_HEAVY_MIN: rows longer than this go to the slab pipeline (default: the last team bucket's limit)
  const int heavy_min = getenv("EALS_HEAVY_MIN") ? std::max(32, atoi(getenv("EALS_HEAVY_MIN"))) : kBucketMax[kHeavyBucket - 1];
  for (int n = 0; n < kLut; n++)
    if (n > heavy_min) lut[n] = (uint8_t)kHeavyBucket;
  std::vector<uint8_t> bucket((size_t)std::max(s.rows, 1));
  {
    // stable counting sort, chunked over host threads: per-chunk histograms, then per-chunk bases
    int T = 1;
    int cnt_t[kMaxHostThreads][kNumBuckets];
    for (auto& c : cnt_t) for (int& v : c) v = 0;
    const int64_t* hp = s.h_ptr.data();
    parallel_chunks(s.rows, &T, [&](int t, int64_t b0, int64_t b1) {
      int local[kNumBuckets] = {0};
      for (int64_t r = b0; r < b1; r++) {
        const int64_t n = hp[r + 1] - hp[r];
        const uint8_t b = lut[std::min<int64_t>(n, kLut - 1)];
        bucket[r] = b;
        local[b]++;
      }
      for (int b = 0; b < kNumBuckets; b++) cnt_t[t][b] = local[b];
    });
    for (int b = 0; b < kNumBuckets; b++)
      for (int t = 0; t < T; t++) count[b] += cnt_t[t][b];
    s.first[0] = 0;
    for (int b = 0; b < kNumBuckets; b++) s.first[b + 1] = s.first[b] + count[b];
    int base_t[kMaxHostThreads][kNumBuckets];
    for (int b = 0; b < kNumBuckets; b++) {
      int at = s.first[b];
      for (int t = 0; t < T; t++) { base_t[t][b] = at; at += cnt_t[t][b]; }
    }
    int T2 = 1;
    parallel_chunks(s.rows, &T2, [&](int t, int64_t b0, int64_t b1) {
      int fill[kNumBuckets];
      for (int b = 0; b < kNumBuckets; b++) fill[b] = base_t[t][b];
      for (int64_t r = b0; r < b1; r++) order[fill[bucket[r]]++] = (int32_t)r;
    });
  }
  // long rows: longest first, so the tail of the launch is made of the cheapest rows
  std::stable_sort(order.begin() + s.first[kHeavyBucket], order.begin() + s.first[kHeavyBucket + 1],
                   [&](int a, int b) {
                     return s.h_ptr[a + 1] - s.h_ptr[a] > s.h_ptr[b + 1] - s.h_ptr[b];
                   });
  OK(dev_reserve(&s.order, &s.cap_order, order.size()));
  CU(cudaMemcpyAsync(s.order, order.data(), sizeof(int32_t) * order.size(), cudaMemcpyHostToDevice, m->stream));

  if (sorted_flag) {
    int h_flags[6] = {0, 0, 0, 0, 0, 0};
    CU(cudaMemcpyAsync(h_flags, sorted_flag, sizeof(h_flags), cudaMemcpyDeviceToHost, m->stream));
    CU(cudaStreamSynchronize(m->stream));
    unsigned long long h_counts[2];
    std::memcpy(h_counts, h_flags + 2, sizeof(h_counts));
    if (h_flags[0] || h_counts[0] != h_counts[1])
      return fail(EALS_ERR_ARG, "indices inside a row must be strictly ascending and in range");
  }
  tm.lap("side: bucket rows + validate");
  // heavy rows -> slabs ("units") of kSlab nonzeros and batches of rows
  {
    const int hb = s.first[kHeavyBucket], he = s.first[kHeavyBucket + 1];
    s.n_hrows = he - hb;
    std::vector<int32_t> hrow_id, grp_unit0, grp_cnt;
    std::vector<int64_t> hrow_poff;
    int64_t n_units_total = 0;
    // EALS_SLAB=128|256: nonzeros per slab = threads per heavy_step CTA
    s.slab = (getenv("EALS_SLAB") && atoi(getenv("EALS_SLAB")) == 256) ? 256 : 128;
    s.h_hrow_unit0.clear(); s.h_hrow_units.clear(); s.batches.clear(); s.h_row_to_hrow.clear();
    s.h_hrow_grp0.clear(); s.h_hrow_grps.clear();
    {
      int64_t hn = 0;
      for (int h = 0; h < s.n_hrows; h++) { const int r = order[hb + h]; hn += s.h_ptr[r + 1] - s.h_ptr[r]; }
      (void)hn;
      hrow_poff.reserve((size_t)s.n_hrows);
      hrow_id.reserve((size_t)s.n_hrows); s.h_hrow_unit0.reserve((size_t)s.n_hrows); s.h_hrow_units.reserve((size_t)s.n_hrows);
    }
    int64_t poff = 0, batch_nnz = 0;
    int64_t batch_limit = kDefaultBatchNnz;
    if (const char* e = getenv("EALS_HEAVY_BATCH_NNZ")) batch_limit = std::max<int64_t>(atoll(e), 1);
    if (s.n_hrows) s.h_row_to_hrow.assign((size_t)s.rows, -1);
    HeavyBatch cur{0, 0, 0, 0};
    for (int h = 0; h < s.n_hrows; h++) {
      const int r = order[hb + h];
      const int64_t n = s.h_ptr[r + 1] - s.h_ptr[r];
      if (h > cur.h0 && batch_nnz + n > batch_limit) {
        cur.h1 = h; cur.u1 = (int)n_units_total;
        s.batches.push_back(cur);
        cur = HeavyBatch{h, h, cur.u1, cur.u1};
        batch_nnz = 0;
      }
      batch_nnz += n;
      s.h_row_to_hrow[r] = h;
      hrow_id.push_back(r);
      s.h_hrow_unit0.push_back((int)n_units_total);
      hrow_poff.push_back(poff);
      const int nunits = (int)((n + s.slab - 1) / s.slab);
      n_units_total += nunits;
      if (n_units_total >= 0x7fffffffLL) return fail(EALS_ERR_UNSUPPORTED, "too many slabs of heavy rows");
      s.h_hrow_units.push_back(nunits);
      s.h_hrow_grp0.push_back((int)grp_unit0.size());
      s.h_hrow_grps.push_back((nunits + 31) / 32);
      for (int q = 0; q < nunits; q += 32) {
        grp_unit0.push_back(s.h_hrow_unit0.back() + q);
        grp_cnt.push_back(std::min(32, nunits - q));
      }
      poff += n;
    }
    if (s.n_hrows) {
      cur.h1 = s.n_hrows; cur.u1 = (int)n_units_total;
      s.batches.push_back(cur);
    }
    s.n_units = (int)n_units_total;
    s.heavy_nnz = poff;
    s.max_batch_units = 0;
    for (const auto& b : s.batches) s.max_batch_units = std::max(s.max_batch_units, b.u1 - b.u0);
    auto up32 = [&](int32_t** d, size_t* cap, const std::vector<int32_t>& v) -> int {
      OK(dev_reserve(d, cap, v.size()));
      if (!v.empty()) CU(cudaMemcpyAsync(*d, v.data(), sizeof(int32_t) * v.size(), cudaMemcpyHostToDevice, m->stream));
      return EALS_OK;
    };
    OK(dev_reserve(&s.units_canon, &s.cap_units_canon, std::max<size_t>((size_t)s.n_units, 1)));
    OK(up32(&s.hrow_id, &s.cap_hrow_id, hrow_id)); OK(up32(&s.hrow_unit0, &s.cap_hrow_unit0, s.h_hrow_unit0));
    OK(dev_reserve(&s.hrow_poff, &s.cap_hrow_poff, std::max<size_t>(hrow_poff.size(), 1)));
    if (s.n_units > 0) {
      CU(cudaMemcpyAsync(s.hrow_poff, hrow_poff.data(), sizeof(int64_t) * hrow_poff.size(), cudaMemcpyHostToDevice, m->stream));
      unit_fill_kernel<<<(s.n_units + 255) / 256, 256, 0, m->stream>>>(s.ptr, s.hrow_id, s.hrow_unit0, s.hrow_poff,
                                                                       s.n_hrows, s.n_units, s.slab, s.units_canon);
      OK(check_launch(m));
    }
    OK(up32(&s.hrow_units, &s.cap_hrow_units, s.h_hrow_units));
    OK(up32(&s.hrow_grp0, &s.cap_hrow_grp0, s.h_hrow_grp0)); OK(up32(&s.hrow_grps, &s.cap_hrow_grps, s.h_hrow_grps));
    OK(up32(&s.grp_unit0, &s.cap_grp_unit0, grp_unit0)); OK(up32(&s.grp_cnt, &s.cap_grp_cnt, grp_cnt));
    s.n_groups = (int)grp_unit0.size();
    OK(build_launch_order(m, s));
    OK(dev_reserve(&s.pred, &s.cap_pred, (size_t)s.heavy_nnz));
    OK(dev_reserve(&s.delta, &s.cap_delta, (size_t)s.n_hrows * 16));
    CU(cudaStreamSynchronize(m->stream));   // the host vectors above go out of scope
    // size the partials scratch now: a reallocation in the middle of a sweep would synchronise
    {
      int max_groups = 0;
      for (const auto& b : s.batches)
        max_groups = std::max(max_groups, s.h_hrow_grp0[b.h1 - 1] + s.h_hrow_grps[b.h1 - 1] - s.h_hrow_grp0[b.h0]);
      OK(ensure_partials(m, (size_t)(s.max_batch_units + max_groups + 2) * eals::kPartLen));
    }
  }
  tm.lap("side: heavy units + upload");
  CU(cudaStreamSynchronize(m->stream));
  return EALS_OK;
}

// ---- the reference's factor initialisation, in parallel, bit for bit ---------------------------------------
// DenseMat::init (DenseMat.cpp:54-62) draws rows*cols values from std::normal_distribution<double> over a
// default-constructed std::default_random_engine = minstd_rand0 (x' = 16807 x mod 2^31-1, seed 1).  libstdc++'s
// normal_distribution is Marsaglia's polar method (random.tcc:1811-1847): an ATTEMPT draws two uniforms
// (generate_canonical<double,53> = two engine draws each, random.tcc:3349-3381), is rejected unless
// 0 < x^2 + y^2 <= 1, and an accepted attempt yields two values (y*mult first, x*mult on the next call).  Every
// attempt consumes exactly four engine draws whether accepted or not, so attempt j starts at stream position
// 4j — reachable directly, the LCG has an O(log n) skip-ahead (a^n mod m).  The attempt stream is cut into
// chunks; pass 1 counts the accepted attempts of every chunk (the same two generate_canonical calls and the same
// test, no log / sqrt), a prefix sum gives every chunk its output offset, pass 2 runs the REAL
// std::normal_distribution over an engine positioned at the chunk's first attempt for exactly the counted number
// of values.  Same libm, same instantiations as the sequential loop — same bits (tested against the oracle),
// seconds instead of tens of seconds at 10M x 128.
uint64_t minstd0_state_after(uint64_t draws) {
  const uint64_t mod = 2147483647ull;
  uint64_t result = 1, base = 16807ull;      // seed 1 (random.h:1592-1593, 1641)
  while (draws) {
    if (draws & 1) result = result * base % mod;
    base = base * base % mod;
    draws >>= 1;
  }
  return result;                              // = 16807^draws mod m: the engine state after `draws` draws from seed 1
}

void init_stream(double mean, double stdev, double* out, size_t n) {
  size_t chunk = 1 << 16;                     // attempts per chunk
  if (const char* e = getenv("EALS_INIT_CHUNK")) chunk = std::max<size_t>(8, strtoull(e, nullptr, 10));
  const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
  const size_t T = std::min<size_t>(hw, 32);
  size_t produced = 0, first_chunk = 0;
  while (produced < n) {
    // a wave of chunks that will almost surely cover what is left (acceptance rate pi/4), at least one per thread
    const size_t left_attempts = (size_t)((double)(n - produced) / 2.0 / 0.78) + 64;
    const size_t wave = std::max<size_t>(1, std::min<size_t>((left_attempts + chunk - 1) / chunk, T * 64));
    std::vector<size_t> acc(wave, 0);
    auto over_chunks = [&](auto fn) {
      std::vector<std::thread> th;
      const size_t nt = std::min(T, wave);
      for (size_t t = 0; t < nt; t++)
        th.emplace_back([&, t] { for (size_t c = t; c < wave; c += nt) fn(c); });
      for (auto& x : th) x.join();
    };
    over_chunks([&](size_t c) {               // pass 1: accepted attempts of chunk c
      std::minstd_rand0 eng((std::minstd_rand0::result_type)minstd0_state_after(4 * (first_chunk + c) * (uint64_t)chunk));
      size_t a = 0;
      for (size_t j = 0; j < chunk; j++) {
        const double x = 2.0 * std::generate_canonical<double, std::numeric_limits<double>::digits>(eng) - 1.0;
        const double y = 2.0 * std::generate_canonical<double, std::numeric_limits<double>::digits>(eng) - 1.0;
        const double r2 = x * x + y * y;
        a += !(r2 > 1.0 || r2 == 0.0);
      }
      acc[c] = a;
    });
    std::vector<size_t> off(wave + 1, produced);
    for (size_t c = 0; c < wave; c++) off[c + 1] = off[c] + 2 * acc[c];
    over_chunks([&](size_t c) {               // pass 2: the real distribution over the chunk's own engine
      if (off[c] >= n) return;
      std::minstd_rand0 eng((std::minstd_rand0::result_type)minstd0_state_after(4 * (first_chunk + c) * (uint64_t)chunk));
      std::normal_distribution<double> distribution(mean, stdev);
      const size_t end = std::min(n, off[c + 1]);
      for (size_t t = off[c]; t < end; t++) out[t] = distribution(eng);
    });
    produced = std::min(n, off[wave]);
    first_chunk += wave;
  }
}

// Wi — MF_fastALS.cpp:55-72, on the host with the same libm pow and the same summation order.
int compute_item_weights(eals_model* m, int space, const int64_t* col_ptr_full) {
  const int N = m->N;
  std::vector<int64_t> cp((size_t)N + 1);
  if (space == EALS_DEVICE) {
    CU(cudaMemcpy(cp.data(), col_ptr_full, sizeof(int64_t) * (N + 1), cudaMemcpyDeviceToHost));
  } else {
    std::memcpy(cp.data(), col_ptr_full, sizeof(int64_t) * (N + 1));
  }
  std::vector<double> p((size_t)N);
  double sum = 0, Z = 0;
  for (int i = 0; i < N; i++) {
    p[i] = (double)(int)(cp[i + 1] - cp[i]);
    sum += p[i];
  }
  for (int i = 0; i < N; i++) {
    p[i] /= sum;
    p[i] = pow(p[i], m->p.alpha);
    Z += p[i];
  }
  for (int i = 0; i < N; i++) p[i] = m->p.w0 * p[i] / Z;
  CU(cudaMemcpyAsync(m->Wi, p.data(), sizeof(double) * N, cudaMemcpyHostToDevice, m->stream));
  CU(cudaStreamSynchronize(m->stream));
  return EALS_OK;
}

int ensure_partials(eals_model* m, size_t n) {
  if (n <= m->partials_len) return EALS_OK;
  if (m->capturing) return fail(EALS_ERR_STATE, "scratch would have to grow inside a captured epoch");
  cudaFree(m->partials);
  m->partials = nullptr;
  m->partials_len = 0;
  OK(dev_alloc(&m->partials, n));
  m->partials_len = n;
  return EALS_OK;
}

cudaEvent_t take_event(eals_model* m) {
  cudaEvent_t e = nullptr;
  if (!m->pool.empty()) { e = m->pool.back(); m->pool.pop_back(); }
  else cudaEventCreate(&e);
  return e;
}

// Fold finished event pairs into the accumulators (caller has synchronised the stream).
void fold_timings(eals_model* m) {
  for (int t = 0; t < T_COUNT; t++) {
    for (auto& pr : m->pending[t]) {
      float f = 0;
      if (pr.second && cudaEventElapsedTime(&f, pr.first, pr.second) == cudaSuccess) {
        m->acc_ms[t] += f;
        m->acc_calls[t]++;
        m->last_ms[t] = f;
      }
      m->pool.push_back(pr.first);
      if (pr.second) m->pool.push_back(pr.second);
    }
    m->pending[t].clear();
  }
}

void tic(eals_model* m, int which) {
  if (m->capturing) return;      // no timing events inside a captured epoch
  if (m->pending[which].size() >= 2048) { cudaStreamSynchronize(m->stream); fold_timings(m); }
  cudaEvent_t e = take_event(m);
  cudaEventRecord(e, m->stream);
  m->pending[which].emplace_back(e, nullptr);
}
void toc(eals_model* m, int which) {
  if (m->capturing) return;
  cudaEvent_t e = take_event(m);
  cudaEventRecord(e, m->stream);
  m->pending[which].back().second = e;
}

// ---- dispatch on the leading dimension (16, 32, 64, 128, 256) ---------------------------------
#define DISPATCH_LD(LDV, ...)                                              \
  switch (LDV) {                                                           \
    case 16: { constexpr int LD = 16; __VA_ARGS__; } break;                \
    case 32: { constexpr int LD = 32; __VA_ARGS__; } break;                \
    case 64: { constexpr int LD = 64; __VA_ARGS__; } break;                \
    case 128: { constexpr int LD = 128; __VA_ARGS__; } break;              \
    case 256: { constexpr int LD = 256; __VA_ARGS__; } break;              \
    default: return fail(EALS_ERR_UNSUPPORTED, "leading dimension %d", LDV); \
  }

template <int LD, int MAXM, bool USER>
int launch_cd_warp_block(eals_model* m, const CdSide& a, const int32_t* order, int first, int count) {
  if (count <= 0) return EALS_OK;
  using Sm = eals::WarpBlockSmem<LD, MAXM>;
  // persistent CTAs, one per SM: S cache + as many row-warps as fit the 227 KB of shared memory
  const size_t budget = 227 * 1024 - Sm::kS;
  int wpb = (int)std::min<size_t>(Sm::kMaxWarps, std::max<size_t>(1, budget / Sm::kBytesPerWarp));
  static int env_wpb = getenv("EALS_WARP_WPB") ? atoi(getenv("EALS_WARP_WPB")) : 0;
  if (env_wpb > 0) wpb = std::min(env_wpb, wpb);
  const size_t smem = Sm::kS + Sm::kBytesPerWarp * wpb;
  auto kern = eals::cd_warp_block_kernel<LD, MAXM, USER>;
  CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int grid = std::min((count + wpb - 1) / wpb, m->sm_count);
  kern<<<grid, wpb * 32, smem, m->stream>>>(a, order, first, count);
  return check_launch(m);
}

template <int LD, int TW, int MW, bool USER>
int launch_cd_row_block(eals_model* m, const CdSide& a, const int32_t* order, int first, int count) {
  if (count <= 0) return EALS_OK;
  using Sm = eals::RowBlockSmem<LD, TW, MW>;
  auto kern = eals::cd_row_block_kernel<LD, TW, MW, USER>;
  CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Sm::kBytes));
  kern<<<count, TW * 32, Sm::kBytes, m->stream>>>(a, order, first);
  return check_launch(m);
}

eals::HeavyUnits heavy_units(const Side& s) {
  eals::HeavyUnits hu;
  hu.units = nullptr;
  hu.hrow_id = s.hrow_id;
  hu.hrow_grp0 = s.hrow_grp0; hu.hrow_grps = s.hrow_grps; hu.grp_unit0 = s.grp_unit0; hu.grp_cnt = s.grp_cnt;
  return hu;
}

// One batch of heavy rows: prediction cache, then per factor block a partials launch (which also
// applies the previous block's cache update) and a solve launch.
template <int LD, bool USER>
int run_heavy_batch(eals_model* m, Side& s, const CdSide& a, const HeavyBatch& b, bool canonical) {
  const int nu = b.u1 - b.u0, nh = b.h1 - b.h0;
  if (nu <= 0) return EALS_OK;
  eals::HeavyUnits hu = heavy_units(s);
  const bool no_order = getenv("EALS_HEAVY_ORDER") && getenv("EALS_HEAVY_ORDER")[0] == '0';   // A/B runs and tests
  hu.units = ((canonical && !no_order) ? s.units_launch : s.units_canon) + b.u0;   // neighbour order for whole batches
  const int nblocks = (m->K + eals::kFB - 1) / eals::kFB;
  // group sums (one per <= 32 consecutive units of a row) live behind the unit partials
  const int g0 = s.h_hrow_grp0[b.h0];
  const int ngroups = s.h_hrow_grp0[b.h1 - 1] + s.h_hrow_grps[b.h1 - 1] - g0;
  OK(ensure_partials(m, (size_t)(nu + ngroups) * eals::kPartLen));
  double* part = m->partials;
  double* part2 = m->partials + (size_t)nu * eals::kPartLen;
  auto step = s.slab == 256 ? eals::heavy_step_kernel<LD, USER, 256> : eals::heavy_step_kernel<LD, USER, 128>;
  const int step_smem = (int)(s.slab == 256 ? eals::HeavySmem<256>::kBytes : eals::HeavySmem<128>::kBytes);
  CU(cudaFuncSetAttribute(step, cudaFuncAttributeMaxDynamicSharedMemorySize, step_smem));
  if (!a.use_cache) {
    eals::heavy_pred_kernel<LD><<<nu, eals::kBlkThreads, 0, m->stream>>>(a, hu, s.pred);
    OK(check_launch(m));
  }
  for (int fb = 0; fb <= nblocks; fb++) {
    if (fb == nblocks && !a.pc_out.n) break;   // last cache update: only when the symmetric cache keeps the result
    step<<<nu, s.slab, step_smem, m->stream>>>(a, hu, b.u0, fb, nblocks, s.pred, s.delta, part);
    OK(check_launch(m));
    if (fb == nblocks) break;
    eals::heavy_reduce_kernel<<<ngroups, eals::kBlkThreads, 0, m->stream>>>(part, hu, g0, b.u0, part2);
    OK(check_launch(m));
    eals::heavy_solve_kernel<LD, USER><<<nh, eals::kBlkThreads, 0, m->stream>>>(a, hu, b.h0, g0, fb, part2, s.delta);
    OK(check_launch(m));
  }
  return EALS_OK;
}

// timed: the whole-side launches go to the sweep sub-phase timers (eals_timings_detail); fold-in runs the same
// kernels untimed, so the timers keep reporting training sweeps only.
template <int LD, bool USER>
int launch_cd(eals_model* m, Side& s, const CdSide& a, int only_row, bool timed) {
  if (only_row >= 0) {  // single-row API: a one-entry order list in scratch
    const int64_t n = s.h_ptr[only_row + 1] - s.h_ptr[only_row];
    if (n == 0) return EALS_OK;
    if (!s.h_row_to_hrow.empty() && s.h_row_to_hrow[only_row] >= 0) {
      const int h = s.h_row_to_hrow[only_row];
      return run_heavy_batch<LD, USER>(m, s, a, HeavyBatch{h, h + 1, s.h_hrow_unit0[h], s.h_hrow_unit0[h] + s.h_hrow_units[h]}, false);
    }
    OK(ensure_partials(m, 16));
    int32_t* one = reinterpret_cast<int32_t*>(m->partials);
    CU(cudaMemcpyAsync(one, &only_row, sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
    if (n <= 32) return launch_cd_warp_block<LD, 1, USER>(m, a, one, 0, 1);
    if (n <= 64) return launch_cd_warp_block<LD, 2, USER>(m, a, one, 0, 1);
    if (n <= 96) return launch_cd_warp_block<LD, 3, USER>(m, a, one, 0, 1);
    if (n <= 128) return launch_cd_warp_block<LD, 4, USER>(m, a, one, 0, 1);
    if (n <= 256) return launch_cd_row_block<LD, 4, 2, USER>(m, a, one, 0, 1);
    if (n <= 384) return launch_cd_row_block<LD, 4, 3, USER>(m, a, one, 0, 1);
    return launch_cd_row_block<LD, 8, 2, USER>(m, a, one, 0, 1);
  }
  // heavy rows first: their launch chain is the longest
  const int t0 = USER ? T_U_HEAVY : T_I_HEAVY;
  if (timed) tic(m, t0);
  for (const HeavyBatch& b : s.batches) OK((run_heavy_batch<LD, USER>(m, s, a, b, true)));
  if (timed) { toc(m, t0); tic(m, t0 + 1); }
  OK((launch_cd_row_block<LD, 8, 2, USER>(m, a, s.order, s.first[7], s.first[8] - s.first[7])));   // 385..512
  OK((launch_cd_row_block<LD, 4, 3, USER>(m, a, s.order, s.first[6], s.first[7] - s.first[6])));   // 257..384
  OK((launch_cd_row_block<LD, 4, 2, USER>(m, a, s.order, s.first[5], s.first[6] - s.first[5])));   // 129..256
  if (timed) { toc(m, t0 + 1); tic(m, t0 + 2); }
  // one warp per row up to 128 nonzeros: no CTA barrier anywhere in the row loop
  OK((launch_cd_warp_block<LD, 4, USER>(m, a, s.order, s.first[4], s.first[5] - s.first[4])));
  OK((launch_cd_warp_block<LD, 3, USER>(m, a, s.order, s.first[3], s.first[4] - s.first[3])));
  OK((launch_cd_warp_block<LD, 2, USER>(m, a, s.order, s.first[2], s.first[3] - s.first[2])));
  OK((launch_cd_warp_block<LD, 1, USER>(m, a, s.order, s.first[1], s.first[2] - s.first[1])));
  if (timed) toc(m, t0 + 2);
  return EALS_OK;
}

// Launch the routing copy the last sweep left behind: on the side stream (after the sweep's kernels), or on the
// model's own stream.
int launch_route(eals_model* m, bool on_side_stream) {
  if (!m->route_todo) return EALS_OK;
  const bool user = m->route_todo == 1;
  m->route_todo = 0;
  static const bool inline_route = getenv("EALS_ROUTE_INLINE") && getenv("EALS_ROUTE_INLINE")[0] == '1';
  const Side& s = user ? m->users : m->items;
  const eals::PcOut& out = user ? m->out_to_items : m->out_to_users;
  cudaStream_t rs = m->stream;
  if (on_side_stream && !inline_route) {
    CU(cudaStreamWaitEvent(m->side_stream, m->ev_swept, 0));
    rs = m->side_stream;
  }
  if (m->copy_route) {
    // One peer-to-peer copy per destination rank (copy engines: no SM, runs under the Gram kernel): my segment of
    // the destination-ordered staging array -> my slot of the destination's receive area.
    const int me = m->rank, nr = m->n_ranks;
    const double* stage = user ? m->pc_stage_u : m->pc_stage_i;
    // side stream + two helpers (round-robin over the destinations) when the copies run beside the Gram
    cudaStream_t lanes[3] = {rs, rs, rs};
    static const bool no_fan = getenv("EALS_COPY_FAN") && getenv("EALS_COPY_FAN")[0] == '0';
    const bool fan = rs != m->stream && nr > 2 && !no_fan;
    if (fan) {
      for (int c = 0; c < 2; c++) {
        if (!m->copy_stream[c]) {
          CU(cudaStreamCreateWithFlags(&m->copy_stream[c], cudaStreamNonBlocking));
          CU(cudaEventCreateWithFlags(&m->ev_copied[c], cudaEventDisableTiming));
        }
        CU(cudaStreamWaitEvent(m->copy_stream[c], m->ev_swept, 0));
        lanes[c + 1] = m->copy_stream[c];
      }
    }
    int n_copy = 0;
    long long seg = 0;
    for (int r = 0; r < nr; r++) {
      // user sweep: I am the user-owner `me`, destination = item-owner r; item sweep: I am the item-owner, dest = user-owner r
      const long long cnt = user ? m->pair_cnt[me][r] : m->pair_cnt[r][me];
      long long off = 0;                                       // senders before me in r's receive area
      for (int q = 0; q < me; q++) off += user ? m->pair_cnt[q][r] : m->pair_cnt[r][q];
      const long long dst_n = (long long)out.bound[r + 1] - (long long)out.bound[r];   // values in r's cache
      if (cnt > 0 && r != me)      // my own segment stays where it is: pc_unpack_kernel reads it from the staging array
        CU(cudaMemcpyAsync(out.base[r] + recv_offset(dst_n) + off, stage + seg, sizeof(double) * (size_t)cnt, cudaMemcpyDefault,
                           lanes[n_copy++ % 3]));
      seg += cnt;
    }
    if (fan)                       // the helpers rejoin the side stream: ev_routed below covers all copies
      for (int c = 0; c < 2; c++) {
        CU(cudaEventRecord(m->ev_copied[c], m->copy_stream[c]));
        CU(cudaStreamWaitEvent(m->side_stream, m->ev_copied[c], 0));
      }
    if (seg != s.nnz) return fail(EALS_ERR_STATE, "routing table does not cover the staged predictions (%lld of %lld)", seg, (long long)s.nnz);
    (user ? m->unpack_i_pending : m->unpack_u_pending) = true;      // SPMD: every rank sweeps the same side now
  } else {
    const int grid = (int)std::min<int64_t>((s.nnz + 255) / 256, 4 * m->sm_count);
    eals::pc_route_kernel<<<grid, 256, 0, rs>>>(user ? m->pc_stage_u : m->pc_stage_i, user ? m->route_dst_u : m->route_dst_i, s.nnz, out);
    OK(check_launch(m));
  }
  if (rs != m->stream) {
    CU(cudaEventRecord(m->ev_routed, m->side_stream));
    m->route_pending = true;
  }
  return EALS_OK;
}

// The routing copy of the previous sweep must be complete (in stream order) before anything that follows on
// the model's stream is allowed to mean "this half-epoch is done".
int join_route(eals_model* m) {
  OK(launch_route(m, false));
  if (m->route_pending) {
    CU(cudaStreamWaitEvent(m->stream, m->ev_routed, 0));
    m->route_pending = false;
  }
  return EALS_OK;
}

// Receive areas filled by the other ranks' copies (complete once the all-reduce after their sweep has completed,
// which the host layer issues between the half-epochs) -> the prediction caches.
int unpack_pending(eals_model* m) {
  for (int side = 0; side < 2; side++) {
    bool& pend = side == 0 ? m->unpack_u_pending : m->unpack_i_pending;
    if (!pend) continue;
    pend = false;
    const bool valid = side == 0 ? m->pc_u_valid : m->pc_i_valid;
    const int64_t n = side == 0 ? m->users.nnz : m->items.nnz;
    if (!valid || n == 0) continue;
    double* cache = side == 0 ? m->pc_u : m->pc_i;
    // my own segment: slot range in the receive order, and where it sits in the staging array of the side that sent it
    const int me = m->rank;
    long long lo = 0, src_off = 0;
    for (int q = 0; q < me; q++) {
      lo += side == 0 ? m->pair_cnt[me][q] : m->pair_cnt[q][me];        // senders before me in MY receive area
      src_off += side == 0 ? m->pair_cnt[q][me] : m->pair_cnt[me][q];   // destinations before me in MY staging array
    }
    const long long cnt = m->pair_cnt[me][me];
    const double* local_src = (side == 0 ? m->pc_stage_i : m->pc_stage_u) + src_off;   // pc_u is fed by the ITEM sweep's staging
    const int grid = (int)std::min<int64_t>((n + 255) / 256, 8 * m->sm_count);
    pc_unpack_kernel<<<grid, 256, 0, m->stream>>>(cache + recv_offset(n), side == 0 ? m->recv_idx_u : m->recv_idx_i, n, cache,
                                                  local_src, lo, lo + cnt);
    OK(check_launch(m));
  }
  return EALS_OK;
}

int sweep(eals_model* m, bool user, int only_row) {
  if (!m->factors_set) return fail(EALS_ERR_STATE, "factors not initialised (eals_init_factors / eals_set_factors)");
  OK(join_route(m));
  OK(unpack_pending(m));
  Side& s = user ? m->users : m->items;
  CdSide a;
  a.ptr = s.ptr; a.idx = s.idx; a.val = s.val;
  a.X = user ? m->U : m->V;
  a.Y = user ? m->V : m->U;
  a.S = user ? m->SV : m->SU;
  a.Wi = m->Wi;
  a.row_base = s.row_base;
  a.K = m->K;
  a.reg = m->p.reg;
  a.pc_in = nullptr; a.pc_map = nullptr; a.pc_out = eals::PcOut{}; a.use_cache = 0; a.pc_stage = nullptr;
  a.peers = user ? m->peersU : m->peersV;
  static const bool fence = getenv("EALS_PEER_FENCE") && getenv("EALS_PEER_FENCE")[0] == '1';
  a.fence = fence ? 1 : 0;   // off by default: grid completion already orders the peer stores (cd_sweep.cuh, peers_release)
  if (only_row >= 0) {
    m->pc_u_valid = m->pc_i_valid = false;   // a single-row update changes factors behind the cache's back
    if (user) m->su_fresh = false;           // ... and U behind SU's back (MF_fastALS.cpp:243-322 never touches SU)
  } else if (m->pcache_on && m->pc_attached) {
    bool& in_valid = user ? m->pc_u_valid : m->pc_i_valid;
    bool& out_valid = user ? m->pc_i_valid : m->pc_u_valid;
    if (m->pred_refresh_every > 0 && m->sweeps_since_fresh >= m->pred_refresh_every) in_valid = false;
    a.pc_in = user ? m->pc_u : m->pc_i;
    a.pc_map = user ? m->map_u : m->map_i;
    a.pc_out = user ? m->out_to_items : m->out_to_users;
    if (m->routed) {     // staged: the map is the slot in destination order (build_routes)
      a.pc_stage = user ? m->pc_stage_u : m->pc_stage_i;
      a.pc_map = user ? m->route_src_u : m->route_src_i;
    }
    a.use_cache = in_valid ? 1 : 0;
    m->sweeps_since_fresh = in_valid ? m->sweeps_since_fresh + 1 : 0;
    in_valid = false;    // this side's cache describes the factors BEFORE this sweep
    out_valid = true;    // every nonzero's final prediction is stored on the other side by this sweep
  }
  if (user) { DISPATCH_LD(m->LD, OK((launch_cd<LD, true>(m, s, a, only_row, true)))); }
  else      { DISPATCH_LD(m->LD, OK((launch_cd<LD, false>(m, s, a, only_row, true)))); }
  if (a.pc_stage && s.nnz > 0) {
    // Second phase: staged predictions to their owners, in destination order.  Nobody needs them before the
    // NEXT half-epoch's sweep, so the copy is launched by gram() on a side stream right behind the Gram's main
    // kernel (a small persistent grid that shares the SMs with it) and joined before gram() returns — i.e.
    // before the all-reduce that orders the ranks.  Round 1 had it on the sweep's stream: 7 % of the step at
    // 2 GPUs.  A caller that never calls gram() gets it inline at the next sweep / sync (join_route).
    if (!m->side_stream) {
      CU(cudaStreamCreateWithFlags(&m->side_stream, cudaStreamNonBlocking));
      CU(cudaEventCreateWithFlags(&m->ev_swept, cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&m->ev_routed, cudaEventDisableTiming));
    }
    CU(cudaEventRecord(m->ev_swept, m->stream));
    m->route_todo = user ? 1 : 2;
  }
  return sync_if_debug(m);
}

template <int LD>
int launch_gram(eals_model* m, const double* X, const double* w, int r0, int r1, double* S) {
  using C = eals::GramCfg<LD>;
  int nslabs = std::max(1, std::min(2 * m->sm_count, (r1 - r0 + 127) / 128));
  OK(ensure_partials(m, (size_t)C::NPAIR * nslabs * C::TB * C::TB));
  // diagonal block pairs (all of them for K <= 128): lower-triangular tiles only; LD = 256 adds the full (1, 0) block
  eals::gram_partial_kernel<LD, true><<<dim3(nslabs, C::NB), eals::kGramThreads, 0, m->stream>>>(X, w, r0, r1, m->partials, 0, 2);
  OK(check_launch(m));
  if (C::NB == 2) {
    eals::gram_partial_kernel<LD, false><<<dim3(nslabs, 1), eals::kGramThreads, 0, m->stream>>>(X, w, r0, r1, m->partials, 1, 1);
    OK(check_launch(m));
  }
  OK(launch_route(m, true));     // the pending prediction-cache routing shares the SMs with the kernel above
  const int total = C::NPAIR * C::TB * C::TB;
  eals::gram_reduce_kernel<LD><<<(total + 255) / 256, 256, 0, m->stream>>>(m->partials, nslabs, m->K, S);
  return check_launch(m);
}

int gram(eals_model* m, bool user, bool full) {
  const double* X = user ? m->U : m->V;
  const double* w = user ? nullptr : m->Wi;
  const int r0 = full ? 0 : (user ? m->ub : m->ib);
  const int r1 = full ? (user ? m->M : m->N) : (user ? m->ue : m->ie);
  double* S = user ? m->SU : m->SV;
  DISPATCH_LD(m->LD, OK(launch_gram<LD>(m, X, w, r0, r1, S)));
  if (user) m->su_fresh = true;
  OK(join_route(m));
  return sync_if_debug(m);
}

// Position-dependent 64-bit checksum of a buffer of doubles: sum over t of mix(bits[t] ^ t * golden) mod 2^64 —
// an associative sum, so the result does not depend on the thread schedule.  Used to prove that the U / V
// replicas of all ranks are bit-identical (eals_factor_hash).
__global__ void hash_doubles_kernel(const double* __restrict__ x, size_t n, unsigned long long* __restrict__ out) {
  unsigned long long acc = 0;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (size_t)gridDim.x * blockDim.x) {
    unsigned long long v = (unsigned long long)__double_as_longlong(x[t]) ^ ((unsigned long long)t * 0x9E3779B97F4A7C15ull);
    v ^= v >> 30; v *= 0xBF58476D1CE4E5B9ull; v ^= v >> 27; v *= 0x94D049BB133111EBull; v ^= v >> 31;   // splitmix64 finaliser
    acc += v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(eals::kFullMask, acc, o);
  if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

// Scatter dense [n][K] (host or device) into the padded [n][LD] device layout and back.
__global__ void pad_rows_kernel(const double* __restrict__ src, double* __restrict__ dst, size_t n, int K, int LD) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * LD) return;
  const size_t r = t / LD;
  const int c = (int)(t % LD);
  dst[t] = c < K ? src[r * K + c] : 0.0;
}
__global__ void unpad_rows_kernel(const double* __restrict__ src, double* __restrict__ dst, size_t n, int K, int LD) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * K) return;
  const size_t r = t / K;
  const int c = (int)(t % K);
  dst[t] = src[r * LD + c];
}

int upload_dense(eals_model* m, double* dst, const double* src, size_t n, int space) {
  const int K = m->K, LD = m->LD;
  if (n == 0) return EALS_OK;
  if (K == LD) return copy_in(dst, src, n * K, space, m->stream);
  const double* dsrc = src;
  double* tmp = nullptr;
  if (space != EALS_DEVICE) {
    OK(dev_alloc(&tmp, n * K));
    CU(cudaMemcpyAsync(tmp, src, n * K * sizeof(double), cudaMemcpyHostToDevice, m->stream));
    dsrc = tmp;
  }
  const size_t total = n * LD;
  pad_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, m->stream>>>(dsrc, dst, n, K, LD);
  OK(check_launch(m));
  if (tmp) { CU(cudaStreamSynchronize(m->stream)); cudaFree(tmp); }
  return EALS_OK;
}

int download_dense(eals_model* m, double* dst, const double* src, size_t n, int space) {
  const int K = m->K, LD = m->LD;
  if (n == 0) return EALS_OK;
  const cudaMemcpyKind kind = space == EALS_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  if (K == LD) {
    CU(cudaMemcpyAsync(dst, src, n * K * sizeof(double), kind, m->stream));
    CU(cudaStreamSynchronize(m->stream));
    return EALS_OK;
  }
  double* ddst = dst;
  double* tmp = nullptr;
  if (space != EALS_DEVICE) {
    OK(dev_alloc(&tmp, n * K));
    ddst = tmp;
  }
  const size_t total = n * K;
  unpad_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, m->stream>>>(src, ddst, n, K, LD);
  OK(check_launch(m));
  if (tmp) CU(cudaMemcpyAsync(dst, tmp, total * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
  CU(cudaStreamSynchronize(m->stream));
  cudaFree(tmp);
  return EALS_OK;
}

template <int LD>
int launch_loss_rows(eals_model* m, const eals::LossSide& a, Side& s, int* n_partials) {
  const int short_first = s.first[1], short_count = s.first[kMidBucket] - s.first[1];
  const int long_first = s.first[kMidBucket], long_count = s.first[kNumBuckets] - s.first[kMidBucket];
  const int g_short = short_count ? std::min((short_count + 7) / 8, 8 * m->sm_count) : 0;
  const int g_long = long_count ? std::min(long_count, 8 * m->sm_count) : 0;
  OK(ensure_partials(m, (size_t)std::max(1, g_short + g_long)));
  if (g_short) {
    eals::loss_rows_kernel<LD, 32><<<g_short, eals::kLossThreads, 0, m->stream>>>(a, s.order, short_first, short_count, m->partials);
    OK(check_launch(m));
  }
  if (g_long) {
    eals::loss_rows_kernel<LD, 256><<<g_long, eals::kLossThreads, 0, m->stream>>>(a, s.order, long_first, long_count, m->partials + g_short);
    OK(check_launch(m));
  }
  *n_partials = g_short + g_long;
  return EALS_OK;
}

int loss_terms_enqueue(eals_model* m) {
  if (!m->factors_set) return fail(EALS_ERR_STATE, "factors not initialised");
  CU(cudaSetDevice(m->p.device));
  OK(join_route(m));
  OK(unpack_pending(m));
  tic(m, T_LOSS);
  eals::LossSide a;
  Side& s = m->users;
  a.ptr = s.ptr; a.idx = s.idx; a.val = s.val;
  a.X = m->U; a.Y = m->V; a.Wi = m->Wi; a.row_base = s.row_base;
  int np = 0;
  if (m->pcache_on && m->pc_attached && m->pc_u_valid) {   // every prediction is already cached: stream it, no gather
    np = 8 * m->sm_count;
    OK(ensure_partials(m, (size_t)np));
    eals::loss_cached_kernel<<<np, eals::kLossThreads, 0, m->stream>>>(s.idx, s.val, m->pc_u, m->Wi, s.nnz, m->partials);
    OK(check_launch(m));
  } else {
    DISPATCH_LD(m->LD, OK(launch_loss_rows<LD>(m, a, s, &np)));
  }
  eals::sum_partials_kernel<<<1, 256, 0, m->stream>>>(m->partials, np, m->terms + 0, 0);
  OK(check_launch(m));
  const int g = 4 * m->sm_count;
  OK(ensure_partials(m, (size_t)g));
  eals::sumsq_kernel<<<g, 256, 0, m->stream>>>(m->U, (size_t)m->ub * m->LD, (size_t)m->ue * m->LD, m->partials);
  OK(check_launch(m));
  eals::sum_partials_kernel<<<1, 256, 0, m->stream>>>(m->partials, g, m->terms + 1, 0);
  OK(check_launch(m));
  eals::sumsq_kernel<<<g, 256, 0, m->stream>>>(m->V, (size_t)m->ib * m->LD, (size_t)m->ie * m->LD, m->partials);
  OK(check_launch(m));
  eals::sum_partials_kernel<<<1, 256, 0, m->stream>>>(m->partials, g, m->terms + 2, 0);
  OK(check_launch(m));
  // sum_u u^T SV u (MF_fastALS.cpp:199-200) = <U^T U, SV>_F.  The cached SU is U^T U only while it is
  // fresh; after single-row updates (update_user_thread / updateModel, which leave SU alone as the
  // reference does) the Gram of the CURRENT U goes to a scratch block — SU itself must stay stale.
  const double* su_now = m->SU;
  if (!m->su_fresh) {
    if (!m->S_tmp) OK(dev_alloc(&m->S_tmp, (size_t)m->LD * m->LD));
    DISPATCH_LD(m->LD, OK(launch_gram<LD>(m, m->U, nullptr, 0, m->M, m->S_tmp)));
    su_now = m->S_tmp;
  }
  eals::frob_inner_kernel<<<1, 256, 0, m->stream>>>(su_now, m->SV, m->K, m->LD, m->terms + 3);
  OK(check_launch(m));
  toc(m, T_LOSS);
  return EALS_OK;
}

int loss_terms_fetch(eals_model* m, double terms[4]) {
  CU(cudaSetDevice(m->p.device));
  CU(cudaMemcpyAsync(terms, m->terms, 4 * sizeof(double), cudaMemcpyDeviceToHost, m->stream));
  CU(cudaStreamSynchronize(m->stream));
  return EALS_OK;
}

int loss_terms(eals_model* m, double terms[4]) {
  OK(loss_terms_enqueue(m));
  return loss_terms_fetch(m, terms);
}

}  // namespace

#include "retrieval.cuh"

// ================================================================================================
extern "C" {

int eals_abi_version(void) { return EALS_ABI_VERSION; }
const char* eals_last_error(void) { return g_err; }

void eals_default_params(eals_params* p) {
  std::memset(p, 0, sizeof(*p));
  p->struct_bytes = (int32_t)sizeof(eals_params);
  p->factors = 64;      // main.cpp:133-144
  p->topk = 10;
  p->w0 = 10;
  p->alpha = 0.75;
  p->reg = 0.01;
  p->init_mean = 0;
  p->init_stdev = 0.01;
  p->input_space = EALS_HOST;
}

int eals_destroy(eals_model* m) {
  if (!m) return EALS_OK;
  cudaSetDevice(m->p.device);
  if (m->stream) cudaStreamSynchronize(m->stream);
  eals_ipc_detach(m);
  free_side(m->users);
  free_side(m->items);
  cudaFree(m->U); cudaFree(m->V); cudaFree(m->SU); cudaFree(m->SV); cudaFree(m->Wi);
  cudaFree(m->terms); cudaFree(m->partials); cudaFree(m->flags); cudaFree(m->S_tmp);
  cudaFree(m->pc_u); cudaFree(m->pc_i); cudaFree(m->map_u); cudaFree(m->map_i);
  cudaFree(m->pc_stage_u); cudaFree(m->pc_stage_i);
  cudaFree(m->route_src_u); cudaFree(m->route_dst_u); cudaFree(m->route_src_i); cudaFree(m->route_dst_i);
  cudaFree(m->recv_idx_u); cudaFree(m->recv_idx_i);
  for (void* p : m->graveyard) cudaFree(p);
  delete m->eval;
  cudaFree(m->full_rp); cudaFree(m->full_cp); cudaFree(m->full_ci); cudaFree(m->full_ri); cudaFree(m->route_tmp);
  fold_timings(m);
  for (cudaEvent_t e : m->pool) cudaEventDestroy(e);
  if (m->epoch_graph) cudaGraphExecDestroy(m->epoch_graph);
  for (int c = 0; c < 2; c++)
    if (m->copy_stream[c]) { cudaStreamSynchronize(m->copy_stream[c]); cudaStreamDestroy(m->copy_stream[c]); cudaEventDestroy(m->ev_copied[c]); }
  if (m->side_stream) { cudaStreamSynchronize(m->side_stream); cudaStreamDestroy(m->side_stream); cudaEventDestroy(m->ev_swept); cudaEventDestroy(m->ev_routed); }
  if (m->own_stream) cudaStreamDestroy(m->own_stream);
  delete m;
  return EALS_OK;
}

int eals_create(const eals_params* params, const int64_t* row_ptr, const int32_t* col_idx,
                const double* row_val, const int64_t* col_ptr, const int32_t* row_idx,
                const double* col_val, eals_model** out) {
  if (!out) return fail(EALS_ERR_ARG, "out is null");
  *out = nullptr;
  if (!params || params->struct_bytes != (int32_t)sizeof(eals_params))
    return fail(EALS_ERR_ARG, "params null or struct_bytes mismatch");
  if (!row_ptr || !col_ptr || (!col_idx && !row_idx)) return fail(EALS_ERR_ARG, "matrix arrays are null");
  if (!col_idx || !row_idx) return fail(EALS_ERR_ARG, "both CSR and CSC index arrays are required");
  if ((row_val == nullptr) != (col_val == nullptr)) return fail(EALS_ERR_ARG, "row_val and col_val must both be given or both be null");
  if (params->n_users <= 0 || params->n_items <= 0) return fail(EALS_ERR_ARG, "empty matrix");
  if (params->factors < 1 || params->factors > 256) return fail(EALS_ERR_UNSUPPORTED, "factors must be in 1..256");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(EALS_ERR_CUDA, "no CUDA device: libeals_b200 has no CPU fallback");
  if (params->device < 0 || params->device >= ndev) return fail(EALS_ERR_ARG, "device %d out of range", params->device);

  eals_model* m = new (std::nothrow) eals_model();
  if (!m) return fail(EALS_ERR_ALLOC, "host allocation failed");
  m->p = *params;
  m->K = params->factors;
  m->LD = eals::leading_dim_for(m->K);
  m->M = params->n_users;
  m->N = params->n_items;
  m->ub = params->user_begin; m->ue = params->user_end;
  m->ib = params->item_begin; m->ie = params->item_end;
  if (m->ub == 0 && m->ue == 0) m->ue = m->M;
  if (m->ib == 0 && m->ie == 0) m->ie = m->N;
  m->n_ranks = std::max(1, params->n_ranks);
  m->rank = params->rank;
  auto bail = [&](int code) { eals_destroy(m); return code; };
  if (m->ub < 0 || m->ue > m->M || m->ub > m->ue || m->ib < 0 || m->ie > m->N || m->ib > m->ie)
    return bail(fail(EALS_ERR_ARG, "owned ranges out of bounds"));
  if (m->n_ranks > 1) {
    const eals_params& q = *params;
    bool ok = m->n_ranks <= 8 && q.rank >= 0 && q.rank < m->n_ranks && q.user_bounds[0] == 0 && q.item_bounds[0] == 0 &&
              q.user_bounds[m->n_ranks] == m->M && q.item_bounds[m->n_ranks] == m->N &&
              q.user_bounds[q.rank] == m->ub && q.user_bounds[q.rank + 1] == m->ue &&
              q.item_bounds[q.rank] == m->ib && q.item_bounds[q.rank + 1] == m->ie;
    for (int r = 0; ok && r < m->n_ranks; r++)
      ok = q.user_bounds[r] <= q.user_bounds[r + 1] && q.item_bounds[r] <= q.item_bounds[r + 1];
    if (!ok) return bail(fail(EALS_ERR_ARG, "inconsistent multi-rank layout (n_ranks, rank, user_bounds, item_bounds)"));
  }

#define TRY(call) do { int r__ = (call); if (r__ != EALS_OK) return bail(r__); } while (0)
#define TRYCU(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return bail(fail(EALS_ERR_CUDA, "%s -> %s", #call, cudaGetErrorString(e__))); } while (0)
  TRYCU(cudaSetDevice(params->device));
  TRYCU(cudaStreamCreateWithFlags(&m->own_stream, cudaStreamNonBlocking));
  m->stream = m->own_stream;
  TRYCU(cudaDeviceGetAttribute(&m->sm_count, cudaDevAttrMultiProcessorCount, params->device));
  TRY(dev_alloc(&m->U, (size_t)m->M * m->LD));
  TRY(dev_alloc(&m->V, (size_t)m->N * m->LD));
  TRY(dev_alloc(&m->SU, (size_t)m->LD * m->LD));
  TRY(dev_alloc(&m->SV, (size_t)m->LD * m->LD));
  TRY(dev_alloc(&m->Wi, (size_t)m->N));
  TRY(dev_alloc(&m->terms, 4));
  TRY(dev_alloc(&m->flags, 16));
  TRYCU(cudaMemsetAsync(m->U, 0, sizeof(double) * (size_t)m->M * m->LD, m->stream));
  TRYCU(cudaMemsetAsync(m->V, 0, sizeof(double) * (size_t)m->N * m->LD, m->stream));
  TRYCU(cudaMemsetAsync(m->SU, 0, sizeof(double) * (size_t)m->LD * m->LD, m->stream));
  TRYCU(cudaMemsetAsync(m->SV, 0, sizeof(double) * (size_t)m->LD * m->LD, m->stream));
  TRYCU(cudaMemsetAsync(m->terms, 0, sizeof(double) * 4, m->stream));
  TRY(build_side(m, m->users, m->ub, m->ue, m->N, params->input_space, row_ptr, col_idx, row_val, m->flags));
  TRY(build_side(m, m->items, m->ib, m->ie, m->M, params->input_space, col_ptr, row_idx, col_val, m->flags + 8));
  TRY(compute_item_weights(m, params->input_space, col_ptr));
  TRY(build_pred_cache(m, params->input_space, row_ptr, col_idx, col_ptr, row_idx));
  TRYCU(cudaStreamSynchronize(m->stream));
#undef TRY
#undef TRYCU
  *out = m;
  return EALS_OK;
}

int eals_set_train(eals_model* m, int32_t input_space, const int64_t* row_ptr, const int32_t* col_idx,
                   const double* row_val, const int64_t* col_ptr, const int32_t* row_idx,
                   const double* col_val) {
  if (!m || !row_ptr || !col_idx || !col_ptr || !row_idx) return fail(EALS_ERR_ARG, "null argument");
  if ((row_val == nullptr) != (col_val == nullptr)) return fail(EALS_ERR_ARG, "row_val and col_val must both be given or both be null");
  CU(cudaSetDevice(m->p.device));
  m->config_gen++;
  OK(build_side(m, m->users, m->ub, m->ue, m->N, input_space, row_ptr, col_idx, row_val, m->flags));
  OK(build_side(m, m->items, m->ib, m->ie, m->M, input_space, col_ptr, row_idx, col_val, m->flags + 8));
  return build_pred_cache(m, input_space, row_ptr, col_idx, col_ptr, row_idx);
}

int eals_refresh_S(eals_model* m) {
  if (!m) return fail(EALS_ERR_ARG, "null model");
  CU(cudaSetDevice(m->p.device));
  OK(gram(m, true, true));
  OK(gram(m, false, true));
  return EALS_OK;
}

int eals_init_factors(eals_model* m) {
  if (!m) return fail(EALS_ERR_ARG, "null model");
  CU(cudaSetDevice(m->p.device));
  // DenseMat::init (DenseMat.cpp:54-62): a fresh default-seeded engine per matrix, so U and V are
  // prefixes of ONE stream; generated once, bit-identical to the reference's sequential loop (init_stream).
  const size_t rows = (size_t)std::max(m->M, m->N);
  std::vector<double> stream;
  try {
    stream.resize(rows * m->K);
  } catch (const std::bad_alloc&) {
    return fail(EALS_ERR_ALLOC, "host allocation of the init stream failed");
  }
  const auto t_init0 = std::chrono::steady_clock::now();
  init_stream(m->p.init_mean, m->p.init_stdev, stream.data(), stream.size());
  m->init_stream_s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_init0).count();
  OK(upload_dense(m, m->U, stream.data(), (size_t)m->M, EALS_HOST));
  OK(upload_dense(m, m->V, stream.data(), (size_t)m->N, EALS_HOST));
  CU(cudaStreamSynchronize(m->stream));
  m->factors_set = true;
  m->pc_u_valid = m->pc_i_valid = false;
  return eals_refresh_S(m);
}

int eals_set_factors(eals_model* m, int32_t space, const double* U, const double* V) {
  if (!m) return fail(EALS_ERR_ARG, "null model");
  CU(cudaSetDevice(m->p.device));
  if (U) OK(upload_dense(m, m->U, U, (size_t)m->M, space));
  if (V) OK(upload_dense(m, m->V, V, (size_t)m->N, space));
  CU(cudaStreamSynchronize(m->stream));
  m->factors_set = true;
  m->pc_u_valid = m->pc_i_valid = false;
  return eals_refresh_S(m);
}

int eals_get_factors(eals_model* m, int32_t space, double* U, double* V) {
  if (!m) return fail(EALS_ERR_ARG, "null model");
  CU(cudaSetDevice(m->p.device));
  if (U) OK(download_dense(m, U, m->U, (size_t)m->M, space));
  if (V) OK(download_dense(m, V, m->V, (size_t)m->N, space));
  return EALS_OK;
}

namespace {
struct CkptHeader {
  char magic[8];
  int32_t version, factors;
  int64_t n_users, n_items;
};
constexpr char kCkptMagic[8] = {'E', 'A', 'L', 'S', 'B', '2', '0', '0'};
constexpr size_t kCkptChunkRows = 1 << 18;
}  // namespace

int eals_save_factors(eals_model* m, const char* path) {
  if (!m || !path) return fail(EALS_ERR_ARG, "null argument");
  if (!m->factors_set) return fail(EALS_ERR_STATE, "factors not initialised");
  CU(cudaSetDevice(m->p.device));
  FILE* f = fopen(path, "wb");
  if (!f) return fail(EALS_ERR_ARG, "cannot open %s for writing", path);
  CkptHeader h;
  std::memcpy(h.magic, kCkptMagic, 8);
  h.version = 1; h.factors = m->K; h.n_users = m->M; h.n_items = m->N;
  bool ok = fwrite(&h, sizeof(h), 1, f) == 1;
  std::vector<double> buf(kCkptChunkRows * (size_t)m->K);
  int rc = EALS_OK;
  for (int side = 0; side < 2 && ok && rc == EALS_OK; side++) {
    const size_t n = side == 0 ? (size_t)m->M : (size_t)m->N;
    const double* src = side == 0 ? m->U : m->V;
    for (size_t r0 = 0; r0 < n && ok && rc == EALS_OK; r0 += kCkptChunkRows) {
      const size_t nr = std::min(kCkptChunkRows, n - r0);
      rc = download_dense(m, buf.data(), src + r0 * m->LD, nr, EALS_HOST);
      ok = rc == EALS_OK && fwrite(buf.data(), sizeof(double), nr * m->K, f) == nr * m->K;
    }
  }
  if (ok && rc == EALS_OK) {
    std::vector<double> wi((size_t)m->N);
    rc = eals_get_item_weights(m, EALS_HOST, wi.data());
    ok = rc == EALS_OK && fwrite(wi.data(), sizeof(double), wi.size(), f) == wi.size();
  }
  ok = (fclose(f) == 0) && ok;
  if (rc != EALS_OK) return rc;
  return ok ? EALS_OK : fail(EALS_ERR_ARG, "short write to %s", path);
}

int eals_load_factors(eals_model* m, const char* path) {
  if (!m || !path) return fail(EALS_ERR_ARG, "null argument");
  CU(cudaSetDevice(m->p.device));
  FILE* f = fopen(path, "rb");
  if (!f) return fail(EALS_ERR_ARG, "cannot open %s", path);
  CkptHeader h;
  if (fread(&h, sizeof(h), 1, f) != 1 || std::memcmp(h.magic, kCkptMagic, 8) != 0 || h.version != 1) {
    fclose(f);
    return fail(EALS_ERR_ARG, "%s is not an eals_b200 factor checkpoint (version 1)", path);
  }
  if (h.factors != m->K || h.n_users != m->M || h.n_items != m->N) {
    fclose(f);
    return fail(EALS_ERR_ARG, "checkpoint is %lld x %lld, K=%d; the model is %d x %d, K=%d", (long long)h.n_users,
                (long long)h.n_items, h.factors, m->M, m->N, m->K);
  }
  std::vector<double> buf(kCkptChunkRows * (size_t)m->K);
  int rc = EALS_OK;
  bool ok = true;
  for (int side = 0; side < 2 && ok && rc == EALS_OK; side++) {
    const size_t n = side == 0 ? (size_t)m->M : (size_t)m->N;
    double* dst = side == 0 ? m->U : m->V;
    for (size_t r0 = 0; r0 < n && ok && rc == EALS_OK; r0 += kCkptChunkRows) {
      const size_t nr = std::min(kCkptChunkRows, n - r0);
      ok = fread(buf.data(), sizeof(double), nr * m->K, f) == nr * m->K;
      if (ok) rc = upload_dense(m, dst + r0 * m->LD, buf.data(), nr, EALS_HOST);
      if (rc == EALS_OK && cudaStreamSynchronize(m->stream) != cudaSuccess) rc = fail(EALS_ERR_CUDA, "checkpoint upload");
    }
  }
  std::vector<double> wi((size_t)m->N);
  if (ok && rc == EALS_OK) ok = fread(wi.data(), sizeof(double), wi.size(), f) == wi.size();
  fclose(f);
  if (rc != EALS_OK) return rc;
  if (!ok) return fail(EALS_ERR_ARG, "%s is truncated", path);
  m->factors_set = true;
  m->pc_u_valid = m->pc_i_valid = false;
  CU(cudaMemcpyAsync(m->Wi, wi.data(), sizeof(double) * m->N, cudaMemcpyHostToDevice, m->stream));
  CU(cudaStreamSynchronize(m->stream));
  return eals_refresh_S(m);
}

int eals_get_factor_row(eals_model* m, int32_t which, int32_t row, double* out) {
  if (!m || !out) return fail(EALS_ERR_ARG, "null argument");
  if (which != EALS_BUF_U && which != EALS_BUF_V) return fail(EALS_ERR_ARG, "which must be EALS_BUF_U or EALS_BUF_V");
  const int n = which == EALS_BUF_U ? m->M : m->N;
  if (row < 0 || row >= n) return fail(EALS_ERR_ARG, "row %d out of range", row);
  CU(cudaSetDevice(m->p.device));
  const double* src = (which == EALS_BUF_U ? m->U : m->V) + (size_t)row * m->LD;
  CU(cudaMemcpyAsync(out, src, sizeof(double) * m->K, cudaMemcpyDeviceToHost, m->stream));
  CU(cudaStreamSynchronize(m->stream));
  return EALS_OK;
}

int eals_set_item_weights(eals_model* m, int32_t space, const double* Wi) {
  if (!m || !Wi) return fail(EALS_ERR_ARG, "null argument");
  CU(cudaSetDevice(m->p.device));
  OK(copy_in(m->Wi, Wi, (size_t)m->N, space, m->stream));
  CU(cudaStreamSynchronize(m->stream));
  if (m->factors_set) OK(gram(m, false, true));
  return EALS_OK;
}

int eals_get_item_weights(eals_model* m, int32_t space, double* Wi) {
  if (!m || !Wi) return fail(EALS_ERR_ARG, "null argument");
  CU(cudaSetDevice(m->p.device));
  CU(cudaMemcpyAsync(Wi, m->Wi, sizeof(double) * m->N,
                     space == EALS_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, m->stream));
  CU(cudaStreamSynchronize(m->stream));
  return EALS_OK;
}

int eals_get_S(eals_model* m, int32_t space, double* SU, double* SV) {
  if (!m) return fail(EALS_ERR_ARG, "null model");
  CU(cudaSetDevice(m->p.device));
  if (SU) OK(download_dense(m, SU, m->SU, (size_t)m->K, space));
  if (SV) OK(download_dense(m, SV, m->SV, (size_t)m->K, space));
  return EALS_OK;
}

int eals_sweep_users(eals_model* m) {
  if (!m) return fail(EALS_ERR_ARG, "null model");
  CU(cudaSetDevice(m->p.device));
  tic(m, T_USER_SWEEP);
  OK(sweep(m, true, -1));
  toc(m, T_USER_SWEEP);
  return EALS_OK;
}
int eals_sweep_items(eals_model* m) {
  if (!m) return fail(EALS_ERR_ARG, "null model");
  CU(cudaSetDevice(m->p.device));
  tic(m, T_ITEM_SWEEP);
  OK(sweep(m, false, -1));
  toc(m, T_ITEM_SWEEP);
  return EALS_OK;
}
int eals_gram_users(eals_model* m) {
  if (!m) return fail(EALS_ERR_ARG, "null model");
  CU(cudaSetDevice(m->p.device));
  tic(m, T_USER_GRAM);
  OK(gram(m, true, false));
  toc(m, T_USER_GRAM);
  return EALS_OK;
}
int eals_gram_items(eals_model* m) {
  if (!m) return fail(EALS_ERR_ARG, "null model");
  CU(cudaSetDevice(m->p.device));
  tic(m, T_ITEM_GRAM);
  OK(gram(m, false, false));
  toc(m, T_ITEM_GRAM);
  return EALS_OK;
}
int eals_update_user(eals_model* m) {
  OK(eals_sweep_users(m));
  return eals_gram_users(m);
}
int eals_update_item(eals_model* m) {
  OK(eals_sweep_items(m));
  return eals_gram_items(m);
}

// n epochs (update_user + update_item each).  use_graph: the epoch is captured ONCE into a CUDA graph — after
// one ordinary epoch, so that every scratch buffer has its final size and the symmetric prediction cache is in
// its steady state — and replayed; the graph is dropped whenever the matrix, the stream or the cache state
// changes.  Single-rank models only (between ranks the exchange is issued by the host layer).
int eals_run_epochs(eals_model* m, int32_t n, int32_t use_graph) {
  if (!m || n < 0) return fail(EALS_ERR_ARG, "bad argument");
  if (!m->factors_set) return fail(EALS_ERR_STATE, "factors not initialised");
  CU(cudaSetDevice(m->p.device));
  const bool graph_ok = use_graph && m->n_ranks <= 1 && m->peersU.n == 0 && !(m->p.flags & EALS_FLAG_SYNC_EACH_CALL) &&
                        m->pred_refresh_every == 0;
  int done = 0;
  if (graph_ok && n > 0) {
    // steady state: both caches valid (or no cache at all) — reached after one ordinary epoch
    const bool steady = !m->pcache_on || !m->pc_attached || (m->pc_u_valid && !m->pc_i_valid);
    if (!steady || m->epoch_graph == nullptr || m->graph_key != m->config_gen) {
      OK(eals_update_user(m)); OK(eals_update_item(m));      // ordinary epoch: sizes scratch, settles the cache state
      done = 1;
    }
    if (done < n && (m->epoch_graph == nullptr || m->graph_key != m->config_gen)) {
      if (m->epoch_graph) { cudaGraphExecDestroy(m->epoch_graph); m->epoch_graph = nullptr; }
      cudaGraph_t g = nullptr;
      // The legacy default stream (what a host that shares "the current stream" may have handed us) cannot be
      // captured: record on the model's own stream; the finished graph is launched on m->stream all the same.
      cudaStream_t user_stream = m->stream;
      m->stream = m->own_stream;
      const cudaError_t e0 = cudaStreamBeginCapture(m->stream, cudaStreamCaptureModeThreadLocal);
      if (e0 != cudaSuccess) {
        m->stream = user_stream;
        cudaGetLastError();
        return fail(EALS_ERR_CUDA, "cudaStreamBeginCapture -> %s", cudaGetErrorString(e0));
      }
      m->capturing = true;
      const long long launches_before = m->launches;
      int rc = eals_update_user(m);
      if (rc == EALS_OK) rc = eals_update_item(m);
      m->capturing = false;
      m->graph_launches_per_epoch = m->launches - launches_before;
      m->launches = launches_before;      // captured, not executed
      const cudaError_t e = cudaStreamEndCapture(m->stream, &g);
      m->stream = user_stream;
      if (e != cudaSuccess) cudaGetLastError();
      if (rc != EALS_OK) { if (g) cudaGraphDestroy(g); return rc; }
      if (e != cudaSuccess) return fail(EALS_ERR_CUDA, "epoch capture -> %s", cudaGetErrorString(e));
      const cudaError_t e2 = cudaGraphInstantiate(&m->epoch_graph, g, 0);
      cudaGraphDestroy(g);
      if (e2 != cudaSuccess) return fail(EALS_ERR_CUDA, "epoch graph instantiation -> %s", cudaGetErrorString(e2));
      m->graph_key = m->config_gen;
      // the captured calls toggled the host-side cache flags exactly as an executed epoch would: still steady
    }
    for (; done < n; done++) {
      CU(cudaGraphLaunch(m->epoch_graph, m->stream));
      m->launches += m->graph_launches_per_epoch;
    }
    return EALS_OK;
  }
  for (; done < n; done++) { OK(eals_update_user(m)); OK(eals_update_item(m)); }
  return EALS_OK;
}

int eals_update_user_row(eals_model* m, int32_t u) {
  if (!m) return fail(EALS_ERR_ARG, "null model");
  if (u < m->ub || u >= m->ue) return fail(EALS_ERR_ARG, "user %d not owned by this model", u);
  CU(cudaSetDevice(m->p.device));
  return sweep(m, true, u - m->ub);
}
int eals_update_item_row(eals_model* m, int32_t i) {
  if (!m) return fail(EALS_ERR_ARG, "null model");
  if (i < m->ib || i >= m->ie) return fail(EALS_ERR_ARG, "item %d not owned by this model", i);
  CU(cudaSetDevice(m->p.device));
  return sweep(m, false, i - m->ib);
}

static int patch_S(eals_model* m, double* S, double scale, const double* old_row, const double* new_row) {
  if (!old_row || !new_row) return fail(EALS_ERR_ARG, "null row");
  CU(cudaSetDevice(m->p.device));
  OK(ensure_partials(m, (size_t)2 * m->K + 16));
  CU(cudaMemcpyAsync(m->partials, old_row, sizeof(double) * m->K, cudaMemcpyHostToDevice, m->stream));
  CU(cudaMemcpyAsync(m->partials + m->K, new_row, sizeof(double) * m->K, cudaMemcpyHostToDevice, m->stream));
  const int total = m->K * m->K;
  eals::gram_patch_kernel<<<(total + 255) / 256, 256, 0, m->stream>>>(S, m->partials, m->partials + m->K, scale, m->K, m->LD);
  OK(check_launch(m));
  CU(cudaStreamSynchronize(m->stream));  // the host rows may be reused by the caller
  return EALS_OK;
}
int eals_patch_SU(eals_model* m, const double* old_row, const double* new_row) {
  if (!m) return fail(EALS_ERR_ARG, "null model");
  return patch_S(m, m->SU, 1.0, old_row, new_row);
}
int eals_patch_SV(eals_model* m, int32_t i, const double* old_row, const double* new_row) {
  if (!m) return fail(EALS_ERR_ARG, "null model");
  if (i < 0 || i >= m->N) return fail(EALS_ERR_ARG, "item out of range");
  double wi = 0;
  CU(cudaSetDevice(m->p.device));
  CU(cudaMemcpyAsync(&wi, m->Wi + i, sizeof(double), cudaMemcpyDeviceToHost, m->stream));
  CU(cudaStreamSynchronize(m->stream));
  return patch_S(m, m->SV, wi, old_row, new_row);
}

int eals_loss_terms(eals_model* m, double terms[4]) {
  if (!m || !terms) return fail(EALS_ERR_ARG, "null argument");
  CU(cudaSetDevice(m->p.device));
  return loss_terms(m, terms);
}
int eals_loss(eals_model* m, double* loss) {
  if (!m || !loss) return fail(EALS_ERR_ARG, "null argument");
  double t[4];
  OK(eals_loss_terms(m, t));
  *loss = m->p.reg * (t[1] + t[2]) + t[0] + t[3];
  return EALS_OK;
}

int eals_predict(eals_model* m, int32_t u, int32_t i, double* score) {
  if (!m || !score) return fail(EALS_ERR_ARG, "null argument");
  if (u < 0 || u >= m->M || i < 0 || i >= m->N) return fail(EALS_ERR_ARG, "index out of range");
  CU(cudaSetDevice(m->p.device));
  OK(ensure_partials(m, 16));
  int32_t* d_gt = reinterpret_cast<int32_t*>(m->partials + 8);
  CU(cudaMemcpyAsync(d_gt, &i, sizeof(int32_t), cudaMemcpyHostToDevice, m->stream));
  eals::eval_gt_score_kernel<<<1, 128, 0, m->stream>>>(m->U, m->V, d_gt, nullptr, u, 1, m->K, m->LD, m->partials);
  OK(check_launch(m));
  CU(cudaMemcpyAsync(score, m->partials, sizeof(double), cudaMemcpyDeviceToHost, m->stream));
  CU(cudaStreamSynchronize(m->stream));
  return EALS_OK;
}

int eals_evaluate(eals_model* m, const int32_t* gt_items, int32_t topk, int32_t mode, double sums[3],
                  double* hr, double* ndcg, double* prec, int32_t* count_larger) {
  if (!m || !gt_items || !sums) return fail(EALS_ERR_ARG, "null argument");
  if (topk < 1) return fail(EALS_ERR_ARG, "topk must be >= 1");
  if (!m->factors_set) return fail(EALS_ERR_STATE, "factors not initialised");
  CU(cudaSetDevice(m->p.device));
  for (int u = m->ub; u < m->ue; u++)
    if (gt_items[u] < 0 || gt_items[u] >= m->N) return fail(EALS_ERR_ARG, "gt item of user %d out of range", u);
  std::vector<int32_t> users((size_t)(m->ue - m->ub));
  for (int u = m->ub; u < m->ue; u++) users[u - m->ub] = u;
  tic(m, T_EVAL);
  const int r = evaluate_slots(m, users, gt_items + m->ub, topk, mode, sums, hr, ndcg, prec, count_larger);
  toc(m, T_EVAL);
  return r;
}

int eals_evaluate_user(eals_model* m, int32_t u, int32_t gt_item, int32_t topk, int32_t mode, double out[3]) {
  if (!m || !out) return fail(EALS_ERR_ARG, "null argument");
  if (u < 0 || u >= m->M || gt_item < 0 || gt_item >= m->N || topk < 1) return fail(EALS_ERR_ARG, "argument out of range");
  if (!m->factors_set) return fail(EALS_ERR_STATE, "factors not initialised");
  CU(cudaSetDevice(m->p.device));
  std::vector<int32_t> users(1, u);
  return evaluate_slots(m, users, &gt_item, topk, mode, out, nullptr, nullptr, nullptr, nullptr);
}

int eals_debug_init_stream(double mean, double stdev, double* out, int64_t n) {
  if (!out || n < 0) return fail(EALS_ERR_ARG, "bad argument");
  init_stream(mean, stdev, out, (size_t)n);
  return EALS_OK;
}

int eals_init_seconds(eals_model* m, double* host_stream_seconds) {
  if (!m || !host_stream_seconds) return fail(EALS_ERR_ARG, "null argument");
  *host_stream_seconds = m->init_stream_s;
  return EALS_OK;
}

int eals_eval_stats(eals_model* m, int64_t out[6]) {
  if (!m || !out) return fail(EALS_ERR_ARG, "null argument");
  const EvalStats& s = m->eval_stats;
  out[0] = s.engine; out[1] = s.candidates; out[2] = s.pairs;
  out[3] = s.blk0.users; out[4] = s.blk0.items; out[5] = (int64_t)(s.blk0.ms * 1000.0);
  return EALS_OK;
}

int eals_recommend(eals_model* m, int32_t space, int32_t n, const int32_t* users, int32_t k, int32_t exclude_seen,
                   int32_t* items, double* scores) {
  return recommend_impl(m, space, n, users, k, exclude_seen, items, scores);
}

int eals_fold_in(eals_model* m, int32_t space, int32_t n, const int64_t* row_ptr, const int32_t* col_idx, const double* val,
                 const double* init, int32_t n_iter, double* out) {
  return fold_in_impl(m, space, n, row_ptr, col_idx, val, init, n_iter, out);
}

int eals_recommend_vectors(eals_model* m, int32_t space, int32_t n, const double* Q, const int64_t* ex_ptr, const int32_t* ex_idx,
                           int32_t k, int32_t* items, double* scores) {
  return recommend_vectors_impl(m, space, n, Q, ex_ptr, ex_idx, k, items, scores);
}

int eals_ranking_metrics(eals_model* m, int32_t space, const int64_t* test_ptr, const int32_t* test_idx, int32_t k,
                         int32_t exclude_seen, double sums[6], int64_t* n_users, double* per_user, int32_t* ranks) {
  return ranking_metrics_impl(m, space, test_ptr, test_idx, k, exclude_seen, sums, n_users, per_user, ranks);
}

int eals_recommend_stats(eals_model* m, int64_t out[7]) {
  if (!m || !out) return fail(EALS_ERR_ARG, "null argument");
  const RecStats& s = m->rec_stats;
  out[0] = s.engine; out[1] = s.seed; out[2] = s.pairs; out[3] = s.left1;
  out[4] = s.blk0.users; out[5] = s.blk0.items; out[6] = (int64_t)(s.blk0.ms * 1000.0);
  return EALS_OK;
}

int eals_leading_dim(const eals_model* m) { return m ? m->LD : 0; }

int eals_device_buffer(eals_model* m, int32_t which, void** dev_ptr, int64_t* bytes) {
  if (!m || !dev_ptr) return fail(EALS_ERR_ARG, "null argument");
  void* p = nullptr;
  int64_t b = 0;
  switch (which) {
    // handing out U or V lets the caller change factors behind the prediction cache's back
    case EALS_BUF_U: p = m->U; b = (int64_t)m->M * m->LD * 8; m->pc_u_valid = m->pc_i_valid = false; break;
    case EALS_BUF_V: p = m->V; b = (int64_t)m->N * m->LD * 8; m->pc_u_valid = m->pc_i_valid = false; break;
    case EALS_BUF_SU: p = m->SU; b = (int64_t)m->K * m->LD * 8; break;
    case EALS_BUF_SV: p = m->SV; b = (int64_t)m->K * m->LD * 8; break;
    case EALS_BUF_WI: p = m->Wi; b = (int64_t)m->N * 8; break;
    case EALS_BUF_LOSS_TERMS: p = m->terms; b = 32; break;
    case EALS_BUF_PC_USER: p = m->pc_u; b = m->pcache_on ? m->users.nnz * 8 : 0; break;
    case EALS_BUF_PC_ITEM: p = m->pc_i; b = m->pcache_on ? m->items.nnz * 8 : 0; break;
    default: return fail(EALS_ERR_ARG, "unknown buffer %d", which);
  }
  *dev_ptr = p;
  if (bytes) *bytes = b;
  return EALS_OK;
}

int eals_stream(eals_model* m, void** cuda_stream) {
  if (!m || !cuda_stream) return fail(EALS_ERR_ARG, "null argument");
  *cuda_stream = (void*)m->stream;
  return EALS_OK;
}

int eals_set_stream(eals_model* m, void* cuda_stream, int32_t restore_own) {
  if (!m) return fail(EALS_ERR_ARG, "null model");
  CU(cudaSetDevice(m->p.device));
  OK(join_route(m));
  CU(cudaStreamSynchronize(m->stream));
  fold_timings(m);
  m->stream = restore_own ? m->own_stream : (cudaStream_t)cuda_stream;
  m->config_gen++;
  return EALS_OK;
}

int eals_ipc_handle(eals_model* m, int32_t which, void* handle_out) {
  if (!m || !handle_out) return fail(EALS_ERR_ARG, "null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == EALS_IPC_HANDLE_BYTES, "IPC handle size");
  void* buf = nullptr;
  switch (which) {
    case EALS_BUF_U: buf = m->U; break;
    case EALS_BUF_V: buf = m->V; break;
    case EALS_BUF_PC_USER: buf = m->pc_u; break;
    case EALS_BUF_PC_ITEM: buf = m->pc_i; break;
    default: return fail(EALS_ERR_ARG, "only U, V and the prediction caches can be shared");
  }
  if (!buf) return fail(EALS_ERR_STATE, "buffer %d does not exist on this model (prediction cache off?)", which);
  CU(cudaSetDevice(m->p.device));
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, buf));
  std::memcpy(handle_out, &h, sizeof(h));
  return EALS_OK;
}

int eals_ipc_generation(eals_model* m) { return m ? m->ipc_gen : -1; }

int eals_ipc_gc(eals_model* m) {
  if (!m) return EALS_OK;
  cudaSetDevice(m->p.device);
  if (m->stream) cudaStreamSynchronize(m->stream);
  for (void* p : m->graveyard) cudaFree(p);
  m->graveyard.clear();
  return EALS_OK;
}

int eals_ipc_detach(eals_model* m) {
  if (!m) return EALS_OK;
  cudaSetDevice(m->p.device);
  if (m->stream) cudaStreamSynchronize(m->stream);
  for (eals::PeerSet* ps : {&m->peersU, &m->peersV}) {
    if (!m->local_peers)
      for (int p = 0; p < ps->n; p++) cudaIpcCloseMemHandle(ps->x[p]);
    ps->n = 0;
  }
  if (m->n_ranks > 1) {
    close_pc_peers(m, m->out_to_users, m->pc_users_attached);
    close_pc_peers(m, m->out_to_items, m->pc_items_attached);
    m->pc_attached = false;
    m->pc_u_valid = m->pc_i_valid = false;
  }
  return EALS_OK;
}

int eals_ipc_attach(eals_model* m, int32_t which, int32_t n_peers, const void* handles) {
  if (!m || (!handles && n_peers > 0)) return fail(EALS_ERR_ARG, "null argument");
  if (n_peers < 0 || n_peers > eals::kMaxPeers) return fail(EALS_ERR_UNSUPPORTED, "at most %d peers", eals::kMaxPeers);
  CU(cudaSetDevice(m->p.device));
  CU(cudaStreamSynchronize(m->stream));
  if (which == EALS_BUF_PC_USER || which == EALS_BUF_PC_ITEM) {
    if (!m->pcache_on) return fail(EALS_ERR_STATE, "prediction cache is off on this model");
    if (m->n_ranks < 2 || n_peers != m->n_ranks - 1)
      return fail(EALS_ERR_ARG, "prediction caches need eals_params.n_ranks - 1 = %d peer handles, got %d", m->n_ranks - 1, n_peers);
    eals::PcOut& out = which == EALS_BUF_PC_USER ? m->out_to_users : m->out_to_items;
    bool& flag = which == EALS_BUF_PC_USER ? m->pc_users_attached : m->pc_items_attached;
    close_pc_peers(m, out, flag);
    int p = 0;
    for (int r = 0; r < m->n_ranks; r++) {
      if (r == m->rank) continue;
      cudaIpcMemHandle_t h;
      std::memcpy(&h, (const char*)handles + (size_t)p++ * EALS_IPC_HANDLE_BYTES, sizeof(h));
      void* ptr = nullptr;
      CU(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
      out.base[r] = (double*)ptr;
    }
    flag = true;
    m->pc_attached = m->pc_users_attached && m->pc_items_attached;
    m->pc_u_valid = m->pc_i_valid = false;
    return EALS_OK;
  }
  if (which != EALS_BUF_U && which != EALS_BUF_V) return fail(EALS_ERR_ARG, "only U, V and the prediction caches can be shared");
  eals::PeerSet& ps = which == EALS_BUF_U ? m->peersU : m->peersV;
  for (int p = 0; p < ps.n; p++) cudaIpcCloseMemHandle(ps.x[p]);
  ps.n = 0;
  for (int p = 0; p < n_peers; p++) {
    cudaIpcMemHandle_t h;
    std::memcpy(&h, (const char*)handles + (size_t)p * EALS_IPC_HANDLE_BYTES, sizeof(h));
    void* ptr = nullptr;
    CU(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
    ps.x[ps.n++] = (double*)ptr;
  }
  return EALS_OK;
}

int eals_factor_hash(eals_model* m, uint64_t out[2]) {
  if (!m || !out) return fail(EALS_ERR_ARG, "null argument");
  CU(cudaSetDevice(m->p.device));
  OK(ensure_partials(m, 16));
  unsigned long long* d = reinterpret_cast<unsigned long long*>(m->partials);
  CU(cudaMemsetAsync(d, 0, 2 * sizeof(unsigned long long), m->stream));
  hash_doubles_kernel<<<4 * m->sm_count, 256, 0, m->stream>>>(m->U, (size_t)m->M * m->LD, d);
  OK(check_launch(m));
  hash_doubles_kernel<<<4 * m->sm_count, 256, 0, m->stream>>>(m->V, (size_t)m->N * m->LD, d + 1);
  OK(check_launch(m));
  unsigned long long h[2];
  CU(cudaMemcpyAsync(h, d, sizeof(h), cudaMemcpyDeviceToHost, m->stream));
  CU(cudaStreamSynchronize(m->stream));
  out[0] = h[0]; out[1] = h[1];
  return EALS_OK;
}

int eals_sync(eals_model* m) {
  if (!m) return fail(EALS_ERR_ARG, "null model");
  CU(cudaSetDevice(m->p.device));
  OK(join_route(m));
  CU(cudaStreamSynchronize(m->stream));
  CU(cudaGetLastError());
  return EALS_OK;
}

int64_t eals_nnz(const eals_model* m) { return m ? m->users.nnz : 0; }
int64_t eals_kernel_launches(const eals_model* m) { return m ? m->launches : 0; }

int eals_timings(eals_model* m, double ms[6]) {
  if (!m || !ms) return fail(EALS_ERR_ARG, "null argument");
  CU(cudaSetDevice(m->p.device));
  CU(cudaStreamSynchronize(m->stream));
  fold_timings(m);
  for (int t = 0; t < kPublicTimers; t++) ms[t] = m->last_ms[t];
  return EALS_OK;
}

int eals_timings_total(eals_model* m, double ms[6], int64_t calls[6], int32_t reset) {
  if (!m) return fail(EALS_ERR_ARG, "null model");
  CU(cudaSetDevice(m->p.device));
  CU(cudaStreamSynchronize(m->stream));
  fold_timings(m);
  for (int t = 0; t < kPublicTimers; t++) {
    if (ms) ms[t] = m->acc_ms[t];
    if (calls) calls[t] = m->acc_calls[t];
  }
  if (reset) for (int t = 0; t < T_COUNT; t++) { m->acc_ms[t] = 0; m->acc_calls[t] = 0; }
  return EALS_OK;
}

int eals_timings_detail(eals_model* m, double ms[6], int64_t calls[6]) {
  if (!m || !ms) return fail(EALS_ERR_ARG, "null argument");
  CU(cudaSetDevice(m->p.device));
  CU(cudaStreamSynchronize(m->stream));
  fold_timings(m);
  for (int t = 0; t < 6; t++) {
    ms[t] = m->acc_ms[T_U_HEAVY + t];
    if (calls) calls[t] = m->acc_calls[T_U_HEAVY + t];
  }
  return EALS_OK;
}

}  // extern "C"

#include "group.cuh"
