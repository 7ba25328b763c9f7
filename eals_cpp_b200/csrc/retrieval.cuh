// retrieval.cuh — the host side of evaluate and recommend: ranking replay, grow-only workspace, the two engines of
// each and the pieces their tcgen05 filter passes share (kernels: eval.cuh, eval_tc.cuh, recommend.cuh).  Included
// from eals_b200.cu ahead of its C entry points: like group.cuh it is part of that one translation unit and uses
// its helpers (fail, CU / OK, dev_reserve, check_launch, StageTimer, ...).

namespace {

double metric_ndcg(int pos) { return std::log(2) / std::log(pos + 2); }  // MF_fastALS.cpp:604-611

// Rank position of gt in the reference's list (MF_fastALS.cpp:641-656) or -1.  `nz` holds the
// (item, (int)score) pairs with a non-zero truncated score, ascending by item; every other item
// has key 0.  The real std::partial_sort_copy runs on a sequence from which only elements that
// cannot pass its `comp(element, heap_top)` test have been dropped, so the result is the one the
// reference gets on the full item list.
struct RankScratch { std::vector<std::pair<int, int>> seq, top; };   // reused across the survivors of a host thread

int reference_rank(const std::vector<std::pair<int, int>>& nz, int n_items, int topk, int gt, RankScratch& ws) {
  auto comp = [](const std::pair<int, int>& l, const std::pair<int, int>& r) { return l.second > r.second; };
  std::vector<std::pair<int, int>>& seq = ws.seq;
  seq.clear();
  const int head = std::min(topk, n_items);
  size_t q = 0;
  bool any_negative = false;
  for (int i = 0; i < head; i++) {
    int key = 0;
    if (q < nz.size() && nz[q].first == i) key = nz[q++].second;
    any_negative |= key < 0;
    seq.emplace_back(i, key);
  }
  if (any_negative) {
    // A negative heap top is displaced by ANY later element with a larger key — zero keys included.  Every
    // accepted element with key >= 0 removes one negative key from the heap for good (it replaces the top,
    // the most negative one), and while a negative is left every element with key >= 0 is accepted.  So the
    // first `neg` non-negative elements after the head matter (walking the items in id order, zeros and
    // listed keys merged), negative keys in that stretch may matter too, and from then on the heap top is
    // >= 0: only positive keys can pass comp(e, top).  (The full 2M-item list per such user made the replay
    // 0.4 s at 10M x 2M.)
    int neg = 0;
    for (const auto& e : seq) neg += e.second < 0;
    int i = head;
    while (neg > 0 && i < n_items) {
      int key = 0;
      if (q < nz.size() && nz[q].first == i) key = nz[q++].second;
      seq.emplace_back(i, key);
      if (key >= 0) neg--;
      i++;
    }
    for (; q < nz.size(); q++)
      if (nz[q].second > 0) seq.push_back(nz[q]);
  } else {
    // heap top stays >= 0: only positive keys can ever pass comp(e, top)
    for (; q < nz.size(); q++)
      if (nz[q].second > 0) seq.push_back(nz[q]);
  }
  std::vector<std::pair<int, int>>& top = ws.top;
  top.assign((size_t)topk, std::make_pair(0, 0));                            // value-initialised (:642)
  std::partial_sort_copy(seq.begin(), seq.end(), top.begin(), top.end(), comp);
  for (int t = 0; t < topk; t++)
    if (top[t].first == gt) return t;
  return -1;
}

// The buffers and events of the workspace free themselves when it is deleted (eals_destroy, on the model's device);
// a copy would free them twice.
struct NoCopy { NoCopy() = default; NoCopy(const NoCopy&) = delete; NoCopy& operator=(const NoCopy&) = delete; };

// Grow-only device workspace of the evaluation (kept across calls: no cudaMalloc / cudaFree per evaluate).
template <typename T>
struct WsBuf : NoCopy {
  T* p = nullptr;
  size_t cap = 0;
  ~WsBuf() { cudaFree(p); }
  int reserve(size_t n) { return dev_reserve(&p, &cap, n); }
};

}  // namespace

// Pinned host staging (grow-only): the ranking keys of a 10M-user evaluation are ~300 MB, pageable copies of
// that size run at a few GB/s.
struct PinnedBuf : NoCopy {
  unsigned char* p = nullptr;
  size_t cap = 0;
  ~PinnedBuf() { if (p) cudaFreeHost(p); }
  int reserve(size_t bytes) {
    if (bytes <= cap) return EALS_OK;
    if (p) cudaFreeHost(p);
    p = nullptr; cap = 0;
    CU(cudaHostAlloc((void**)&p, bytes + bytes / 8 + 64, cudaHostAllocDefault));
    cap = bytes + bytes / 8 + 64;
    return EALS_OK;
  }
};

// Device time of the first filtered item block: the one launch whose shape the host knows exactly, timed for the
// tensor roofline of eval_stats / recommend_stats.
struct BlockTimer : NoCopy {
  cudaEvent_t a = nullptr, b = nullptr;
  long long users = 0, items = 0;   // shape of the timed launch
  ~BlockTimer() { if (a) { cudaEventDestroy(a); cudaEventDestroy(b); } }
  int start(cudaStream_t st) {
    if (!a) { CU(cudaEventCreate(&a)); CU(cudaEventCreate(&b)); }
    CU(cudaEventRecord(a, st));
    return EALS_OK;
  }
  int stop(cudaStream_t st, long long n_users, long long n_items) {
    users = n_users; items = n_items;
    CU(cudaEventRecord(b, st));
    return EALS_OK;
  }
  int read(BlockTiming& out) {   // once the stream has passed stop()
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, a, b));
    out = {users, items, ms};
    return EALS_OK;
  }
};

struct eals_eval_ws {
  PinnedBuf host;
  WsBuf<int32_t> users, gt, cnt, cnt_exact, list_a, list_b, perm, ids, exps, scalars;
  WsBuf<double> gts;
  WsBuf<__half> Uh, Vh, W;
  WsBuf<float> un_hat, un_del, un_h, vn_hat, vn_del, vn_h;
  WsBuf<float4> sp0, sp1;
  WsBuf<float2> tile_norm;
  WsBuf<uint32_t> keys, keys_out;
  WsBuf<uint8_t> flags;
  WsBuf<unsigned char> cub_tmp;
  WsBuf<unsigned long long> counters;   // [0] max |V| bits, [1] pairs, [2] triples
  WsBuf<eals::tc::EvalPair> pairs;
  WsBuf<eals::EvalTriple> triples;
  WsBuf<unsigned long long> tkey, tkey_out;
  WsBuf<int32_t> tval, tval_out;
  WsBuf<int32_t> active;
  WsBuf<double> top_s, thr, pscore;               // recommend: per-slot lists and k-th scores, re-scored pairs
  WsBuf<int32_t> top_i, pval, pval_out, run_cnt, run_off;
  WsBuf<uint32_t> pkey, pkey_out, run_slot;
  BlockTimer blk0;
  // fold-in and recommend_vectors: the histories / exclusion lists (validated and bucketed by build_side, row_base
  // 0), their validation scratch (6 ints each), and the query rows [n][LD] (fold-in's X, padding columns zero)
  Side hist, excl;
  WsBuf<int> hist_check, excl_check;
  WsBuf<double> qx;
  // similar: the normalised catalogue [n_Y][LD] and the offsets of the self-exclusion CSR (its index array is ws.users)
  WsBuf<double> yhat;
  WsBuf<int64_t> self_ptr;
  // ranking metrics: the owned rows of the test matrix (validated by build_side, row_base = the first owned user),
  // per entry its rank, per slot c_R and the certain-count limit, the chunk's train scores, the per-user metrics
  // and the gain / ideal-DCG tables
  Side test;
  WsBuf<int> test_check;
  WsBuf<int32_t> ranks, c_r, lim;
  WsBuf<double> tscore, rm_out, rm_tab;
  eals_eval_ws() = default;
  ~eals_eval_ws() { free_side(hist); free_side(excl); free_side(test); }
};

namespace {

eals_eval_ws& eval_ws(eals_model* m) {
  if (!m->eval) m->eval = new eals_eval_ws();
  return *m->eval;
}

// ---- scan engine 1: exact fp64 tiles (eval.cuh), item chunks with an early-out of decided users --------
// Used for short user lists (evaluate_for_user), as the engine the tensor filter is tested against
// (EALS_EVAL_SCALAR=1) and as its fall-back when the candidate list overflows.
// What both scan engines hand back: the users that survive the reference's early-out (count_larger <= topK,
// MF_fastALS.cpp:633-634) with their exact counts — every other user is decided (zeros) — and, for the
// ranking replay, the survivors' (slot, item, (int)score) triples with a non-zero key as two parallel arrays
// sorted by (slot, item): key = slot << 32 | item, val = (int)score.
struct ScanResult {
  std::vector<int32_t> surv_slot, surv_cnt;      // ascending slot
  std::vector<unsigned long long> own_key;       // storage when the arrays do not live in the pinned staging
  std::vector<int32_t> own_val;
  const unsigned long long* key = nullptr;
  const int32_t* val = nullptr;
  size_t n_keys = 0;
};

int scan_exact(eals_model* m, int n, const int32_t* d_users, const double* d_gts, int topk, bool want_triples, ScanResult& out) {
  eals_eval_ws& ws = eval_ws(m);
  std::vector<int32_t> cnt((size_t)n, 0);
  const int K = m->K, LD = m->LD, N = m->N;
  OK(ws.cnt.reserve((size_t)n));
  OK(ws.active.reserve((size_t)n));
  int32_t *d_count = ws.cnt.p, *d_active = ws.active.p;
  CU(cudaMemsetAsync(d_count, 0, sizeof(int32_t) * n, m->stream));
  const int item_tiles = (N + eals::kEvalTile - 1) / eals::kEvalTile;
  // Count strictly larger scores chunk by chunk of items.  The reference gives (0,0,0) as soon as the
  // count exceeds topK (MF_fastALS.cpp:633-634) and the total does not depend on the scan order, so a
  // user whose count already exceeds topK after a chunk is decided and leaves the active list.
  {
    std::vector<int32_t> active((size_t)n);
    for (int s = 0; s < n; s++) active[s] = s;
    std::vector<int32_t> cnt_a;
    int64_t chunk = 4096;
    if (const char* e = getenv("EALS_EVAL_FIRST_CHUNK")) chunk = std::max<int64_t>(64, atoll(e));
    for (int64_t i0 = 0; i0 < N && !active.empty(); i0 += chunk, chunk *= 4) {
      const int i1 = (int)std::min<int64_t>(N, i0 + chunk);
      const int na = (int)active.size();
      CU(cudaMemcpyAsync(d_active, active.data(), sizeof(int32_t) * na, cudaMemcpyHostToDevice, m->stream));
      const long long utiles = (na + eals::kEvalTile - 1) / eals::kEvalTile;
      const long long itiles = (i1 - (int)i0 + eals::kEvalTile - 1) / eals::kEvalTile;
      const long long max_ut = std::max<long long>(1, 0x7fffffffLL / itiles);   // grid limit
      for (long long ut0 = 0; ut0 < utiles; ut0 += max_ut) {
        const long long ut1 = std::min(utiles, ut0 + max_ut);
        const int a0 = (int)(ut0 * eals::kEvalTile), a1 = (int)std::min<long long>(na, ut1 * eals::kEvalTile);
        eals::eval_tile_kernel<0><<<(unsigned)((ut1 - ut0) * itiles), eals::kEvalThreads, 0, m->stream>>>(
            m->U, m->V, d_users, d_active + a0, 0, a1 - a0, (int)i0, i1, K, LD, d_gts, d_count, nullptr, nullptr, 0);
        OK(check_launch(m));
      }
      if (na == n) {
        CU(cudaMemcpyAsync(cnt.data(), d_count, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, m->stream));
        CU(cudaStreamSynchronize(m->stream));
      } else {
        OK(ensure_partials(m, (size_t)(na + 1) / 2 + 1));
        int32_t* d_tmp = reinterpret_cast<int32_t*>(m->partials);
        eals::gather_i32_kernel<<<(na + 255) / 256, 256, 0, m->stream>>>(d_count, d_active, na, d_tmp);
        OK(check_launch(m));
        cnt_a.resize((size_t)na);
        CU(cudaMemcpyAsync(cnt_a.data(), d_tmp, sizeof(int32_t) * na, cudaMemcpyDeviceToHost, m->stream));
        CU(cudaStreamSynchronize(m->stream));
        for (int a = 0; a < na; a++) cnt[active[a]] = cnt_a[a];
      }
      size_t keep = 0;
      for (int a = 0; a < na; a++)
        if (cnt[active[a]] <= topk) active[keep++] = active[a];
      active.resize(keep);
    }
  }
  // survivors of the early-out
  std::vector<int32_t>& surv = out.surv_slot;
  surv.clear(); out.surv_cnt.clear();
  for (int s = 0; s < n; s++)
    if (cnt[s] <= topk) { surv.push_back(s); out.surv_cnt.push_back(cnt[s]); }
  out.key = nullptr; out.val = nullptr; out.n_keys = 0;
  const int ns = (int)surv.size();
  if (!want_triples || ns == 0) return EALS_OK;
  // ... and their (item, (int)score) pairs with a non-zero key
  CU(cudaMemcpyAsync(d_active, surv.data(), sizeof(int32_t) * ns, cudaMemcpyHostToDevice, m->stream));
  OK(ws.counters.reserve(4));
  unsigned long long* d_nt = ws.counters.p + 2;
  unsigned long long cap = 1ull << 20, got = 0;
  const long long utiles = (ns + eals::kEvalTile - 1) / eals::kEvalTile;
  const long long max_ut = std::max<long long>(1, 0x7fffffffLL / item_tiles);
  for (int attempt = 0; attempt < 2; attempt++) {
    OK(ws.triples.reserve((size_t)cap));
    CU(cudaMemsetAsync(d_nt, 0, sizeof(unsigned long long), m->stream));
    for (long long ut0 = 0; ut0 < utiles; ut0 += max_ut) {
      const long long ut1 = std::min(utiles, ut0 + max_ut);
      const int a0 = (int)(ut0 * eals::kEvalTile), a1 = (int)std::min<long long>(ns, ut1 * eals::kEvalTile);
      eals::eval_tile_kernel<1><<<(unsigned)((ut1 - ut0) * item_tiles), eals::kEvalThreads, 0, m->stream>>>(
          m->U, m->V, d_users, d_active + a0, 0, a1 - a0, 0, N, K, LD, nullptr, nullptr, ws.triples.p, d_nt, cap);
      OK(check_launch(m));
    }
    CU(cudaMemcpyAsync(&got, d_nt, sizeof(got), cudaMemcpyDeviceToHost, m->stream));
    CU(cudaStreamSynchronize(m->stream));
    if (got <= cap) break;
    cap = got;  // exact size known now: the second pass cannot overflow
  }
  std::vector<eals::EvalTriple> tr((size_t)got);
  if (got) CU(cudaMemcpy(tr.data(), ws.triples.p, sizeof(eals::EvalTriple) * got, cudaMemcpyDeviceToHost));
  std::sort(tr.begin(), tr.end(), [](const eals::EvalTriple& a, const eals::EvalTriple& b) {
    return a.slot != b.slot ? a.slot < b.slot : a.item < b.item;
  });
  out.own_key.resize(tr.size()); out.own_val.resize(tr.size());
  for (size_t t = 0; t < tr.size(); t++) {
    out.own_key[t] = ((unsigned long long)(uint32_t)tr[t].slot << 32) | (uint32_t)tr[t].item;
    out.own_val[t] = tr[t].key;
  }
  out.key = out.own_key.data(); out.val = out.own_val.data(); out.n_keys = tr.size();
  return EALS_OK;
}

// ---- scan engine 2: tcgen05 filter + exact re-score of the candidates (eval_tc.cuh) ---------------------
typedef CUresult (*TensorMapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                      const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int make_half_map(CUtensorMap* map, const __half* base, size_t rows, int KP) {
  static TensorMapEncodeFn encode = nullptr;
  if (!encode) {
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", (void**)&encode, cudaEnableDefault, &q) != cudaSuccess || !encode)
      return fail(EALS_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  }
  const cuuint64_t gdim[2] = {(cuuint64_t)KP, (cuuint64_t)std::max<size_t>(rows, 1)};
  const cuuint64_t gstr[1] = {(cuuint64_t)KP * 2};
  const cuuint32_t box[2] = {(cuuint32_t)eals::tc::kKC, (cuuint32_t)eals::tc::kTM}, estr[2] = {1, 1};
  const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, (void*)base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(EALS_ERR_CUDA, "cuTensorMapEncodeTiled -> %d", (int)r);
  return EALS_OK;
}

template <int NKC, int MODE>
int launch_filter(eals_model* m, const CUtensorMap& mapU, const CUtensorMap& mapV, const eals::tc::TcArgs& a) {
  using C = eals::tc::Cfg<NKC>;
  auto kern = eals::tc::eval_filter_kernel<NKC, MODE>;
  const size_t smem = MODE != 0 ? C::kSmemEmit : C::kSmem;
  CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // one CTA per SM: the kernel cuts the item range into chunks when there are fewer user tiles than SMs
  kern<<<m->sm_count, eals::tc::kThreads, smem, m->stream>>>(mapU, mapV, a);
  return check_launch(m);
}
template <int MODE>
int launch_filter_k(eals_model* m, int nkc, const CUtensorMap& mapU, const CUtensorMap& mapV, const eals::tc::TcArgs& a) {
  switch (nkc) {
    case 1: return launch_filter<1, MODE>(m, mapU, mapV, a);
    case 2: return launch_filter<2, MODE>(m, mapU, mapV, a);
    case 3: return launch_filter<3, MODE>(m, mapU, mapV, a);
    case 4: return launch_filter<4, MODE>(m, mapU, mapV, a);
  }
  return fail(EALS_ERR_UNSUPPORTED, "factors %d in the tensor-core evaluation", nkc * 64);
}

// survivors' triples out of the re-scored candidate pairs
__global__ void pairs_to_triples_kernel(const eals::tc::EvalPair* __restrict__ pairs, const unsigned long long* __restrict__ n_pairs,
                                        const int32_t* __restrict__ cnt_hi, const int32_t* __restrict__ cnt_exact, int topk,
                                        unsigned long long* __restrict__ out_key, int32_t* __restrict__ out_val,
                                        unsigned long long* __restrict__ n_out) {
  const unsigned long long n = *n_pairs;
  for (unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (unsigned long long)gridDim.x * blockDim.x) {
    const eals::tc::EvalPair pr = pairs[t];
    const bool keep = pr.key != 0 && cnt_hi[pr.slot] <= topk && cnt_exact[pr.slot] <= topk;
    // warp-aggregated append (tens of millions of keys at the 10M x 2M scale)
    const unsigned ballot = __ballot_sync(__activemask(), keep);
    if (!keep) continue;
    const int lane = threadIdx.x & 31, leader = __ffs(ballot) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(n_out, (unsigned long long)__popc(ballot));
    base = __shfl_sync(ballot, base, leader);
    const unsigned long long pos = base + __popc(ballot & ((1u << lane) - 1u));
    out_key[pos] = ((unsigned long long)(uint32_t)pr.slot << 32) | (uint32_t)pr.item;
    out_val[pos] = pr.key;
  }
}

__global__ void set_i32_kernel(int32_t* p, int32_t v) { *p = v; }

// ---- pieces shared by the filter passes of evaluate and recommend ----

// Lists of at least 128 users with at most 256 factors run on the tcgen05 filter.  EALS_EVAL_SCALAR=1 keeps every
// list on the exact engine, the one the filter is tested against.
bool use_tc_engine(const eals_model* m, int n) {
  return n >= 128 && m->K <= 256 && !(getenv("EALS_EVAL_SCALAR") && getenv("EALS_EVAL_SCALAR")[0] == '1');
}

// Key bits of a slot below n (at least 1), for the radix sorts by slot.
int slot_bits(int n) { int bits = 1; while ((1ll << bits) < n) bits++; return bits; }

// The pair buffer's first and hard cap: the caller's defaults unless EALS_EVAL_PAIR_CAP (at least 16) or
// EALS_EVAL_PAIR_HARD_CAP is set, and the hard cap at most max_hard.
void read_pair_caps(unsigned long long& cap, unsigned long long& hard_cap, unsigned long long max_hard) {
  if (const char* e = getenv("EALS_EVAL_PAIR_CAP")) cap = std::max<unsigned long long>(16, strtoull(e, nullptr, 10));
  if (const char* e = getenv("EALS_EVAL_PAIR_HARD_CAP")) hard_cap = strtoull(e, nullptr, 10);
  hard_cap = std::min(hard_cap, max_hard);
}

// The item blocks of a filter pass, tiles [it0, it1) from item i0 on.  The first block holds EALS_EVAL_FIRST_CHUNK
// items (default 32768, at least one tile), each next one 4x as many up to 262144: the fp16 block stays in the L2
// while all user tiles pass over it.  Every block ends on a tile boundary.
struct ItemBlocks {
  int64_t n_items, i0, i1 = 0, len = 32768;
  int it0 = 0, it1 = 0;
  ItemBlocks(int N, int64_t start) : n_items(N), i0(start) {
    if (const char* e = getenv("EALS_EVAL_FIRST_CHUNK")) len = std::max<int64_t>(eals::tc::kTN, atoll(e));
    tiles();
  }
  void next() { i0 = (int64_t)it1 * eals::tc::kTN; len = std::min<int64_t>(len * 4, 262144); tiles(); }
  void tiles() { i1 = std::min(n_items, i0 + len); it0 = (int)(i0 / eals::tc::kTN); it1 = (int)((i1 + eals::tc::kTN - 1) / eals::tc::kTN); }
};

// One device-wide cub call f(tmp, bytes): the size query, grow-only scratch in ws.cub_tmp, the run (one launch).
template <typename F>
int cub_call(eals_model* m, const char* what, F f) {
  eals_eval_ws& ws = eval_ws(m);
  size_t bytes = 0;
  f(nullptr, bytes);
  OK(ws.cub_tmp.reserve(bytes + 16));
  if (f(ws.cub_tmp.p, bytes) != cudaSuccess) return fail(EALS_ERR_CUDA, "%s", what);
  m->launches++;
  return EALS_OK;
}

// Working-set compaction: out = the entries of `in` (nullptr: the slots 0 .. n-1) whose ws.flags are set, their
// number to d_count.  Only enqueues work; the caller decides whether the host needs the count.
int select_flagged(eals_model* m, const int32_t* in, int n, int32_t* out, int32_t* d_count) {
  uint8_t* flags = eval_ws(m).flags.p;
  auto run = [&](auto first) {
    return cub_call(m, "working-set compaction", [&](void* tmp, size_t& bytes) {
      return cub::DeviceSelect::Flagged(tmp, bytes, first, flags, out, d_count, n, m->stream); });
  };
  return in ? run(in) : run(thrust::counting_iterator<int32_t>(0));
}

// The working list of a filter pass: `cur` (nullptr: the slots 0 .. n-1) and the two buffers it alternates between.
struct WorkList {
  const int32_t* cur = nullptr;
  int32_t *next, *spare;
  explicit WorkList(eals_eval_ws& ws) : next(ws.list_a.p), spare(ws.list_b.p) {}
};

// Compaction of the working list: its first n entries whose ws.flags are set (the caller's flag kernel) -> wl.next,
// their number -> d_n, their fp16 rows ws.Uh -> ws.W; wl.next becomes the list.  Only enqueues work: the count stays
// on the device for the next filter launch.
int compact_list(eals_model* m, WorkList& wl, int n, int32_t* d_n) {
  eals_eval_ws& ws = eval_ws(m);
  const int KP = (m->K + eals::tc::kKC - 1) / eals::tc::kKC * eals::tc::kKC;
  OK(select_flagged(m, wl.cur, n, wl.next, d_n));
  eals::tc::gather_rows_kernel<<<8 * m->sm_count, 256, 0, m->stream>>>(ws.Uh.p, KP, wl.next, d_n, ws.W.p);
  OK(check_launch(m));
  wl.cur = wl.next;
  std::swap(wl.next, wl.spare);
  return EALS_OK;
}

// Preparation of the tcgen05 filter for the rows X[d_rows[0 .. n)] (d_rows nullable: X[0 .. n); evaluate and
// recommend) against the catalogue Y [N][LD] (V, or a normalised U / V for similar): fp16 copies of Y in
// decreasing-norm order (ws.perm: rank -> row of Y) and of the query rows, their norms, the per-tile catalogue norms
// and the per-slot thresholds from `d_thr` (the exact gt score, or a user's k-th score).  Every call prepares its
// catalogue again, so nothing of one catalogue carries over to a call on another.
// The catalogue half (once per call of ranking_metrics, which prepares several chunks of rows against it) ...
int tc_prepare_items(eals_model* m, const double* Y, int N) {
  namespace tc = eals::tc;
  eals_eval_ws& ws = eval_ws(m);
  const int K = m->K, LD = m->LD;
  const int nkc = (K + tc::kKC - 1) / tc::kKC, KP = nkc * tc::kKC;
  const int n_tiles = (N + tc::kTN - 1) / tc::kTN;
  cudaStream_t st = m->stream;
  // ---- preparation: fp16 copies, norms, item order ----
  OK(ws.counters.reserve(4));
  OK(ws.keys.reserve((size_t)N)); OK(ws.keys_out.reserve((size_t)N)); OK(ws.ids.reserve((size_t)N)); OK(ws.perm.reserve((size_t)N));
  OK(ws.Vh.reserve((size_t)N * KP)); OK(ws.vn_hat.reserve((size_t)N)); OK(ws.vn_del.reserve((size_t)N)); OK(ws.vn_h.reserve((size_t)N));
  OK(ws.tile_norm.reserve((size_t)n_tiles));
  unsigned long long* d_vmax = ws.counters.p;
  CU(cudaMemsetAsync(ws.counters.p, 0, 4 * sizeof(unsigned long long), st));
  tc::absmax_kernel<<<4 * m->sm_count, 256, 0, st>>>(Y, (size_t)N, K, LD, d_vmax);
  OK(check_launch(m));
  tc::item_sort_keys_kernel<<<(unsigned)(((size_t)N * 32 + 255) / 256), 256, 0, st>>>(Y, K, LD, N, ws.keys.p, ws.ids.p);
  OK(check_launch(m));
  OK(cub_call(m, "item norm sort", [&](void* tmp, size_t& bytes) {
    return cub::DeviceRadixSort::SortPairs(tmp, bytes, ws.keys.p, ws.keys_out.p, ws.ids.p, ws.perm.p, N, 0, 32, st); }));
  {
    tc::PrepOut o{ws.Vh.p, ws.vn_hat.p, ws.vn_del.p, ws.vn_h.p, nullptr};
    tc::prep_rows_kernel<false><<<(unsigned)(((size_t)N * 32 + 255) / 256), 256, 0, st>>>(Y, K, LD, KP, N, ws.perm.p, 0, d_vmax, o);
    OK(check_launch(m));
    tc::tile_norm_kernel<<<n_tiles, 32, 0, st>>>(ws.vn_h.p, ws.vn_del.p, N, n_tiles, ws.tile_norm.p);
    OK(check_launch(m));
  }
  return EALS_OK;
}

// ... and the row half: fp16 copies of X[d_rows[0 .. n)], their norms and the per-slot thresholds.
int tc_prepare_rows(eals_model* m, int n, const double* X, const int32_t* d_rows, const double* d_thr) {
  namespace tc = eals::tc;
  eals_eval_ws& ws = eval_ws(m);
  const int K = m->K, LD = m->LD;
  const int nkc = (K + tc::kKC - 1) / tc::kKC, KP = nkc * tc::kKC;
  cudaStream_t st = m->stream;
  OK(ws.Uh.reserve((size_t)n * KP)); OK(ws.W.reserve(((size_t)n + 2 * tc::kTM) * KP));
  OK(ws.un_hat.reserve((size_t)n)); OK(ws.un_del.reserve((size_t)n)); OK(ws.un_h.reserve((size_t)n)); OK(ws.exps.reserve((size_t)n));
  OK(ws.sp0.reserve((size_t)n)); OK(ws.sp1.reserve((size_t)n));
  OK(ws.cnt.reserve((size_t)n)); OK(ws.cnt_exact.reserve((size_t)n));
  OK(ws.list_a.reserve((size_t)n)); OK(ws.list_b.reserve((size_t)n)); OK(ws.flags.reserve((size_t)n));
  OK(ws.scalars.reserve(8));
  const unsigned long long* d_vmax = ws.counters.p;   // max |V|, from tc_prepare_items
  {
    tc::PrepOut o{ws.Uh.p, ws.un_hat.p, ws.un_del.p, ws.un_h.p, ws.exps.p};
    tc::prep_rows_kernel<true><<<(unsigned)(((size_t)n * 32 + 255) / 256), 256, 0, st>>>(X, K, LD, KP, n, d_rows, 0, d_vmax, o);
    OK(check_launch(m));
    const double gamma = (double)KP * (1.0 / 2097152.0);   // KP * 2^-21
    tc::slot_params_kernel<<<(n + 255) / 256, 256, 0, st>>>(d_thr, ws.exps.p, d_vmax, ws.un_hat.p, ws.un_del.p, ws.un_h.p, n, gamma, ws.sp0.p, ws.sp1.p);
    OK(check_launch(m));
  }
  return EALS_OK;
}

int tc_prepare(eals_model* m, const double* Y, int N, int n, const double* X, const int32_t* d_rows, const double* d_thr) {
  OK(tc_prepare_items(m, Y, N));
  return tc_prepare_rows(m, n, X, d_rows, d_thr);
}

// What a count pass hands back: the survivors of the certain count (a device list of n_cand slots) and their `pairs`
// emitted pairs in ws.pairs (that count also at d_pairs on the device); or `overflow` when the pairs would exceed the
// hard cap: the filter is not filtering, and the caller's exact engine answers instead.
struct CountPass {
  const int32_t* surv = nullptr;
  int n_cand = 0;
  unsigned long long pairs = 0;
  unsigned long long* d_pairs = nullptr;
  bool overflow = false;
};

// Count-and-emit pass of the tcgen05 filter over n slots that tc_prepare_rows has prepared (evaluate, ranking
// metrics).  MODE 0 walks the item blocks and counts, per slot, the items certainly ahead of its threshold into
// ws.cnt; between blocks the working set keeps the slots whose count is below their limit, lim[s] (lim nullable:
// lim_all for every slot), compacted on the device.  compact_first also compacts once before the first block, for
// slots that start at their limit; `timed` times the first block into ws.blk0.  The survivors then go through the
// filter in emission mode EMIT over the whole catalogue: a first buffer of pairs_per_cand pairs per survivor
// (2^20 .. 2^27), then one more attempt at the exact size; beyond the hard cap (2^30 pairs, 16 GB) it overflows.
// Both caps as read_pair_caps gives them, the first never above the hard one.
// ws.cnt_exact is zeroed for the caller's re-score of the pairs.
template <int EMIT>
int count_pass(eals_model* m, int n, const int32_t* lim, int lim_all, bool compact_first, bool timed, unsigned long long pairs_per_cand,
               StageTimer& tm, CountPass& out) {
  namespace tc = eals::tc;
  eals_eval_ws& ws = eval_ws(m);
  const int K = m->K, N = m->N;
  const int nkc = (K + tc::kKC - 1) / tc::kKC, KP = nkc * tc::kKC;
  const int n_tiles = (N + tc::kTN - 1) / tc::kTN;
  cudaStream_t st = m->stream;
  out = CountPass{};
  CU(cudaMemsetAsync(ws.cnt.p, 0, sizeof(int32_t) * n, st));
  CU(cudaMemsetAsync(ws.cnt_exact.p, 0, sizeof(int32_t) * n, st));
  CUtensorMap mapV, mapU0, mapW;
  OK(make_half_map(&mapV, ws.Vh.p, (size_t)N, KP));
  OK(make_half_map(&mapU0, ws.Uh.p, (size_t)n, KP));
  OK(make_half_map(&mapW, ws.W.p, (size_t)n + 2 * tc::kTM, KP));
  int32_t* d_n = ws.scalars.p;          // size of the working list
  set_i32_kernel<<<1, 1, 0, st>>>(d_n, n);
  OK(check_launch(m));

  // ---- MODE 0 over L2-sized item blocks, working set compacted on the device between them ----
  tc::TcArgs a{};
  a.sp0 = ws.sp0.p; a.sp1 = ws.sp1.p; a.tile_norm = ws.tile_norm.p; a.n_items = N; a.cnt_hi = ws.cnt.p; a.perm = ws.perm.p;
  WorkList wl(ws);
  auto compact = [&](void) -> int {     // slots of the list still below their limit
    tc::below_limit_flags_kernel<<<(n + 255) / 256, 256, 0, st>>>(wl.cur, d_n, n, ws.cnt.p, lim, lim_all, ws.flags.p);
    OK(check_launch(m));
    return compact_list(m, wl, n, d_n);
  };
  if (compact_first) OK(compact());
  for (ItemBlocks blk(N, 0); blk.i0 < N; blk.next()) {
    a.act = wl.cur; a.n_act = d_n; a.it0 = blk.it0; a.it1 = blk.it1;
    const bool first_block = timed && blk.i0 == 0;
    if (first_block) OK(ws.blk0.start(st));
    OK(launch_filter_k<0>(m, nkc, wl.cur ? mapW : mapU0, mapV, a));
    if (first_block) OK(ws.blk0.stop(st, n, std::min<int64_t>(N, (int64_t)a.it1 * tc::kTN)));
    OK(compact());
    if (tm.on) {
      int left = 0;
      cudaMemcpy(&left, d_n, sizeof(int), cudaMemcpyDeviceToHost);
      char what[96];
      snprintf(what, sizeof(what), "filter: items [%lld, %lld) -> %d left", (long long)blk.i0, (long long)blk.i1, left);
      tm.lap(what);
    }
  }
  // ---- emission for the survivors ----
  out.surv = wl.cur;
  out.d_pairs = ws.counters.p + 1;
  CU(cudaMemcpyAsync(&out.n_cand, d_n, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  if (out.n_cand == 0) return EALS_OK;
  unsigned long long cap = std::min<unsigned long long>(1ull << 27, std::max<unsigned long long>(1ull << 20, pairs_per_cand * (unsigned long long)out.n_cand));
  unsigned long long hard_cap = 1ull << 30;
  read_pair_caps(cap, hard_cap, ~0ull);
  cap = std::min(cap, hard_cap);
  unsigned long long& got = out.pairs;
  for (int attempt = 0; attempt < 2; attempt++) {
    OK(ws.pairs.reserve((size_t)cap));
    CU(cudaMemsetAsync(out.d_pairs, 0, sizeof(unsigned long long), st));
    a.act = wl.cur; a.n_act = d_n; a.it0 = 0; a.it1 = n_tiles;
    a.pairs = ws.pairs.p; a.n_pairs = out.d_pairs; a.cap_pairs = cap;
    OK(launch_filter_k<EMIT>(m, nkc, mapW, mapV, a));
    CU(cudaMemcpyAsync(&got, out.d_pairs, sizeof(got), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (got <= cap) break;
    if (attempt == 1 || got > hard_cap) { out.overflow = true; return EALS_OK; }
    cap = got;
  }
  tm.lap("filter: candidate emission");
  return EALS_OK;
}

// Fills `out` and m->eval_stats (engine 1), or returns with neither touched when the pair list overflows.
int scan_tc(eals_model* m, int n, const int32_t* d_users, const double* d_gts, int topk, bool want_triples, ScanResult& out) {
  namespace tc = eals::tc;
  eals_eval_ws& ws = eval_ws(m);
  StageTimer tm;
  const int K = m->K, LD = m->LD;
  cudaStream_t st = m->stream;
  OK(tc_prepare(m, m->V, m->N, n, m->U, d_users, d_gts));
  tm.lap("eval: fp16 copies, norms, item order");
  // a user is decided once its certain count exceeds topK (limit topK + 1, kept from overflowing); the candidates
  // go through MODE 1, which also emits the pairs whose truncated key may be non-zero
  CountPass cp;
  OK(count_pass<1>(m, n, nullptr, (int)std::min<int64_t>((int64_t)topk + 1, INT32_MAX), false, true, 1024, tm, cp));
  if (cp.overflow) return EALS_OK;
  const int n_cand = cp.n_cand;
  const unsigned long long got = cp.pairs;
  if (got) {
    tc::eval_rescore_kernel<<<16 * m->sm_count, 128, 0, st>>>(m->U, m->V, K, LD, d_users, 0, d_gts, ws.pairs.p, cp.d_pairs, got,
                                                              ws.cnt_exact.p);
    OK(check_launch(m));
  }
  tm.lap("eval: exact re-score");
  // candidates and their exact counts (a few per cent of the users at most); everybody else is decided
  std::vector<int32_t> cand((size_t)n_cand), cand_cnt((size_t)n_cand);
  unsigned long long n_tr = 0;
  if (n_cand > 0) {
    OK(ws.active.reserve((size_t)n_cand));
    eals::gather_i32_kernel<<<(n_cand + 255) / 256, 256, 0, st>>>(ws.cnt_exact.p, cp.surv, n_cand, ws.active.p);
    OK(check_launch(m));
    CU(cudaMemcpyAsync(cand.data(), cp.surv, sizeof(int32_t) * n_cand, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(cand_cnt.data(), ws.active.p, sizeof(int32_t) * n_cand, cudaMemcpyDeviceToHost, st));
  }
  if (want_triples && got) {
    OK(ws.tkey.reserve((size_t)got)); OK(ws.tval.reserve((size_t)got));
    unsigned long long* d_nt = ws.counters.p + 2;
    pairs_to_triples_kernel<<<8 * m->sm_count, 256, 0, st>>>(ws.pairs.p, cp.d_pairs, ws.cnt.p, ws.cnt_exact.p, topk, ws.tkey.p, ws.tval.p, d_nt);
    OK(check_launch(m));
    CU(cudaMemcpyAsync(&n_tr, d_nt, sizeof(n_tr), cudaMemcpyDeviceToHost, st));
  }
  CU(cudaStreamSynchronize(st));
  out.surv_slot.clear(); out.surv_cnt.clear();
  for (int c = 0; c < n_cand; c++)
    if (cand_cnt[(size_t)c] <= topk) { out.surv_slot.push_back(cand[(size_t)c]); out.surv_cnt.push_back(cand_cnt[(size_t)c]); }
  out.key = nullptr; out.val = nullptr; out.n_keys = 0;
  if (n_tr) {   // (slot, item) order on the device, then one copy each into pinned host memory
    if (n_tr >= 0x7fffffffull) return fail(EALS_ERR_UNSUPPORTED, "too many ranking keys (%llu)", n_tr);
    OK(ws.tkey_out.reserve((size_t)n_tr)); OK(ws.tval_out.reserve((size_t)n_tr));
    const int end_bit = 32 + slot_bits(n);
    OK(cub_call(m, "ranking key sort", [&](void* tmp, size_t& bytes) {
      return cub::DeviceRadixSort::SortPairs(tmp, bytes, ws.tkey.p, ws.tkey_out.p, ws.tval.p, ws.tval_out.p, (int)n_tr, 0, end_bit, st); }));
    OK(ws.host.reserve((size_t)n_tr * 12 + 64));
    unsigned long long* hk = reinterpret_cast<unsigned long long*>(ws.host.p);
    int32_t* hv = reinterpret_cast<int32_t*>(ws.host.p + (size_t)n_tr * 8);
    CU(cudaMemcpyAsync(hk, ws.tkey_out.p, sizeof(unsigned long long) * n_tr, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(hv, ws.tval_out.p, sizeof(int32_t) * n_tr, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    out.key = hk; out.val = hv; out.n_keys = (size_t)n_tr;
  }
  tm.lap("eval: counts + keys to host");
  if (getenv("EALS_VERBOSE") && getenv("EALS_VERBOSE")[0] == '1')
    fprintf(stderr, "[eals] evaluate (tcgen05 filter): %d users, %d candidates after the certain count, %llu pairs re-scored exactly, %llu keys\n",
            n, n_cand, got, n_tr);
  BlockTiming blk0;
  OK(ws.blk0.read(blk0));
  m->eval_stats = EvalStats{1, n_cand, (long long)got, blk0};
  return EALS_OK;
}

int evaluate_slots(eals_model* m, const std::vector<int32_t>& users_h, const int32_t* gt_slot_h, int topk,
                   int mode, double sums[3], double* hr, double* ndcg, double* prec, int32_t* count_larger) {
  const int n = (int)users_h.size();
  sums[0] = sums[1] = sums[2] = 0;
  m->eval_stats = EvalStats{};   // scan_tc fills them when it answers; the exact engine leaves them zero
  if (n == 0) return EALS_OK;
  eals_eval_ws& ws = eval_ws(m);
  const int K = m->K, LD = m->LD, N = m->N;
  OK(ws.users.reserve((size_t)n)); OK(ws.gt.reserve((size_t)n)); OK(ws.gts.reserve((size_t)n));
  CU(cudaMemcpyAsync(ws.gt.p, gt_slot_h, sizeof(int32_t) * n, cudaMemcpyHostToDevice, m->stream));
  CU(cudaMemcpyAsync(ws.users.p, users_h.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, m->stream));
  eals::eval_gt_score_kernel<<<(n + 127) / 128, 128, 0, m->stream>>>(m->U, m->V, ws.gt.p, ws.users.p, 0, n, K, LD, ws.gts.p);
  OK(check_launch(m));
  ScanResult res;
  const bool want_triples = mode != EALS_EVAL_EXACT;
  if (use_tc_engine(m, n)) OK(scan_tc(m, n, ws.users.p, ws.gts.p, topk, want_triples, res));
  if (m->eval_stats.engine == 0) OK(scan_exact(m, n, ws.users.p, ws.gts.p, topk, want_triples, res));
  StageTimer tm_host;

  // Only the survivors can score; all other users get (0, 0, 0) and count_larger = topK + 1.
  const size_t ns = res.surv_slot.size();
  std::vector<int> pos(ns, -1);
  if (mode == EALS_EVAL_EXACT) {
    for (size_t t = 0; t < ns; t++)
      if (res.surv_cnt[t] < topk) pos[t] = res.surv_cnt[t];
  } else {
    // Replay of the reference's ranking (MF_fastALS.cpp:641-656) with the real libstdc++ partial_sort_copy,
    // the survivors spread over the host threads; a survivor's (item, key) stream is its range of the sorted
    // key arrays.
    const unsigned long long* key = res.key;
    const int32_t* val = res.val;
    const size_t nk = res.n_keys;
    parallel_chunks((int64_t)ns, nullptr, [&](int, int64_t b0, int64_t b1) {
      std::vector<std::pair<int, int>> nz;
      RankScratch scratch;
      for (int64_t t = b0; t < b1; t++) {
        const int s = res.surv_slot[(size_t)t];
        const unsigned long long lo = (unsigned long long)(uint32_t)s << 32;
        size_t q = nk ? (size_t)(std::lower_bound(key, key + nk, lo) - key) : 0;
        nz.clear();
        for (; q < nk && (key[q] >> 32) == (unsigned long long)(uint32_t)s; q++)
          nz.emplace_back((int)(key[q] & 0xffffffffu), val[q]);
        pos[(size_t)t] = reference_rank(nz, N, topk, gt_slot_h[s], scratch);
      }
    }, 256);
  }
  if (hr) std::fill(hr, hr + n, 0.0);
  if (ndcg) std::fill(ndcg, ndcg + n, 0.0);
  if (prec) std::fill(prec, prec + n, 0.0);
  if (count_larger) std::fill(count_larger, count_larger + n, topk + 1);
  for (size_t t = 0; t < ns; t++) {     // ascending slot: the same summation order as a loop over all users
    const int s = res.surv_slot[t];
    double r0 = 0, r1 = 0, r2 = 0;
    if (pos[t] >= 0) { r0 = 1; r1 = metric_ndcg(pos[t]); r2 = 1.0 / (pos[t] + 1); }
    if (hr) hr[s] = r0;
    if (ndcg) ndcg[s] = r1;
    if (prec) prec[s] = r2;
    if (count_larger) count_larger[s] = res.surv_cnt[t];
    sums[0] += r0; sums[1] += r1; sums[2] += r2;
  }
  tm_host.lap("eval: host ranking replay + metrics");
  return EALS_OK;
}

// ---- top-k retrieval (recommend.cuh) --------------------------------------------------------------------
namespace rec = eals::rec;

// What the engines answer: slot s asks for the top-k rows of the catalogue Y [nY][LD] for row rows[s] of X (rows
// nullable: row s), its excluded catalogue rows being row (that row - ex_base) of the CSR ex_ptr / ex_idx (ex_ptr
// nullable: none).  recommend: the model's U, the users, the owned train rows, catalogue V; recommend_vectors: the
// query vectors copied to [n][LD], the identity, the caller's exclusion lists, catalogue V; similar: the normalised
// query rows copied to [n][LD], the identity, each query's own id, the normalised U or V.
struct RecQuery {
  const double* X;
  const int32_t* rows;
  const int64_t* ex_ptr;
  const int32_t* ex_idx;
  int ex_base;
  const double* Y;
  int nY;
  RecQuery from(int s0, int LD) const {   // the same query for the slots s0 ..
    RecQuery q = *this;
    if (rows) q.rows += s0;
    else { q.X += (size_t)s0 * LD; if (q.ex_ptr) q.ex_ptr += s0; }
    return q;
  }
};

rec::MergeArgs rec_args(eals_model* m, const RecQuery& q, int k) {
  eals_eval_ws& ws = eval_ws(m);
  rec::MergeArgs a{};
  a.U = q.X; a.V = q.Y; a.K = m->K; a.LD = m->LD; a.users = q.rows; a.k = k;
  a.top_s = ws.top_s.p; a.top_i = ws.top_i.p; a.thr = ws.thr.p;
  a.ptr = q.ex_ptr; a.idx = q.ex_idx; a.row_base = q.ex_base;
  return a;
}

int rec_reset(eals_model* m, int n, int k) {
  eals_eval_ws& ws = eval_ws(m);
  rec::rec_init_kernel<<<4 * m->sm_count, 256, 0, m->stream>>>(ws.top_s.p, ws.top_i.p, (size_t)n * k, ws.thr.p, n);
  return check_launch(m);
}

// the listed slots (list nullable: slots 0 .. n_list-1) against the items order[r0 .. r1), every score exact
int rec_merge_exact(eals_model* m, rec::MergeArgs a, const int32_t* list, int n_list, const int32_t* order, int r0, int r1) {
  if (n_list <= 0 || r1 <= r0) return EALS_OK;
  a.list = list; a.order = order; a.r0 = r0; a.r1 = r1;
  rec::rec_merge_kernel<rec::SRC_EXACT><<<n_list, rec::kThreads, 0, m->stream>>>(a);
  return check_launch(m);
}

// Engine 1: exact fp64 scores of every item.  Short lists, the reference of the tensor-core engine
// (EALS_EVAL_SCALAR=1) and its fall-back.
int rec_exact(eals_model* m, int n, const RecQuery& q, int k) {
  OK(rec_reset(m, n, k));
  return rec_merge_exact(m, rec_args(m, q, k), nullptr, n, nullptr, 0, q.nY);
}

// Engine 2: tcgen05 filter.  Seed: the highest-norm items scored exactly (extended tile by tile for users whose
// list is not full).  Then item blocks in norm order: the filter emits (user, item) only where acc >= t^ - E
// (t = the user's current k-th score), the pairs are re-scored exactly and merged, t rises, and a user leaves
// the working set once a Cauchy-Schwarz bound on every remaining item is below t (DESIGN.md §3.5).  Fills `stats`
// (engine 1) when it answers; leaves them as they are when the filter stops filtering.
int rec_tc(eals_model* m, int n, const RecQuery& q, int k, RecStats& stats) {
  namespace tc = eals::tc;
  eals_eval_ws& ws = eval_ws(m);
  StageTimer tm;
  const int K = m->K, N = q.nY;
  const int nkc = (K + tc::kKC - 1) / tc::kKC, KP = nkc * tc::kKC;
  const int n_tiles = (N + tc::kTN - 1) / tc::kTN;
  const int ut = nkc <= 2 ? 2 : 1;
  cudaStream_t st = m->stream;
  OK(rec_reset(m, n, k));
  OK(tc_prepare(m, q.Y, N, n, q.X, q.rows, ws.thr.p));
  const double gamma = (double)KP * (1.0 / 2097152.0);
  auto params = [&]() -> int {   // per-slot filter thresholds from the current k-th scores
    tc::slot_params_kernel<<<(n + 255) / 256, 256, 0, st>>>(ws.thr.p, ws.exps.p, ws.counters.p, ws.un_hat.p, ws.un_del.p, ws.un_h.p, n,
                                                            gamma, ws.sp0.p, ws.sp1.p);
    return check_launch(m);
  };
  // rem[t] >= max |v^| over the items of tiles t.. (|v^| <= |vh| + |dv|), rounded up; rem[n_tiles] = 0
  std::vector<float2> tn((size_t)n_tiles);
  CU(cudaMemcpyAsync(tn.data(), ws.tile_norm.p, sizeof(float2) * n_tiles, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  std::vector<float> rem((size_t)n_tiles + 1, 0.f);
  for (int t = n_tiles - 1; t >= 0; t--)
    rem[(size_t)t] = std::max(rem[(size_t)t + 1], std::nextafter(tn[(size_t)t].x + tn[(size_t)t].y, std::numeric_limits<float>::infinity()));
  int32_t* d_n = ws.scalars.p;          // [0]: working-list size, [1]: scratch, [2]: size of a chunk of the list
  const rec::MergeArgs base = rec_args(m, q, k);

  // ---- seed ----
  const int seed = (int)std::min<int64_t>(N, ((int64_t)k + tc::kTN - 1) / tc::kTN * tc::kTN);
  OK(rec_merge_exact(m, base, nullptr, n, ws.perm.p, 0, seed));
  {
    const int32_t* lst = nullptr;
    int nl = n, r_end = seed, step = tc::kTN;
    int32_t* bufs[2] = {ws.list_a.p, ws.list_b.p};
    for (int b = 0; nl > 0 && r_end < N; b ^= 1) {
      rec::rec_unfilled_flags_kernel<<<(nl + 255) / 256, 256, 0, st>>>(lst, nullptr, nl, ws.thr.p, ws.flags.p);
      OK(check_launch(m));
      OK(select_flagged(m, lst, nl, bufs[b], d_n));
      CU(cudaMemcpyAsync(&nl, d_n, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));
      lst = bufs[b];
      const int r1 = (int)std::min<int64_t>(N, (int64_t)r_end + step);
      OK(rec_merge_exact(m, base, lst, nl, ws.perm.p, r_end, r1));
      r_end = r1;
      step *= 2;
    }
  }
  tm.lap("recommend: prep + exact seed");

  // ---- item blocks ----
  WorkList wl(ws);
  int n_act = n;
  auto compact = [&](int it_next) -> int {   // users that may still gain an item from tile it_next on
    OK(params());
    rec::rec_keep_flags_kernel<<<(n_act + 255) / 256, 256, 0, st>>>(wl.cur, nullptr, n_act, ws.un_hat.p, ws.sp0.p, ws.thr.p,
                                                                    rem[(size_t)it_next], ws.flags.p);
    OK(check_launch(m));
    OK(compact_list(m, wl, n_act, d_n));
    CU(cudaMemcpyAsync(&n_act, d_n, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return EALS_OK;
  };
  OK(compact(seed / tc::kTN));
  CUtensorMap mapV;
  OK(make_half_map(&mapV, ws.Vh.p, (size_t)N, KP));
  tc::TcArgs a{};
  a.sp0 = ws.sp0.p; a.sp1 = ws.sp1.p; a.tile_norm = ws.tile_norm.p; a.n_items = N; a.perm = ws.perm.p; a.n_act = d_n + 2;
  unsigned long long* d_np = ws.counters.p + 1;
  unsigned long long cap = 1ull << 24, hard_cap = 1ull << 28;
  read_pair_caps(cap, hard_cap, 0x7fffffffull);   // the sort and run-length encoding of the pairs count in int
  cap = std::min(cap, hard_cap);
  const int quantum = ut * tc::kTM;
  int chunk = std::max(quantum, (n_act + quantum - 1) / quantum * quantum);
  RecStats s;
  s.left1 = n_act;
  bool first = true;
  for (ItemBlocks blk(N, seed); blk.i0 < N && n_act > 0; blk.next()) {
    a.it0 = blk.it0; a.it1 = blk.it1;
    for (int p0 = 0; p0 < n_act;) {
      const int nc = std::min(chunk, n_act - p0);
      set_i32_kernel<<<1, 1, 0, st>>>(d_n + 2, nc);
      OK(check_launch(m));
      CUtensorMap mapW;
      OK(make_half_map(&mapW, ws.W.p + (size_t)p0 * KP, (size_t)(n + 2 * tc::kTM - p0), KP));
      OK(ws.pairs.reserve((size_t)cap));
      a.act = wl.cur + p0; a.pairs = ws.pairs.p; a.n_pairs = d_np; a.cap_pairs = cap;
      CU(cudaMemsetAsync(d_np, 0, sizeof(unsigned long long), st));
      const bool timed = first && p0 == 0 && nc == n_act;
      if (timed) OK(ws.blk0.start(st));
      OK(launch_filter_k<2>(m, nkc, mapW, mapV, a));
      if (timed) OK(ws.blk0.stop(st, nc, std::min<int64_t>(N, (int64_t)a.it1 * tc::kTN) - blk.i0));
      unsigned long long got = 0;
      CU(cudaMemcpyAsync(&got, d_np, sizeof(got), cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));
      if (got > cap) {
        if (got <= hard_cap) { cap = got; continue; }            // a larger buffer, same chunk
        if (nc > quantum) {                                       // fewer users per pass
          chunk = std::max<long long>(quantum, (long long)((double)nc * ((double)hard_cap / (double)got) / 2) / quantum * quantum);
          continue;
        }
        return EALS_OK;                                           // the filter is not filtering: exact engine instead
      }
      if (timed) OK(ws.blk0.read(s.blk0));
      if (got) {
        OK(ws.pscore.reserve((size_t)got)); OK(ws.pkey.reserve((size_t)got)); OK(ws.pkey_out.reserve((size_t)got));
        OK(ws.pval.reserve((size_t)got)); OK(ws.pval_out.reserve((size_t)got));
        OK(ws.run_slot.reserve((size_t)got)); OK(ws.run_cnt.reserve((size_t)got)); OK(ws.run_off.reserve((size_t)got));
        rec::rec_rescore_kernel<tc::EvalPair><<<16 * m->sm_count, 128, 0, st>>>(q.X, q.Y, K, m->LD, q.rows, ws.pairs.p, got,
                                                                               ws.pscore.p, ws.pkey.p, ws.pval.p);
        OK(check_launch(m));
        const int ng = (int)got, end_bit = slot_bits(n);
        OK(cub_call(m, "candidate sort", [&](void* tmp, size_t& bytes) {
          return cub::DeviceRadixSort::SortPairs(tmp, bytes, ws.pkey.p, ws.pkey_out.p, ws.pval.p, ws.pval_out.p, ng, 0, end_bit, st); }));
        OK(cub_call(m, "candidate runs", [&](void* tmp, size_t& bytes) {
          return cub::DeviceRunLengthEncode::Encode(tmp, bytes, ws.pkey_out.p, ws.run_slot.p, ws.run_cnt.p, d_n + 1, ng, st); }));
        int n_runs = 0;
        CU(cudaMemcpyAsync(&n_runs, d_n + 1, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        OK(cub_call(m, "candidate offsets", [&](void* tmp, size_t& bytes) {
          return cub::DeviceScan::ExclusiveSum(tmp, bytes, ws.run_cnt.p, ws.run_off.p, n_runs, st); }));
        rec::MergeArgs ma = base;
        ma.run_slot = reinterpret_cast<const int32_t*>(ws.run_slot.p); ma.run_off = ws.run_off.p; ma.run_cnt = ws.run_cnt.p;
        ma.pos_pair = ws.pval_out.p; ma.pair_item = &ws.pairs.p[0].item; ma.pair_stride = 4; ma.pair_score = ws.pscore.p;
        rec::rec_merge_kernel<rec::SRC_PAIRS><<<n_runs, rec::kThreads, 0, st>>>(ma);
        OK(check_launch(m));
      }
      s.pairs += (long long)got;
      p0 += nc;
    }
    OK(compact(a.it1));
    if (first) s.left1 = n_act;
    first = false;
    if (tm.on) {
      char what[96];
      snprintf(what, sizeof(what), "recommend: items [%lld, %lld) -> %d users left", (long long)blk.i0, (long long)a.it1 * tc::kTN, n_act);
      tm.lap(what);
    }
  }
  s.engine = 1; s.seed = seed;
  stats = s;
  return EALS_OK;
}

// The device bytes of the per-slot lists of a top-k call, and of a chunk of ranking_metrics' test entries:
// EALS_REC_LIST_BYTES, default 4 GiB.
size_t list_budget() {
  size_t bytes = (size_t)4 << 30;
  if (const char* e = getenv("EALS_REC_LIST_BYTES")) bytes = std::max<size_t>(1, strtoull(e, nullptr, 10));
  return bytes;
}

// The number of slots whose lists of k entries (12 bytes each) fit the budget, at least 1.
size_t list_slots(int k) { return std::max<size_t>(1, list_budget() / (12 * (size_t)k)); }

// Answers the slots 0 .. n-1 of q into items / scores (host or device memory as `space` says) and m->rec_stats.
int rec_answer(eals_model* m, int space, int n, const RecQuery& q, int k, int32_t* items, double* scores) {
  eals_eval_ws& ws = eval_ws(m);
  // Per-slot lists for at most `per` slots at a time: the slots are answered in balanced chunks, each a complete call
  // of an engine.
  const int max_per = (int)std::min<size_t>((size_t)n, list_slots(k));
  const int n_chunks = (n + max_per - 1) / max_per, per = (n + n_chunks - 1) / n_chunks;
  const size_t pk = (size_t)per * k;
  OK(ws.top_s.reserve(pk)); OK(ws.top_i.reserve(pk)); OK(ws.thr.reserve((size_t)per));
  const cudaMemcpyKind kind = space == EALS_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  RecStats total;
  for (int s0 = 0; s0 < n; s0 += per) {
    const int nc = std::min(per, n - s0);
    const size_t nck = (size_t)nc * k;
    const RecQuery qc = q.from(s0, m->LD);
    RecStats c;   // stays zero for a chunk of the exact engine
    if (use_tc_engine(m, nc)) OK(rec_tc(m, nc, qc, k, c));
    if (c.engine == 0) OK(rec_exact(m, nc, qc, k));
    if (s0 == 0) total = c;                              // engine, seed and the first block from chunk 0
    else { total.pairs += c.pairs; total.left1 += c.left1; }
    if (c.engine == 0) { total.engine = 0; total.seed = 0; }   // tcgen05 and its seed only if every chunk ran there
    rec::rec_finish_kernel<<<4 * m->sm_count, 256, 0, m->stream>>>(ws.top_i.p, nck);
    OK(check_launch(m));
    CU(cudaMemcpyAsync(items + (size_t)s0 * k, ws.top_i.p, sizeof(int32_t) * nck, kind, m->stream));
    if (scores) CU(cudaMemcpyAsync(scores + (size_t)s0 * k, ws.top_s.p, sizeof(double) * nck, kind, m->stream));
    CU(cudaStreamSynchronize(m->stream));   // the lists are reused by the next chunk
  }
  m->rec_stats = total;
  CU(cudaStreamSynchronize(m->stream));
  return EALS_OK;
}

// The argument checks of every top-k call (recommend, recommend_vectors, ranking_metrics with n = 0), on a model or a
// group alike.
int check_topk_args(int space, int n, int k) {
  if (n < 0) return fail(EALS_ERR_ARG, "n must be >= 0");
  if (k < 1 || k > rec::kMaxK) return fail(EALS_ERR_ARG, "k must be in [1, %d], got %d", rec::kMaxK, k);
  if (space != EALS_HOST && space != EALS_DEVICE) return fail(EALS_ERR_ARG, "space must be EALS_HOST or EALS_DEVICE");
  return EALS_OK;
}

// ... and what a model must have for them.
int rec_check_args(eals_model* m, int space, int n, int k) {
  OK(check_topk_args(space, n, k));
  if (!m->factors_set) return fail(EALS_ERR_STATE, "factors not initialised");
  if (m->K > rec::kMaxFactors) return fail(EALS_ERR_UNSUPPORTED, "recommend supports up to %d factors", rec::kMaxFactors);
  return EALS_OK;
}

// The first position of the device ids d_ids[0 .. n) outside [lo, hi) -> *pos and its id -> *id; *pos = -1 when every
// id is inside.  Synchronises.
int find_outside(eals_model* m, const int32_t* d_ids, int n, int lo, int hi, int* pos, int* id) {
  const int none = 0x7fffffff;
  int bad = none;
  CU(cudaMemcpyAsync(m->flags, &none, sizeof(int), cudaMemcpyHostToDevice, m->stream));
  rec::rec_check_users_kernel<<<(n + 255) / 256, 256, 0, m->stream>>>(d_ids, n, lo, hi, m->flags);
  OK(check_launch(m));
  CU(cudaMemcpyAsync(&bad, m->flags, sizeof(int), cudaMemcpyDeviceToHost, m->stream));
  CU(cudaStreamSynchronize(m->stream));
  *pos = -1;
  if (bad != none) {
    *pos = bad - 1;
    CU(cudaMemcpy(id, d_ids + (bad - 1), sizeof(int), cudaMemcpyDeviceToHost));
  }
  return EALS_OK;
}

int recommend_impl(eals_model* m, int space, int n, const int32_t* users, int k, int exclude, int32_t* items, double* scores) {
  if (!m || (n > 0 && (!users || !items))) return fail(EALS_ERR_ARG, "null argument");
  OK(rec_check_args(m, space, n, k));
  CU(cudaSetDevice(m->p.device));
  if (n == 0) return EALS_OK;
  if (space == EALS_HOST)
    for (int s = 0; s < n; s++) {
      if (users[s] < 0 || users[s] >= m->M) return fail(EALS_ERR_ARG, "user %d (position %d) outside [0, %d)", users[s], s, m->M);
      if (users[s] < m->ub || users[s] >= m->ue)
        return fail(EALS_ERR_ARG, "user %d (position %d) outside this model's users [%d, %d)", users[s], s, m->ub, m->ue);
    }
  eals_eval_ws& ws = eval_ws(m);
  OK(ws.users.reserve((size_t)n));
  OK(copy_in(ws.users.p, users, (size_t)n, space, m->stream));
  if (space == EALS_DEVICE) {
    int pos = -1, u = 0;
    OK(find_outside(m, ws.users.p, n, m->ub, m->ue, &pos, &u));
    if (pos >= 0) {
      if (u < 0 || u >= m->M) return fail(EALS_ERR_ARG, "user %d (position %d) outside [0, %d)", u, pos, m->M);
      return fail(EALS_ERR_ARG, "user %d (position %d) outside this model's users [%d, %d)", u, pos, m->ub, m->ue);
    }
  }
  RecQuery q{m->U, ws.users.p, nullptr, nullptr, 0, m->V, m->N};
  if (exclude) { q.ex_ptr = m->users.ptr; q.ex_idx = m->users.idx; q.ex_base = m->users.row_base; }
  return rec_answer(m, space, n, q, k, items, scores);
}

// ---- fold-in and top-k for arbitrary query vectors (DESIGN.md §3.6) ---------------------------------------------

// A CSR of n caller rows over the items (histories, exclusion lists), validated like the train matrix and bucketed
// into `s`.  Heavy rows may grow the shared scratch m->partials; a captured epoch graph refers to the old buffer, so
// it is captured again at the next eals_run_epochs.
int build_query_side(eals_model* m, Side& s, WsBuf<int>& check, int n, int space, const int64_t* ptr, const int32_t* idx,
                     const double* val, int begin = 0) {   // rows begin .. begin + n of ptr
  OK(check.reserve(8));
  const double* partials = m->partials;
  const int rc = build_side(m, s, begin, begin + n, m->N, space, ptr, idx, val, check.p);
  if (m->partials != partials) m->config_gen++;
  return rc;
}

// The argument checks of fold-in, on a model or a group alike.
int check_fold_in_args(int space, int n, int n_iter) {
  if (n < 0) return fail(EALS_ERR_ARG, "n must be >= 0");
  if (n_iter < 1) return fail(EALS_ERR_ARG, "n_iter must be >= 1, got %d", n_iter);
  if (space != EALS_HOST && space != EALS_DEVICE) return fail(EALS_ERR_ARG, "space must be EALS_HOST or EALS_DEVICE");
  return EALS_OK;
}

// n_iter passes of update_user_thread (MF_fastALS.cpp:243-322) over each history row, from `init` (NULL: zeros),
// with the model's V, SV, Wi and reg: the user CD kernels on a CdSide whose X is the workspace, no peers, no
// prediction cache (every pass recomputes the predictions), untimed.  Nothing of the model changes.
int fold_in_impl(eals_model* m, int space, int n, const int64_t* row_ptr, const int32_t* col_idx, const double* val,
                 const double* init, int n_iter, double* out) {
  if (!m || (n > 0 && (!row_ptr || !col_idx || !out))) return fail(EALS_ERR_ARG, "null argument");
  OK(check_fold_in_args(space, n, n_iter));
  if (!m->factors_set) return fail(EALS_ERR_STATE, "factors not initialised");
  CU(cudaSetDevice(m->p.device));
  if (n == 0) return EALS_OK;
  eals_eval_ws& ws = eval_ws(m);
  OK(build_query_side(m, ws.hist, ws.hist_check, n, space, row_ptr, col_idx, val));
  OK(ws.qx.reserve((size_t)n * m->LD));
  if (init) OK(upload_dense(m, ws.qx.p, init, (size_t)n, space));   // padding columns written as zeros
  else CU(cudaMemsetAsync(ws.qx.p, 0, sizeof(double) * (size_t)n * m->LD, m->stream));
  CdSide a{};
  a.ptr = ws.hist.ptr; a.idx = ws.hist.idx; a.val = ws.hist.val;
  a.X = ws.qx.p; a.Y = m->V; a.S = m->SV; a.Wi = m->Wi;
  a.row_base = 0; a.K = m->K; a.reg = m->p.reg;
  for (int it = 0; it < n_iter; it++) DISPATCH_LD(m->LD, OK((launch_cd<LD, true>(m, ws.hist, a, -1, false))));
  return download_dense(m, out, ws.qx.p, (size_t)n, space);
}

// Top-k of the query vectors Q[0 .. n) ([n][K]) with the same engines and contract as recommend (Q[s] stands in for
// U[u]), the items of row s of the optional CSR ex_ptr / ex_idx left out.
int recommend_vectors_impl(eals_model* m, int space, int n, const double* Q, const int64_t* ex_ptr, const int32_t* ex_idx,
                           int k, int32_t* items, double* scores) {
  if (!m || (n > 0 && (!Q || !items))) return fail(EALS_ERR_ARG, "null argument");
  if ((ex_ptr == nullptr) != (ex_idx == nullptr)) return fail(EALS_ERR_ARG, "ex_ptr and ex_idx must both be given or both be null");
  OK(rec_check_args(m, space, n, k));
  CU(cudaSetDevice(m->p.device));
  if (n == 0) return EALS_OK;
  eals_eval_ws& ws = eval_ws(m);
  if (ex_ptr) OK(build_query_side(m, ws.excl, ws.excl_check, n, space, ex_ptr, ex_idx, nullptr));
  OK(ws.qx.reserve((size_t)n * m->LD));
  OK(upload_dense(m, ws.qx.p, Q, (size_t)n, space));
  const int none = 0x7fffffff;
  int bad = none;
  CU(cudaMemcpyAsync(m->flags, &none, sizeof(int), cudaMemcpyHostToDevice, m->stream));
  rec::rec_check_finite_kernel<<<std::min((unsigned)(((size_t)n * m->K + 255) / 256), 8u * m->sm_count), 256, 0, m->stream>>>(
      ws.qx.p, n, m->K, m->LD, m->flags);
  OK(check_launch(m));
  CU(cudaMemcpyAsync(&bad, m->flags, sizeof(int), cudaMemcpyDeviceToHost, m->stream));
  CU(cudaStreamSynchronize(m->stream));
  if (bad != none) return fail(EALS_ERR_ARG, "query row %d has a non-finite entry", bad - 1);
  RecQuery q{ws.qx.p, nullptr, nullptr, nullptr, 0, m->V, m->N};
  if (ex_ptr) { q.ex_ptr = ws.excl.ptr; q.ex_idx = ws.excl.idx; }
  return rec_answer(m, space, n, q, k, items, scores);
}

// ---- similar items and similar users (DESIGN.md §3.8) ------------------------------------------------------------

// For each id q of the catalogue Y (which = EALS_BUF_V: V, the items; EALS_BUF_U: U, the users) the k rows r != q of
// highest cosine score seq_dot(Yhat[q], Yhat[r]), Yhat = Y with every row normalised (sim_normalize_kernel).  That is
// recommend_vectors on the normalised catalogue with the normalised query rows and each query's own row as its one
// excluded entry: the same engines, order, padding, limits, chunking and fall-backs.  U and V are replicated, so any
// id in [0, n_Y) may be asked for on any rank.
int similar_impl(eals_model* m, int which, int space, int n, const int32_t* ids, int k, int32_t* out_ids, double* scores) {
  if (!m || (n > 0 && (!ids || !out_ids))) return fail(EALS_ERR_ARG, "null argument");
  if (which != EALS_BUF_U && which != EALS_BUF_V) return fail(EALS_ERR_ARG, "which must be EALS_BUF_U or EALS_BUF_V");
  OK(rec_check_args(m, space, n, k));
  CU(cudaSetDevice(m->p.device));
  if (n == 0) return EALS_OK;
  const bool users = which == EALS_BUF_U;
  const double* Y = users ? m->U : m->V;
  const int nY = users ? m->M : m->N, LD = m->LD;
  const char* what = users ? "user" : "item";
  if (space == EALS_HOST)
    for (int s = 0; s < n; s++)
      if (ids[s] < 0 || ids[s] >= nY) return fail(EALS_ERR_ARG, "%s %d (position %d) outside [0, %d)", what, ids[s], s, nY);
  eals_eval_ws& ws = eval_ws(m);
  OK(ws.users.reserve((size_t)n));
  OK(copy_in(ws.users.p, ids, (size_t)n, space, m->stream));
  if (space == EALS_DEVICE) {
    int pos = -1, id = 0;
    OK(find_outside(m, ws.users.p, n, 0, nY, &pos, &id));
    if (pos >= 0) return fail(EALS_ERR_ARG, "%s %d (position %d) outside [0, %d)", what, id, pos, nY);
  }
  OK(ws.yhat.reserve((size_t)nY * LD));
  OK(ws.qx.reserve((size_t)n * LD));
  OK(ws.self_ptr.reserve((size_t)n + 1));
  rec::sim_normalize_kernel<<<(unsigned)std::min<size_t>(((size_t)nY * 32 + 255) / 256, 64 * (size_t)m->sm_count), 256, 0, m->stream>>>(
      Y, nY, m->K, LD, ws.yhat.p);
  OK(check_launch(m));
  rec::sim_queries_kernel<<<(unsigned)std::min<size_t>(((size_t)n * LD + 255) / 256, 8 * (size_t)m->sm_count), 256, 0, m->stream>>>(
      ws.yhat.p, LD, ws.users.p, n, ws.qx.p, ws.self_ptr.p);
  OK(check_launch(m));
  const RecQuery q{ws.qx.p, nullptr, ws.self_ptr.p, ws.users.p, 0, ws.yhat.p, nY};
  return rec_answer(m, space, n, q, k, out_ids, scores);
}

// ---- ranking metrics on a held-out test matrix (ranking.cuh, DESIGN.md §3.7) ------------------------------------
namespace rk = eals::rk;

// Engine 2 for the test entries of the owned rows [r0, r1) (n entries from e0 on, slot s = entry e0 + s): ranks of the
// slots into d_ranks[0 .. n).  Fills `st` and sets `done` when it answers; leaves both as they are when the
// candidate list overflows (the filter is not filtering: the exact engine answers instead).
int rm_chunk_tc(eals_model* m, int r0, int r1, int k, bool exclude, bool timed, int32_t* d_ranks, EvalStats& st, bool& done) {
  eals_eval_ws& ws = eval_ws(m);
  const Side &T = ws.test, &R = m->users;
  const int K = m->K, LD = m->LD;
  const int64_t e0 = T.h_ptr[(size_t)r0];
  const int n = (int)(T.h_ptr[(size_t)r1] - e0);
  cudaStream_t st_ = m->stream;
  StageTimer tm;
  // ---- slots: user, item, exact score of (u, g); train correction c_R and the certain-count limit ----
  OK(ws.users.reserve((size_t)n)); OK(ws.gt.reserve((size_t)n)); OK(ws.gts.reserve((size_t)n));
  OK(ws.c_r.reserve((size_t)n)); OK(ws.lim.reserve((size_t)n));
  rk::rm_entry_kernel<<<(n + 255) / 256, 256, 0, st_>>>(T.ptr, T.idx, r0, r1, m->ub, e0, n, ws.users.p, ws.gt.p);
  OK(check_launch(m));
  eals::eval_gt_score_kernel<<<(n + 127) / 128, 128, 0, st_>>>(m->U, m->V, ws.gt.p, ws.users.p, 0, n, K, LD, ws.gts.p);
  OK(check_launch(m));
  const int64_t z0 = R.h_ptr[(size_t)r0], nz = R.h_ptr[(size_t)r1] - z0;
  if (exclude && nz > 0) {   // every train nonzero of these users scored once; the entries then only compare
    OK(ws.tscore.reserve((size_t)nz));
    rk::rm_train_score_kernel<<<16 * m->sm_count, 128, 0, st_>>>(m->U, m->V, K, LD, R.ptr, R.idx, T.ptr, r0, r1, m->ub, z0, nz, ws.tscore.p);
    OK(check_launch(m));
  }
  rk::rm_train_count_kernel<<<(unsigned)(((size_t)n * 32 + 255) / 256), 256, 0, st_>>>(exclude ? R.ptr : nullptr, R.idx, ws.tscore.p, z0,
                                                                                       m->ub, ws.users.p, ws.gt.p, ws.gts.p, n, k,
                                                                                       ws.c_r.p, ws.lim.p);
  OK(check_launch(m));
  OK(tc_prepare_rows(m, n, m->U, ws.users.p, ws.gts.p));
  tm.lap("ranking: slots, train correction, fp16 rows");
  // a slot leaves once its certain count reaches k + c_R; the survivors go through MODE 2 (every item not certainly
  // below s_g) for the exact tie-aware count.  Test items that are in the train row (limit 0) never enter the filter.
  CountPass cp;
  OK(count_pass<2>(m, n, ws.lim.p, 0, exclude, timed, 2048, tm, cp));
  if (cp.overflow) return EALS_OK;
  if (cp.pairs) {
    rk::rm_rescore_kernel<<<16 * m->sm_count, 128, 0, st_>>>(m->U, m->V, K, LD, ws.users.p, ws.gt.p, ws.gts.p, ws.pairs.p, cp.pairs,
                                                             ws.cnt_exact.p);
    OK(check_launch(m));
  }
  rk::rm_rank_kernel<<<(n + 255) / 256, 256, 0, st_>>>(n, ws.cnt.p, ws.lim.p, ws.cnt_exact.p, ws.c_r.p, k, d_ranks);
  OK(check_launch(m));
  CU(cudaStreamSynchronize(st_));
  tm.lap("ranking: exact re-score + ranks");
  if (timed) OK(ws.blk0.read(st.blk0));
  st.engine = 1; st.candidates += cp.n_cand; st.pairs += (long long)cp.pairs;
  done = true;
  return EALS_OK;
}

// Engine 1 for the owned rows [r0, r1): recommend's exact engine (rec_exact) for the users with test entries, a
// list budget's worth at a time, and each test item looked up in its user's list.  d_ranks: every owned entry, -1
// where no list reaches.
int rm_chunk_exact(eals_model* m, int r0, int r1, int k, bool exclude, int32_t* d_ranks) {
  eals_eval_ws& ws = eval_ws(m);
  const Side& T = ws.test;
  std::vector<int32_t> users;
  for (int r = r0; r < r1; r++)
    if (T.h_ptr[(size_t)r + 1] > T.h_ptr[(size_t)r]) users.push_back(m->ub + r);
  const int n = (int)users.size();
  const int per = (int)std::min<size_t>((size_t)std::max(n, 1), list_slots(k));
  for (int d0 = 0; d0 < n; d0 += per) {
    const int nd = std::min(per, n - d0);
    OK(ws.users.reserve((size_t)nd));
    OK(ws.top_s.reserve((size_t)nd * k)); OK(ws.top_i.reserve((size_t)nd * k)); OK(ws.thr.reserve((size_t)nd));
    CU(cudaMemcpyAsync(ws.users.p, users.data() + d0, sizeof(int32_t) * nd, cudaMemcpyHostToDevice, m->stream));
    RecQuery q{m->U, ws.users.p, nullptr, nullptr, 0, m->V, m->N};
    if (exclude) { q.ex_ptr = m->users.ptr; q.ex_idx = m->users.idx; q.ex_base = m->users.row_base; }
    OK(rec_exact(m, nd, q, k));
    rk::rm_lookup_kernel<<<(unsigned)(((size_t)nd * k + 255) / 256), 256, 0, m->stream>>>(ws.top_i.p, k, nd, ws.users.p, m->ub, T.ptr,
                                                                                          T.idx, d_ranks);
    OK(check_launch(m));
    CU(cudaStreamSynchronize(m->stream));   // the users' host slice and the lists are reused by the next piece
  }
  return EALS_OK;
}

// Ranks and metrics at k of the owned rows of the test CSR (M rows, train-matrix rules), DESIGN.md §3.7.
int ranking_metrics_impl(eals_model* m, int space, const int64_t* test_ptr, const int32_t* test_idx, int k, int exclude_seen,
                         double sums[6], int64_t* n_users, double* per_user, int32_t* ranks) {
  if (!m || !test_ptr || !test_idx || !sums || !n_users) return fail(EALS_ERR_ARG, "null argument");
  OK(rec_check_args(m, space, 0, k));
  CU(cudaSetDevice(m->p.device));
  eals_eval_ws& ws = eval_ws(m);
  const int n_rows = m->ue - m->ub;
  const bool exclude = exclude_seen != 0;
  OK(build_query_side(m, ws.test, ws.test_check, n_rows, space, test_ptr, test_idx, nullptr, m->ub));
  const Side &T = ws.test, &R = m->users;
  const int64_t n_ent = T.nnz;
  OK(ws.ranks.reserve((size_t)std::max<int64_t>(n_ent, 1)));
  CU(cudaMemsetAsync(ws.ranks.p, 0xff, sizeof(int32_t) * (size_t)std::max<int64_t>(n_ent, 1), m->stream));   // -1
  m->eval_stats = EvalStats{};
  // ---- ranks, chunk by chunk of whole rows within the device budget ----
  const int KP = (m->K + eals::tc::kKC - 1) / eals::tc::kKC * eals::tc::kKC;
  const size_t budget = list_budget();   // the entries' fp16 rows and working lists, the train scores
  const size_t per_entry = 4 * (size_t)KP + 128, per_nz = exclude ? 8 : 0;
  EvalStats total;
  bool any = false, all_tc = true, items_ready = false;
  for (int r0 = 0; r0 < n_rows;) {
    int r1 = r0;
    size_t cost = 0;
    while (r1 < n_rows) {
      const int64_t ne = T.h_ptr[(size_t)r1 + 1] - T.h_ptr[(size_t)r1], nz = R.h_ptr[(size_t)r1 + 1] - R.h_ptr[(size_t)r1];
      const size_t c = (size_t)ne * per_entry + (size_t)nz * per_nz;
      if (r1 > r0 && (cost + c > budget || T.h_ptr[(size_t)r1 + 1] - T.h_ptr[(size_t)r0] > (1 << 28))) break;
      cost += c;
      r1++;
    }
    const int64_t e0 = T.h_ptr[(size_t)r0];
    const int64_t n = T.h_ptr[(size_t)r1] - e0;
    if (n > 0) {
      EvalStats c;
      bool done = false;
      if (use_tc_engine(m, (int)n)) {   // n <= max(2^28, one row of at most N items)
        if (!items_ready) OK(tc_prepare_items(m, m->V, m->N));
        items_ready = true;
        OK(rm_chunk_tc(m, r0, r1, k, exclude, !any, ws.ranks.p + e0, c, done));
      }
      if (!done) { OK(rm_chunk_exact(m, r0, r1, k, exclude, ws.ranks.p)); all_tc = false; }
      if (!any) total.blk0 = c.blk0;   // the first block of the first chunk
      total.candidates += c.candidates; total.pairs += c.pairs;
      any = true;
    }
    r0 = r1;
  }
  total.engine = any && all_tc ? 1 : 0;
  m->eval_stats = total;
  // ---- per-user metrics on the device, sums on the host in user order ----
  std::vector<double> pu((size_t)n_rows * rk::kMetrics);
  if (n_rows > 0) {
    std::vector<double> tab(2 * (size_t)k + 1);   // gain[0 .. k), idcg[0 .. k]
    double acc = 0.0;
    tab[(size_t)k] = 0.0;
    for (int j = 0; j < k; j++) {
      tab[(size_t)j] = metric_ndcg(j);
      acc += tab[(size_t)j];
      tab[(size_t)k + 1 + j] = acc;
    }
    OK(ws.rm_tab.reserve(tab.size())); OK(ws.rm_out.reserve(pu.size()));
    CU(cudaMemcpyAsync(ws.rm_tab.p, tab.data(), sizeof(double) * tab.size(), cudaMemcpyHostToDevice, m->stream));
    rk::rm_metrics_kernel<<<(unsigned)(((size_t)n_rows * 32 + 127) / 128), 128, 0, m->stream>>>(T.ptr, n_rows, ws.ranks.p, k, ws.rm_tab.p,
                                                                                                 ws.rm_tab.p + k, ws.rm_out.p);
    OK(check_launch(m));
    CU(cudaMemcpyAsync(pu.data(), ws.rm_out.p, sizeof(double) * pu.size(), cudaMemcpyDeviceToHost, m->stream));
    CU(cudaStreamSynchronize(m->stream));
  }
  for (int j = 0; j < rk::kMetrics; j++) sums[j] = 0.0;
  int64_t users = 0;
  for (int r = 0; r < n_rows; r++) {
    if (T.h_ptr[(size_t)r + 1] == T.h_ptr[(size_t)r]) continue;
    users++;
    for (int j = 0; j < rk::kMetrics; j++) sums[j] += pu[(size_t)r * rk::kMetrics + j];
  }
  *n_users = users;
  const cudaMemcpyKind kind = space == EALS_DEVICE ? cudaMemcpyHostToDevice : cudaMemcpyHostToHost;
  if (per_user && n_rows > 0) CU(cudaMemcpy(per_user, pu.data(), sizeof(double) * pu.size(), kind));
  if (ranks && n_ent > 0)
    CU(cudaMemcpy(ranks, ws.ranks.p, sizeof(int32_t) * (size_t)n_ent, space == EALS_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost));
  return EALS_OK;
}

}  // namespace
