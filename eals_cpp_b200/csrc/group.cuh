// group.cuh — eals_group: the multi-GPU split BEHIND the C ABI (included at the end of eals_b200.cu).
//
// The reference is one object driven by one thread (MF_fastALS.h:52-55, MF_fastALS.cpp:112-161).  A group is
// the same thing for N GPUs of one box: ONE process, ONE host thread, N eals_models — rank r on
// devices[r] — each owning a contiguous user range and item range (boundaries by a per-row cost model,
// eals_partition) and holding full replicas of U and V.  Per half-epoch, entirely stream-ordered (no host
// synchronisation inside an epoch):
//
//   sweep   every rank's CD kernels store each finished row into ALL replicas (plain peer pointers over
//           NVLink; cudaDeviceEnablePeerAccess) — the all-gather of the updated shard is fused into K1;
//           final predictions are routed to the rank that starts from them in the next half-epoch;
//   Gram    every rank reduces its own rows into a K x K partial;
//   all-reduce   one-shot, over peer memory: every rank sums the N partials IN RANK ORDER with one small
//           kernel (allreduce_fixed_kernel) — so all ranks hold bit-identical S caches, run to run;
//           ordering between ranks is by CUDA events (cudaStreamWaitEvent across devices), which also
//           orders the peer stores before the next half-epoch.
//
// `devices` may name the same GPU several times: "virtual ranks".  The whole sharded path (partition, peer
// stores, routed prediction caches, all-reduce, setTrain re-attachment) then runs on one GPU, which is how
// the 1-GPU test box covers it (tests/test_gpu_multi.py).

struct eals_group {
  int n = 0;
  std::vector<eals_model*> r;
  std::vector<int> dev;
  eals_params base;                      // rank-independent parameters
  std::vector<int32_t> ub, ib;           // [n+1] user / item boundaries
  std::vector<double*> part;             // per rank: staging copy of its partial Gram ([K][LD])
  std::vector<cudaEvent_t> ev_part, ev_red;
  bool events_live = false;
};

namespace {

struct PartSet {
  const double* p[8];
  int n;
};

// out[t] = sum over ranks q = 0..n-1 (in that order) of p[q][t]
__global__ void allreduce_fixed_kernel(PartSet ps, double* __restrict__ out, int len) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= len) return;
  double acc = ps.p[0][t];
  for (int q = 1; q < ps.n; q++) acc += ps.p[q][t];
  out[t] = acc;
}

// fn(rank) on every rank, one host thread per rank (set-up calls that synchronise internally: uploads,
// bucketing, evaluation).  Returns the first non-zero status; its message is copied to the calling thread.
template <typename F>
int parallel_ranks(eals_group* g, F fn) {
  std::vector<int> rc((size_t)g->n, EALS_OK);
  std::vector<std::string> msg((size_t)g->n);
  if (g->n == 1) {
    rc[0] = fn(0);
    return rc[0];
  }
  std::vector<std::thread> th;
  for (int q = 0; q < g->n; q++)
    th.emplace_back([&, q] {
      rc[q] = fn(q);
      if (rc[q] != EALS_OK) msg[q] = g_err;
    });
  for (auto& t : th) t.join();
  for (int q = 0; q < g->n; q++)
    if (rc[q] != EALS_OK) return fail(rc[q], "rank %d: %s", q, msg[q].c_str());
  return EALS_OK;
}

// Per-row cost in nanoseconds on one B200 by kernel family (c4 profile of round 1 / round 2; DESIGN.md §6):
// rows of 1..32 nonzeros cost about the same whatever their length, longer rows cost per nonzero, the slab
// pipeline is the cheapest per nonzero.  Balancing THIS instead of raw nonzeros removes the wait in the Gram
// all-reduce (3.5 ms of a 74 ms epoch at 8 GPUs in round 1).
inline double row_cost_ns(int64_t len) {
  if (len <= 0) return 0.3;
  if (len <= 32) return 13.0;
  if (len <= 128) return 0.47 * (double)len;
  if (len <= 512) return 0.42 * (double)len;
  return 0.37 * (double)len;
}

void partition_rows(const int64_t* ptr, int rows, int n, int32_t* bounds) {
  std::vector<double> pre((size_t)rows + 1);
  pre[0] = 0;
  for (int r = 0; r < rows; r++) pre[(size_t)r + 1] = pre[r] + row_cost_ns(ptr[r + 1] - ptr[r]);
  bounds[0] = 0;
  for (int q = 1; q < n; q++) {
    const double target = pre[rows] * q / n;
    int b = (int)(std::lower_bound(pre.begin(), pre.end(), target) - pre.begin());
    b = std::max(b, bounds[q - 1] + 1);              // every rank owns at least one row
    bounds[q] = std::min(b, rows - (n - q));
  }
  bounds[n] = rows;
}

// Plain-pointer attachment of the other ranks' buffers (same process: no CUDA IPC).
void group_attach(eals_group* g) {
  for (int q = 0; q < g->n; q++) {
    eals_model* m = g->r[q];
    m->local_peers = true;
    m->peersU.n = m->peersV.n = 0;
    for (int o = 0; o < g->n; o++) {
      if (o == q) continue;
      m->peersU.x[m->peersU.n++] = g->r[o]->U;
      m->peersV.x[m->peersV.n++] = g->r[o]->V;
    }
  }
  bool all_pc = g->n > 1;
  for (int q = 0; q < g->n; q++) all_pc = all_pc && g->r[q]->pcache_on;
  for (int q = 0; q < g->n; q++) {
    eals_model* m = g->r[q];
    if (g->n == 1) continue;
    for (int o = 0; o < g->n; o++) {
      m->out_to_users.base[o] = all_pc ? g->r[o]->pc_u : nullptr;
      m->out_to_items.base[o] = all_pc ? g->r[o]->pc_i : nullptr;
    }
    m->pc_users_attached = m->pc_items_attached = m->pc_attached = all_pc;
    m->pc_u_valid = m->pc_i_valid = false;
  }
}

int group_events(eals_group* g) {
  if (g->events_live) return EALS_OK;
  g->ev_part.resize((size_t)g->n); g->ev_red.resize((size_t)g->n); g->part.assign((size_t)g->n, nullptr);
  for (int q = 0; q < g->n; q++) {
    CU(cudaSetDevice(g->dev[q]));
    CU(cudaEventCreateWithFlags(&g->ev_part[q], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&g->ev_red[q], cudaEventDisableTiming));
    CU(cudaEventRecord(g->ev_red[q], g->r[q]->stream));
    OK(dev_alloc(&g->part[q], (size_t)g->r[q]->LD * g->r[q]->LD));
  }
  g->events_live = true;
  return EALS_OK;
}

// S (SU or SV) of every rank <- sum of all ranks' partials, same bits everywhere.
int group_allreduce(eals_group* g, bool user) {
  if (g->n == 1) return EALS_OK;
  OK(group_events(g));
  const size_t len = (size_t)g->r[0]->K * g->r[0]->LD;
  for (int q = 0; q < g->n; q++) {          // stage the partial where the peers may read it
    eals_model* m = g->r[q];
    CU(cudaSetDevice(g->dev[q]));
    for (int o = 0; o < g->n; o++) CU(cudaStreamWaitEvent(m->stream, g->ev_red[o], 0));   // previous readers are done
    CU(cudaMemcpyAsync(g->part[q], user ? m->SU : m->SV, len * sizeof(double), cudaMemcpyDeviceToDevice, m->stream));
    CU(cudaEventRecord(g->ev_part[q], m->stream));
  }
  PartSet ps;
  ps.n = g->n;
  for (int o = 0; o < g->n; o++) ps.p[o] = g->part[o];
  for (int q = 0; q < g->n; q++) {
    eals_model* m = g->r[q];
    CU(cudaSetDevice(g->dev[q]));
    for (int o = 0; o < g->n; o++)
      if (o != q) CU(cudaStreamWaitEvent(m->stream, g->ev_part[o], 0));   // every rank's sweep + Gram of this half-epoch
    allreduce_fixed_kernel<<<(unsigned)((len + 255) / 256), 256, 0, m->stream>>>(ps, user ? m->SU : m->SV, (int)len);
    OK(check_launch(m));
    CU(cudaEventRecord(g->ev_red[q], m->stream));
  }
  return EALS_OK;
}

int group_barrier(eals_group* g) {            // host waits for every rank's stream
  for (int q = 0; q < g->n; q++) OK(eals_sync(g->r[q]));
  return EALS_OK;
}

int group_owner(const std::vector<int32_t>& bounds, int row) {
  return (int)(std::upper_bound(bounds.begin(), bounds.end(), row) - bounds.begin()) - 1;
}

}  // namespace

extern "C" {

int eals_partition(const int64_t* ptr, int32_t n_rows, int32_t n_ranks, int32_t* bounds) {
  if (!ptr || !bounds || n_rows < 1 || n_ranks < 1 || n_ranks > n_rows) return fail(EALS_ERR_ARG, "eals_partition: bad arguments");
  partition_rows(ptr, n_rows, n_ranks, bounds);
  return EALS_OK;
}

int eals_group_destroy(eals_group* g) {
  if (!g) return EALS_OK;
  for (int q = 0; q < (int)g->r.size(); q++)
    if (g->r[q]) { cudaSetDevice(g->dev[q]); cudaStreamSynchronize(g->r[q]->stream); }
  for (int q = 0; q < (int)g->r.size(); q++) {
    if (g->events_live) {
      cudaSetDevice(g->dev[q]);
      cudaEventDestroy(g->ev_part[q]); cudaEventDestroy(g->ev_red[q]); cudaFree(g->part[q]);
    }
    eals_destroy(g->r[q]);
  }
  delete g;
  return EALS_OK;
}

int eals_group_create(const eals_params* params, int32_t n_ranks, const int32_t* devices, const int64_t* row_ptr,
                      const int32_t* col_idx, const double* row_val, const int64_t* col_ptr, const int32_t* row_idx,
                      const double* col_val, eals_group** out) {
  if (!out) return fail(EALS_ERR_ARG, "out is null");
  *out = nullptr;
  if (!params || params->struct_bytes != (int32_t)sizeof(eals_params)) return fail(EALS_ERR_ARG, "params null or struct_bytes mismatch");
  if (n_ranks < 1 || n_ranks > 8) return fail(EALS_ERR_UNSUPPORTED, "a group has 1..8 ranks");
  if (!row_ptr || !col_ptr || !col_idx || !row_idx) return fail(EALS_ERR_ARG, "matrix arrays are null");
  if (params->n_users < n_ranks || params->n_items < n_ranks) return fail(EALS_ERR_ARG, "more ranks than rows");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(EALS_ERR_CUDA, "no CUDA device: libeals_b200 has no CPU fallback");
  eals_group* g = new (std::nothrow) eals_group();
  if (!g) return fail(EALS_ERR_ALLOC, "host allocation failed");
  g->n = n_ranks;
  g->base = *params;
  g->r.assign((size_t)n_ranks, nullptr);
  for (int q = 0; q < n_ranks; q++) {
    const int d = devices ? devices[q] : q;
    if (d < 0 || d >= ndev) { delete g; return fail(EALS_ERR_ARG, "device %d of rank %d out of range (%d devices)", d, q, ndev); }
    g->dev.push_back(d);
  }
  // peer access between every pair of distinct devices (the sweep kernels store into all replicas)
  for (int a = 0; a < n_ranks; a++)
    for (int b = 0; b < n_ranks; b++) {
      if (g->dev[a] == g->dev[b]) continue;
      int can = 0;
      cudaDeviceCanAccessPeer(&can, g->dev[a], g->dev[b]);
      if (!can) { delete g; return fail(EALS_ERR_UNSUPPORTED, "GPU %d cannot access GPU %d (peer access)", g->dev[a], g->dev[b]); }
      cudaSetDevice(g->dev[a]);
      const cudaError_t e = cudaDeviceEnablePeerAccess(g->dev[b], 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { delete g; return fail(EALS_ERR_CUDA, "cudaDeviceEnablePeerAccess -> %s", cudaGetErrorString(e)); }
      cudaGetLastError();
    }
  // boundaries from host copies of the offsets
  const int M = params->n_users, N = params->n_items;
  std::vector<int64_t> rp((size_t)M + 1), cp((size_t)N + 1);
  if (params->input_space == EALS_DEVICE) {
    if (cudaMemcpy(rp.data(), row_ptr, sizeof(int64_t) * (M + 1), cudaMemcpyDeviceToHost) != cudaSuccess ||
        cudaMemcpy(cp.data(), col_ptr, sizeof(int64_t) * (N + 1), cudaMemcpyDeviceToHost) != cudaSuccess) {
      delete g;
      return fail(EALS_ERR_CUDA, "cannot read the offsets");
    }
  } else {
    std::memcpy(rp.data(), row_ptr, sizeof(int64_t) * (M + 1));
    std::memcpy(cp.data(), col_ptr, sizeof(int64_t) * (N + 1));
  }
  g->ub.resize((size_t)n_ranks + 1); g->ib.resize((size_t)n_ranks + 1);
  partition_rows(rp.data(), M, n_ranks, g->ub.data());
  partition_rows(cp.data(), N, n_ranks, g->ib.data());
  const int rc = parallel_ranks(g, [&](int q) -> int {
    eals_params p = *params;
    p.device = g->dev[q];
    p.user_begin = g->ub[q]; p.user_end = g->ub[q + 1];
    p.item_begin = g->ib[q]; p.item_end = g->ib[q + 1];
    p.n_ranks = n_ranks > 1 ? n_ranks : 0;
    p.rank = q;
    for (int t = 0; t <= n_ranks; t++) { p.user_bounds[t] = g->ub[t]; p.item_bounds[t] = g->ib[t]; }
    return eals_create(&p, row_ptr, col_idx, row_val, col_ptr, row_idx, col_val, &g->r[q]);
  });
  if (rc != EALS_OK) { eals_group_destroy(g); return rc; }
  group_attach(g);
  *out = g;
  return EALS_OK;
}

int eals_group_size(const eals_group* g) { return g ? g->n : 0; }

int eals_group_model(eals_group* g, int32_t rank, eals_model** out) {
  if (!g || !out || rank < 0 || rank >= g->n) return fail(EALS_ERR_ARG, "bad rank");
  *out = g->r[rank];
  return EALS_OK;
}

int eals_group_bounds(const eals_group* g, int32_t* user_bounds, int32_t* item_bounds) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  for (int t = 0; t <= g->n; t++) {
    if (user_bounds) user_bounds[t] = g->ub[t];
    if (item_bounds) item_bounds[t] = g->ib[t];
  }
  return EALS_OK;
}

int eals_group_sync(eals_group* g) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  return group_barrier(g);
}

int eals_group_set_train(eals_group* g, int32_t input_space, const int64_t* row_ptr, const int32_t* col_idx,
                         const double* row_val, const int64_t* col_ptr, const int32_t* row_idx, const double* col_val) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  OK(group_barrier(g));
  OK(parallel_ranks(g, [&](int q) { return eals_set_train(g->r[q], input_space, row_ptr, col_idx, row_val, col_ptr, row_idx, col_val); }));
  group_attach(g);                                  // caches may have moved
  for (int q = 0; q < g->n; q++) OK(eals_ipc_gc(g->r[q]));
  return EALS_OK;
}

// Replicate rank 0's U, V (and S caches) on every other rank, device to device.
static int group_broadcast_factors(eals_group* g) {
  eals_model* a = g->r[0];
  OK(eals_sync(a));
  for (int q = 1; q < g->n; q++) {
    eals_model* m = g->r[q];
    CU(cudaSetDevice(g->dev[q]));
    CU(cudaMemcpyAsync(m->U, a->U, sizeof(double) * (size_t)a->M * a->LD, cudaMemcpyDefault, m->stream));
    CU(cudaMemcpyAsync(m->V, a->V, sizeof(double) * (size_t)a->N * a->LD, cudaMemcpyDefault, m->stream));
    CU(cudaMemcpyAsync(m->SU, a->SU, sizeof(double) * (size_t)a->LD * a->LD, cudaMemcpyDefault, m->stream));
    CU(cudaMemcpyAsync(m->SV, a->SV, sizeof(double) * (size_t)a->LD * a->LD, cudaMemcpyDefault, m->stream));
    m->factors_set = true; m->su_fresh = true;
    m->pc_u_valid = m->pc_i_valid = false;
  }
  return group_barrier(g);                          // no rank sweeps before every replica is written
}

int eals_group_init_factors(eals_group* g) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  OK(group_barrier(g));
  OK(eals_init_factors(g->r[0]));                   // the sequential libstdc++ stream once, not once per rank
  return group_broadcast_factors(g);
}

int eals_group_set_factors(eals_group* g, int32_t space, const double* U, const double* V) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  OK(group_barrier(g));
  OK(eals_set_factors(g->r[0], space, U, V));
  return group_broadcast_factors(g);
}

int eals_group_get_factors(eals_group* g, int32_t space, double* U, double* V) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  OK(group_barrier(g));
  return eals_get_factors(g->r[0], space, U, V);
}

int eals_group_get_S(eals_group* g, int32_t space, double* SU, double* SV) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  OK(group_barrier(g));
  return eals_get_S(g->r[0], space, SU, SV);
}

int eals_group_set_item_weights(eals_group* g, int32_t space, const double* Wi) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  OK(group_barrier(g));
  for (int q = 0; q < g->n; q++) OK(eals_set_item_weights(g->r[q], space, Wi));   // every rank rebuilds the FULL SV from its replica
  return EALS_OK;
}

int eals_group_get_item_weights(eals_group* g, int32_t space, double* Wi) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  return eals_get_item_weights(g->r[0], space, Wi);
}

static int group_half_epoch(eals_group* g, bool user) {
  for (int q = 0; q < g->n; q++) OK(user ? eals_sweep_users(g->r[q]) : eals_sweep_items(g->r[q]));
  for (int q = 0; q < g->n; q++) OK(user ? eals_gram_users(g->r[q]) : eals_gram_items(g->r[q]));
  return group_allreduce(g, user);
}

int eals_group_update_user(eals_group* g) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  return group_half_epoch(g, true);
}
int eals_group_update_item(eals_group* g) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  return group_half_epoch(g, false);
}

int eals_group_update_user_row(eals_group* g, int32_t u) {
  if (!g || u < 0 || u >= g->base.n_users) return fail(EALS_ERR_ARG, "user out of range");
  OK(group_barrier(g));
  const int q = group_owner(g->ub, u);
  OK(eals_update_user_row(g->r[q], u));             // the finished row is stored into every replica by the kernel
  OK(eals_sync(g->r[q]));
  for (int o = 0; o < g->n; o++) { g->r[o]->su_fresh = false; g->r[o]->pc_u_valid = g->r[o]->pc_i_valid = false; }
  return EALS_OK;
}
int eals_group_update_item_row(eals_group* g, int32_t i) {
  if (!g || i < 0 || i >= g->base.n_items) return fail(EALS_ERR_ARG, "item out of range");
  OK(group_barrier(g));
  const int q = group_owner(g->ib, i);
  OK(eals_update_item_row(g->r[q], i));
  OK(eals_sync(g->r[q]));
  for (int o = 0; o < g->n; o++) g->r[o]->pc_u_valid = g->r[o]->pc_i_valid = false;
  return EALS_OK;
}
int eals_group_patch_SU(eals_group* g, const double* old_row, const double* new_row) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  for (int q = 0; q < g->n; q++) OK(eals_patch_SU(g->r[q], old_row, new_row));
  return EALS_OK;
}
int eals_group_patch_SV(eals_group* g, int32_t i, const double* old_row, const double* new_row) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  for (int q = 0; q < g->n; q++) OK(eals_patch_SV(g->r[q], i, old_row, new_row));
  return EALS_OK;
}
int eals_group_get_factor_row(eals_group* g, int32_t which, int32_t row, double* out) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  return eals_get_factor_row(g->r[0], which, row, out);
}

int eals_group_loss(eals_group* g, double* loss) {
  if (!g || !loss) return fail(EALS_ERR_ARG, "null argument");
  double t0 = 0, t1 = 0, t2 = 0, t3 = 0;
  for (int q = 0; q < g->n; q++) OK(loss_terms_enqueue(g->r[q]));     // all ranks work at the same time
  for (int q = 0; q < g->n; q++) {
    double t[4];
    OK(loss_terms_fetch(g->r[q], t));
    t0 += t[0]; t1 += t[1]; t2 += t[2];
    if (q == 0) t3 = t[3];                                             // <SU, SV>: complete on every rank
  }
  *loss = g->base.reg * (t1 + t2) + t0 + t3;
  return EALS_OK;
}

int eals_group_predict(eals_group* g, int32_t u, int32_t i, double* score) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  OK(group_barrier(g));
  return eals_predict(g->r[0], u, i, score);
}

int eals_group_evaluate(eals_group* g, const int32_t* gt_items, int32_t topk, int32_t mode, double means[3],
                        double* hr, double* ndcg, double* prec, int32_t* count_larger) {
  if (!g || !gt_items || !means) return fail(EALS_ERR_ARG, "null argument");
  OK(group_barrier(g));
  std::vector<double> sums((size_t)3 * g->n, 0.0);
  OK(parallel_ranks(g, [&](int q) {
    const int b = g->ub[q];
    return eals_evaluate(g->r[q], gt_items, topk, mode, &sums[(size_t)3 * q], hr ? hr + b : nullptr, ndcg ? ndcg + b : nullptr,
                         prec ? prec + b : nullptr, count_larger ? count_larger + b : nullptr);
  }));
  for (int k = 0; k < 3; k++) {
    double s = 0;
    for (int q = 0; q < g->n; q++) s += sums[(size_t)3 * q + k];
    means[k] = s / g->base.n_users;
  }
  return EALS_OK;
}

// Every user goes to the rank that owns its row of the train matrix (U and V are replicated, the seen items are
// the owner's); the ranks run at once, each on its own stream, and the results land in input order.
int eals_group_recommend(eals_group* g, int32_t space, int32_t n, const int32_t* users, int32_t k, int32_t exclude_seen,
                         int32_t* items, double* scores) {
  if (!g || (n > 0 && (!users || !items))) return fail(EALS_ERR_ARG, "null argument");
  OK(check_topk_args(space, n, k));
  OK(group_barrier(g));
  if (n == 0) return EALS_OK;
  std::vector<int32_t> hu((size_t)n);
  if (space == EALS_DEVICE) CU(cudaMemcpy(hu.data(), users, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
  else std::memcpy(hu.data(), users, sizeof(int32_t) * n);
  std::vector<std::vector<int32_t>> pos((size_t)g->n), who((size_t)g->n);
  for (int s = 0; s < n; s++) {
    if (hu[(size_t)s] < 0 || hu[(size_t)s] >= g->base.n_users)
      return fail(EALS_ERR_ARG, "user %d (position %d) outside [0, %d)", hu[(size_t)s], s, g->base.n_users);
    const int q = group_owner(g->ub, hu[(size_t)s]);
    pos[(size_t)q].push_back(s);
    who[(size_t)q].push_back(hu[(size_t)s]);
  }
  const size_t nk = (size_t)n * k;
  std::vector<int32_t> out_i(nk);
  std::vector<double> out_s(nk);
  OK(parallel_ranks(g, [&](int q) -> int {
    const size_t nq = pos[(size_t)q].size();
    if (nq == 0) return EALS_OK;
    std::vector<int32_t> ri(nq * k);
    std::vector<double> rs(nq * k);
    OK(eals_recommend(g->r[q], EALS_HOST, (int32_t)nq, who[(size_t)q].data(), k, exclude_seen, ri.data(), rs.data()));
    for (size_t t = 0; t < nq; t++) {
      const size_t s = (size_t)pos[(size_t)q][t];
      std::memcpy(&out_i[s * k], &ri[t * k], sizeof(int32_t) * k);
      std::memcpy(&out_s[s * k], &rs[t * k], sizeof(double) * k);
    }
    return EALS_OK;
  }));
  if (space == EALS_DEVICE) {
    CU(cudaMemcpy(items, out_i.data(), sizeof(int32_t) * nk, cudaMemcpyHostToDevice));
    if (scores) CU(cudaMemcpy(scores, out_s.data(), sizeof(double) * nk, cudaMemcpyHostToDevice));
  } else {
    std::memcpy(items, out_i.data(), sizeof(int32_t) * nk);
    if (scores) std::memcpy(scores, out_s.data(), sizeof(double) * nk);
  }
  return EALS_OK;
}

}  // extern "C"

namespace {

// The n queries of fold_in / recommend_vectors in balanced contiguous slices over the ranks (V, SV and Wi are
// replicated: any rank can answer any query), the ranks at once.  Device inputs are staged through the host like
// eals_group_recommend's, so each rank reads them whatever device it is on; fn(rank, lo, hi) runs a host-space call.
template <typename F>
int group_slices(eals_group* g, int n, F fn) {
  return parallel_ranks(g, [&](int q) -> int {
    const int lo = (int)((int64_t)n * q / g->n), hi = (int)((int64_t)n * (q + 1) / g->n);
    return hi > lo ? fn(q, lo, hi) : EALS_OK;
  });
}

// A host copy of a CSR of n rows (host or device), offsets rebased to 0; val stays empty for NULL.
struct HostCsr {
  std::vector<int64_t> ptr;
  std::vector<int32_t> idx;
  std::vector<double> val;
  int load(int space, int n, const int64_t* p, const int32_t* i, const double* v) {
    ptr.resize((size_t)n + 1);
    if (space == EALS_DEVICE) CU(cudaMemcpy(ptr.data(), p, sizeof(int64_t) * (n + 1), cudaMemcpyDeviceToHost));
    else std::memcpy(ptr.data(), p, sizeof(int64_t) * (n + 1));
    const int64_t base = ptr[0], nnz = ptr[(size_t)n] - base;
    if (nnz < 0) return fail(EALS_ERR_ARG, "offsets not monotone");
    for (auto& x : ptr) x -= base;
    idx.resize((size_t)std::max<int64_t>(nnz, 1));   // a non-null index array even when every row is empty
    if (v) val.resize((size_t)nnz);
    if (space == EALS_DEVICE) {
      if (nnz) CU(cudaMemcpy(idx.data(), i + base, sizeof(int32_t) * nnz, cudaMemcpyDeviceToHost));
      if (v && nnz) CU(cudaMemcpy(val.data(), v + base, sizeof(double) * nnz, cudaMemcpyDeviceToHost));
    } else {
      if (nnz) std::memcpy(idx.data(), i + base, sizeof(int32_t) * nnz);
      if (v && nnz) std::memcpy(val.data(), v + base, sizeof(double) * nnz);
    }
    return EALS_OK;
  }
  const double* vals(const double* given) const { return given ? val.data() : nullptr; }
};

// Host staging of `count` elements of a host or device array (device: copied; host: the caller's memory).
template <typename T>
int host_view(int space, const T* src, size_t count, std::vector<T>& buf, const T** out) {
  if (!src || space == EALS_HOST) { *out = src; return EALS_OK; }
  buf.resize(count);
  if (count) CU(cudaMemcpy(buf.data(), src, sizeof(T) * count, cudaMemcpyDeviceToHost));
  *out = buf.data();
  return EALS_OK;
}

// Results staged in host memory -> the caller's host or device array.
template <typename T>
int host_result(int space, T* dst, const std::vector<T>& buf) {
  if (space == EALS_DEVICE) CU(cudaMemcpy(dst, buf.data(), sizeof(T) * buf.size(), cudaMemcpyHostToDevice));
  else std::memcpy(dst, buf.data(), sizeof(T) * buf.size());
  return EALS_OK;
}

}  // namespace

extern "C" {

int eals_group_fold_in(eals_group* g, int32_t space, int32_t n, const int64_t* row_ptr, const int32_t* col_idx, const double* val,
                       const double* init, int32_t n_iter, double* out) {
  if (!g || (n > 0 && (!row_ptr || !col_idx || !out))) return fail(EALS_ERR_ARG, "null argument");
  OK(check_fold_in_args(space, n, n_iter));
  OK(group_barrier(g));
  if (n == 0) return EALS_OK;
  const size_t K = (size_t)g->base.factors;
  HostCsr h;
  OK(h.load(space, n, row_ptr, col_idx, val));
  std::vector<double> init_buf, res((size_t)n * K);
  const double* hinit = nullptr;
  OK(host_view(space, init, (size_t)n * K, init_buf, &hinit));
  OK(group_slices(g, n, [&](int q, int lo, int hi) {
    return eals_fold_in(g->r[q], EALS_HOST, hi - lo, h.ptr.data() + lo, h.idx.data(), h.vals(val), hinit ? hinit + lo * K : nullptr,
                        n_iter, res.data() + lo * K);
  }));
  return host_result(space, out, res);
}

int eals_group_recommend_vectors(eals_group* g, int32_t space, int32_t n, const double* Q, const int64_t* ex_ptr,
                                 const int32_t* ex_idx, int32_t k, int32_t* items, double* scores) {
  if (!g || (n > 0 && (!Q || !items))) return fail(EALS_ERR_ARG, "null argument");
  if ((ex_ptr == nullptr) != (ex_idx == nullptr)) return fail(EALS_ERR_ARG, "ex_ptr and ex_idx must both be given or both be null");
  OK(check_topk_args(space, n, k));
  OK(group_barrier(g));
  if (n == 0) return EALS_OK;
  const size_t K = (size_t)g->base.factors;
  HostCsr ex;
  if (ex_ptr) OK(ex.load(space, n, ex_ptr, ex_idx, nullptr));
  std::vector<double> q_buf, out_s((size_t)n * k);
  std::vector<int32_t> out_i((size_t)n * k);
  const double* hq = nullptr;
  OK(host_view(space, Q, (size_t)n * K, q_buf, &hq));
  OK(group_slices(g, n, [&](int q, int lo, int hi) {
    return eals_recommend_vectors(g->r[q], EALS_HOST, hi - lo, hq + lo * K, ex_ptr ? ex.ptr.data() + lo : nullptr,
                                  ex_ptr ? ex.idx.data() : nullptr, k, out_i.data() + (size_t)lo * k, out_s.data() + (size_t)lo * k);
  }));
  OK(host_result(space, items, out_i));
  if (scores) OK(host_result(space, scores, out_s));
  return EALS_OK;
}

// Every rank ranks the test entries of the rows it owns (its train rows are the ones to exclude), the ranks at once;
// the sums are added in rank order.
int eals_group_ranking_metrics(eals_group* g, int32_t space, const int64_t* test_ptr, const int32_t* test_idx, int32_t k,
                               int32_t exclude_seen, double means[6], int64_t* n_users, double* per_user, int32_t* ranks) {
  if (!g || !test_ptr || !test_idx || !means || !n_users) return fail(EALS_ERR_ARG, "null argument");
  OK(check_topk_args(space, 0, k));
  OK(group_barrier(g));
  const int M = g->base.n_users;
  HostCsr t;
  OK(t.load(space, M, test_ptr, test_idx, nullptr));
  std::vector<double> sums((size_t)6 * g->n, 0.0), pu(per_user ? (size_t)M * 6 : 0);
  std::vector<int64_t> cnt((size_t)g->n, 0);
  std::vector<int32_t> rk(ranks ? (size_t)t.ptr[(size_t)M] : 0);
  OK(parallel_ranks(g, [&](int q) {
    const int b = g->ub[q];
    return eals_ranking_metrics(g->r[q], EALS_HOST, t.ptr.data(), t.idx.data(), k, exclude_seen, &sums[(size_t)6 * q], &cnt[(size_t)q],
                                per_user ? pu.data() + (size_t)b * 6 : nullptr, ranks ? rk.data() + t.ptr[(size_t)b] : nullptr);
  }));
  int64_t users = 0;
  for (int q = 0; q < g->n; q++) users += cnt[(size_t)q];
  for (int j = 0; j < 6; j++) {
    double s = 0;
    for (int q = 0; q < g->n; q++) s += sums[(size_t)6 * q + j];
    means[j] = users > 0 ? s / (double)users : 0.0;
  }
  *n_users = users;
  if (per_user) OK(host_result(space, per_user, pu));
  if (ranks && !rk.empty()) OK(host_result(space, ranks, rk));
  return EALS_OK;
}

int eals_group_evaluate_user(eals_group* g, int32_t u, int32_t gt_item, int32_t topk, int32_t mode, double out[3]) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  OK(group_barrier(g));
  return eals_evaluate_user(g->r[0], u, gt_item, topk, mode, out);
}

int eals_group_replicas_consistent(eals_group* g, int32_t* ok) {
  if (!g || !ok) return fail(EALS_ERR_ARG, "null argument");
  OK(group_barrier(g));
  uint64_t first[2] = {0, 0};
  *ok = 1;
  for (int q = 0; q < g->n; q++) {
    uint64_t h[2];
    OK(eals_factor_hash(g->r[q], h));
    if (q == 0) { first[0] = h[0]; first[1] = h[1]; }
    else if (h[0] != first[0] || h[1] != first[1]) *ok = 0;
  }
  return EALS_OK;
}

int eals_group_save_factors(eals_group* g, const char* path) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  OK(group_barrier(g));
  return eals_save_factors(g->r[0], path);
}

int eals_group_load_factors(eals_group* g, const char* path) {
  if (!g) return fail(EALS_ERR_ARG, "null group");
  OK(group_barrier(g));
  OK(eals_load_factors(g->r[0], path));
  std::vector<double> wi((size_t)g->base.n_items);
  OK(eals_get_item_weights(g->r[0], EALS_HOST, wi.data()));
  for (int q = 1; q < g->n; q++) {
    eals_model* m = g->r[q];
    CU(cudaSetDevice(g->dev[q]));
    CU(cudaMemcpyAsync(m->Wi, wi.data(), sizeof(double) * wi.size(), cudaMemcpyHostToDevice, m->stream));
    CU(cudaStreamSynchronize(m->stream));
  }
  return group_broadcast_factors(g);
}

int64_t eals_group_kernel_launches(const eals_group* g) {
  int64_t n = 0;
  if (g) for (eals_model* m : g->r) n += m->launches;
  return n;
}

}  // extern "C"
