/* eals_b200.h — C ABI of libeals_b200.so: the device side of the eALS trainer for NVIDIA B200
 * (sm_100a).  Plain pointers and sizes only; no C++ or torch types cross this boundary.
 *
 * What it replaces.  The reference (QihanW/eals_cpp) has no FFI layer: its boundary is the C++
 * class MF_fastALS (MF_fastALS.h:15-80) driven from main.cpp:227-231,49.  Our host class of the
 * same name (include/MF_fastALS.h) keeps that surface and forwards every hot call to the entry
 * points below; each one names the reference member it stands in for.  A maintainer of the
 * reference binds the same symbols (see INTEGRATION.md).
 *
 * Conventions.
 *  - The popularity weights and the factor initialisation run on the HOST inside the library with
 *    the same libm / libstdc++ calls the reference makes (pow; default_random_engine +
 *    normal_distribution), so they are bit-identical to the reference by construction.
 *  - Every function returns 0 (EALS_OK) or a negative eals_status; eals_last_error() gives the
 *    message for the calling thread.  Nothing throws across the ABI.
 *  - One eals_model lives on ONE GPU and is driven by ONE host thread (the reference's methods are
 *    not reentrant either: MF_fastALS.h:40-45).  Multi-GPU = one process (and one model) per GPU;
 *    each model owns a contiguous user range and item range (eals_params.user_begin ...) and holds
 *    full replicas of U and V.  The exchange between half-epochs (all-gather of the updated factor
 *    rows, all-reduce of the partial K x K Gram) is performed by the host on the device buffers
 *    exposed through eals_device_buffer().
 *  - Index arrays are int32 (row/column ids) and int64 (offsets); values are IEEE fp64.
 *    CSR rows ascend by item id, CSC columns ascend by user id, no duplicates: the order
 *    main.cpp:198-205 fills SparseMat.rows/cols in.
 *  - Sweeps are enqueued on the model's stream and return without waiting; calls that hand a value
 *    back to the host (loss, evaluate, get_*) synchronise.  eals_sync() waits explicitly.
 *  - There is no CPU fallback: without a CUDA device every call fails with EALS_ERR_CUDA.
 */
#ifndef EALS_B200_H
#define EALS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EALS_ABI_VERSION 1

typedef enum eals_status {
  EALS_OK = 0,
  EALS_ERR_ARG = -1,         /* null pointer, bad range, unsorted/duplicate indices ...           */
  EALS_ERR_CUDA = -2,        /* CUDA runtime error (no device, launch failure, ...)               */
  EALS_ERR_ALLOC = -3,       /* device or host allocation failed                                  */
  EALS_ERR_STATE = -4,       /* call not valid in the model's current state                       */
  EALS_ERR_UNSUPPORTED = -5  /* e.g. factors > 256                                                */
} eals_status;

typedef enum eals_space { EALS_HOST = 0, EALS_DEVICE = 1 } eals_space;

typedef enum eals_buffer {
  EALS_BUF_U = 0,     /* [n_users][ld]  fp64, ld = eals_leading_dim(), padding columns are zero   */
  EALS_BUF_V = 1,     /* [n_items][ld]                                                            */
  EALS_BUF_SU = 2,    /* [factors][ld]  S cache U^T U (this rank's partial until reduced)         */
  EALS_BUF_SV = 3,    /* [factors][ld]  S cache V^T diag(Wi) V                                    */
  EALS_BUF_WI = 4,    /* [n_items]                                                                */
  EALS_BUF_LOSS_TERMS = 5,/* [4] fp64, see eals_loss_terms                                        */
  EALS_BUF_PC_USER = 6,   /* prediction cache of the owned user rows' nonzeros (CSR order)         */
  EALS_BUF_PC_ITEM = 7    /* prediction cache of the owned item columns' nonzeros (CSC order)      */
} eals_buffer;

typedef enum eals_eval_mode {
  EALS_EVAL_REFERENCE = 0, /* bug-for-bug: int-truncating comparator + libstdc++ heap order
                              (MF_fastALS.cpp:643-651)                                            */
  EALS_EVAL_EXACT = 1      /* rank position = number of strictly larger scores                    */
} eals_eval_mode;

/* Constructor arguments of MF_fastALS (MF_fastALS.h:52-55) that reach the device side.
 * threadNum, showProgress and showLoss stay in the host class (threadNum is dead in the reference
 * too: MF_fastALS.cpp:30). */
typedef struct eals_params {
  int32_t struct_bytes;   /* sizeof(eals_params), for ABI evolution                               */
  int32_t n_users;        /* userCount                                                            */
  int32_t n_items;        /* itemCount                                                            */
  int32_t factors;        /* K, 1..256                                                            */
  int32_t topk;           /* default topK for evaluate                                            */
  double w0;              /* weight of missing data                                               */
  double alpha;           /* popularity exponent                                                  */
  double reg;             /* L2 regularisation                                                    */
  double init_mean;       /* N(mean, stdev) factor initialisation                                 */
  double init_stdev;
  int32_t device;         /* CUDA ordinal                                                         */
  int32_t input_space;    /* eals_space of the matrix pointers given to eals_create               */
  int32_t user_begin;     /* rows [user_begin, user_end) are updated by this model                */
  int32_t user_end;       /*   (0, n_users for a single GPU; 0,0 means "all")                     */
  int32_t item_begin;
  int32_t item_end;
  int32_t flags;          /* EALS_FLAG_*                                                          */
  int32_t reserved;
  /* Multi-rank layout (optional; n_ranks <= 1 means this model is alone).  rank r owns users
   * [user_bounds[r], user_bounds[r+1]) and items [item_bounds[r], item_bounds[r+1]); the entries for
   * `rank` must equal user_begin/user_end and item_begin/item_end.  With it the symmetric
   * prediction cache also works across ranks (see eals_ipc_attach). */
  int32_t n_ranks;        /* 0..8                                                                 */
  int32_t rank;
  int32_t user_bounds[9];
  int32_t item_bounds[9];
} eals_params;

#define EALS_FLAG_SYNC_EACH_CALL 1 /* debugging: synchronise + check after every enqueue          */

typedef struct eals_model eals_model;

int eals_abi_version(void);
const char* eals_last_error(void);
void eals_default_params(eals_params* p); /* run.sh defaults of main.cpp:133-144                  */

/* MF_fastALS::MF_fastALS (MF_fastALS.cpp:29-92) minus the factor initialisation: copies the train
 * matrix to the device (the caller may free its arrays on return), derives the popularity weights
 * Wi (MF_fastALS.cpp:55-72) and allocates U, V, SU, SV (zero).  row_val / col_val may
 * be NULL: all ratings 1 (what the reference's loader stores, main.cpp:184-185,202); otherwise the
 * value is both the rating and its confidence weight (W is a copy of the ratings,
 * MF_fastALS.cpp:75-82).  All six arrays describe the FULL matrix even when the model owns a
 * sub-range. */
int eals_create(const eals_params* params, const int64_t* row_ptr, const int32_t* col_idx,
                const double* row_val, const int64_t* col_ptr, const int32_t* row_idx,
                const double* col_val, eals_model** out);
int eals_destroy(eals_model* m);

/* MF_fastALS::setTrain (MF_fastALS.cpp:94-104): replace the train matrix (same shape). Wi is kept,
 * as in the reference. */
int eals_set_train(eals_model* m, int32_t input_space, const int64_t* row_ptr,
                   const int32_t* col_idx, const double* row_val, const int64_t* col_ptr,
                   const int32_t* row_idx, const double* col_val);

/* U.init / V.init / initS of the constructor (MF_fastALS.cpp:85-90, DenseMat.cpp:54-62): the
 * default-seeded libstdc++ minstd_rand0 + polar normal stream, the SAME stream for U and V, then
 * both S caches. */
int eals_init_factors(eals_model* m);
/* Host seconds the last eals_init_factors spent generating the normal stream (parallel skip-ahead over the
 * reference's LCG, bit-identical to the sequential loop). */
int eals_init_seconds(eals_model* m, double* host_stream_seconds);
/* The stream alone into a host array (no device needed): what eals_init_factors uploads. */
int eals_debug_init_stream(double mean, double stdev, double* out, int64_t n);

/* MF_fastALS::setUV (MF_fastALS.cpp:106-110), working: dense row-major [n][factors] fp64 in the
 * given space; either pointer may be NULL to keep that side.  Refreshes the S caches (initS). */
int eals_set_factors(eals_model* m, int32_t space, const double* U, const double* V);
int eals_get_factors(eals_model* m, int32_t space, double* U, double* V);
/* One factor row to the host: out[factors] = U[row] (which = EALS_BUF_U) or V[row] (EALS_BUF_V) —
 * U.matrix[u] / V.matrix[i] of the reference (MF_fastALS.h:31-32); what update_user_SU /
 * update_item_SV callers and the online updateModel (MF_fastALS.cpp:223-242) need per step. */
int eals_get_factor_row(eals_model* m, int32_t which, int32_t row, double* out);

/* Factor checkpoint (SURVEY.md §8 f4; the reference has only the broken setUV, MF_fastALS.cpp:106-110):
 * U, V and Wi to / from a binary file (header: magic "EALSB200", version, factors, n_users, n_items; then
 * U [n_users][factors], V [n_items][factors], Wi [n_items], little-endian fp64).  load checks the shape,
 * replaces the factors and weights and rebuilds both S caches (initS); training then resumes as if the
 * model had never been torn down. */
int eals_save_factors(eals_model* m, const char* path);
int eals_load_factors(eals_model* m, const char* path);

/* Public member Wi (MF_fastALS.h:46). set refreshes SV. */
int eals_set_item_weights(eals_model* m, int32_t space, const double* Wi);
int eals_get_item_weights(eals_model* m, int32_t space, double* Wi);

/* initS (MF_fastALS.cpp:583-595) and read-back of SU, SV as dense [factors][factors]. */
int eals_refresh_S(eals_model* m);
int eals_get_S(eals_model* m, int32_t space, double* SU, double* SV);

/* One half-epoch each, as buildModel runs them (MF_fastALS.cpp:127-132 and :146-152):
 * update_user_thread for every owned user (:243-322) then the SU refresh (:324-335; recomputed as
 * a Gram over the owned rows instead of patched row by row); same for items (:338-407, :409-422).
 * Enqueue-only.  With more than one rank the host must all-gather the updated rows of U (V) and
 * all-reduce SU (SV) before the next half-epoch. */
int eals_update_user(eals_model* m);
int eals_update_item(eals_model* m);

/* n epochs = n x (eals_update_user, eals_update_item).  With use_graph != 0 the epoch is captured once into a
 * CUDA graph (after one ordinary epoch, so that scratch sizes and the symmetric prediction cache are in their
 * steady state) and REPLAYED: the yelp-sized configurations are launch-bound — ~170 kernels of a few
 * microseconds per epoch — and a replayed graph removes the per-launch cost.  Bit-identical to the ordinary
 * calls (same kernels, same order).  The graph is rebuilt after eals_set_train / eals_set_stream; the phase
 * timers do not advance during replayed epochs.  Single-rank models only (use_graph is ignored otherwise). */
int eals_run_epochs(eals_model* m, int32_t n, int32_t use_graph);

/* The two stages of the above, separately (for hosts that overlap the exchange). */
int eals_sweep_users(eals_model* m);
int eals_sweep_items(eals_model* m);
int eals_gram_users(eals_model* m);
int eals_gram_items(eals_model* m);

/* Single-row forms MF_fastALS::update_user_thread(u) / update_item_thread(i) — no S refresh — and
 * the rank-1 S patches update_user_SU / update_item_SV (MF_fastALS.cpp:324-335, 409-422) with
 * host vectors of `factors` doubles. */
int eals_update_user_row(eals_model* m, int32_t u);
int eals_update_item_row(eals_model* m, int32_t i);
int eals_patch_SU(eals_model* m, const double* old_row, const double* new_row);
int eals_patch_SV(eals_model* m, int32_t i, const double* old_row, const double* new_row);

/* MF_fastALS::loss (MF_fastALS.cpp:184-206).  terms[0] = sum over OWNED users of the per-nonzero
 * part, terms[1] = |U owned rows|^2, terms[2] = |V owned rows|^2, terms[3] = sum_u u^T SV u over ALL
 * users, taken as <U^T U, SV>_F: the cached SU while it is fresh, a scratch Gram of the current U after
 * single-row user updates (which, as in the reference, leave SU stale).  loss = terms[0] + reg*(terms[1]+terms[2]) +
 * terms[3]; eals_loss forms that for a single-rank model. */
int eals_loss_terms(eals_model* m, double terms[4]);
int eals_loss(eals_model* m, double* loss);

/* MF_fastALS::predict (MF_fastALS.cpp:208-221). */
int eals_predict(eals_model* m, int32_t u, int32_t i, double* score);

/* evaluate_model + evaluate_for_user (main.cpp:37-65, MF_fastALS.cpp:620-662) over the OWNED
 * users.  gt_items: host array indexed by global user id (n_users entries).  sums[3] = sum of
 * hit-ratio, NDCG and reciprocal rank ("prec") over the owned users — divide by n_users after
 * summing across ranks.  Optional per-user host outputs have (user_end-user_begin) entries;
 * count_larger is the number of items scoring strictly above the held-out one, capped at topk+1. */
int eals_evaluate(eals_model* m, const int32_t* gt_items, int32_t topk, int32_t mode,
                  double sums[3], double* hr, double* ndcg, double* prec, int32_t* count_larger);
int eals_evaluate_user(eals_model* m, int32_t u, int32_t gt_item, int32_t topk, int32_t mode,
                       double out[3]);
/* How the last eals_evaluate or eals_ranking_metrics ran (for ranking metrics "users" are test entries, and out[0] is
 * 1 only when every chunk of entries went through the filter): out[0] = 1 when the scores went through the tcgen05
 * fp16 filter (lists of >= 128 users; every close call re-scored in fp64 with the reference's operation order, so
 * the results are identical to the all-fp64 scan), 0 for the exact fp64 tile scan; out[1] = users whose certain count stayed
 * <= topK after the filter (candidates), out[2] = (user, item) pairs re-scored exactly; out[3], out[4], out[5] =
 * users, items and device microseconds of the filter's FIRST item block (every user against the highest-norm
 * items: the one launch of known shape, 2 * users * items * roundup(factors, 64) flop — the tensor roofline). */
int eals_eval_stats(eals_model* m, int64_t out[6]);

/* Top-k retrieval: for each of the n users (global ids, owned by this model), the k items of highest score,
 * score = predict(u, i) bit for bit, ordered by score descending and item id ascending.  With exclude_seen != 0
 * the items of the user's row of the current train matrix (after eals_set_train) are left out.  Slots a user
 * cannot fill (fewer than k eligible items) hold item -1 and score -inf.  items: [n][k] int32, scores: [n][k]
 * double or NULL; users, items and scores are host or device memory as `space` says (EALS_HOST / EALS_DEVICE).
 * 1 <= k <= 1024.  Lists of >= 128 users with factors <= 256 go through the tcgen05 filter (every output decided
 * by exact fp64 comparisons; the same result as the exact engine); EALS_EVAL_SCALAR=1 forces the exact engine. */
int eals_recommend(eals_model* m, int32_t space, int32_t n, const int32_t* users, int32_t k, int32_t exclude_seen,
                   int32_t* items, double* scores);
/* How the last eals_recommend ran (7 values): out[0] = engine (1 tcgen05 filter, 0 exact fp64), out[1] = items of
 * the exact seed, out[2] = candidate pairs re-scored exactly, out[3] = users still in the working set after the
 * first item block, out[4], out[5], out[6] = users, items and device microseconds of the filter's first item
 * block (2 * users * items * roundup(factors, 64) flop). */
int eals_recommend_stats(eals_model* m, int64_t out[7]);

/* Fold-in: the user vectors the eALS online step computes for n histories without touching the model.  row_ptr,
 * col_idx and val are a CSR of n rows over the model's items with the rules of eals_set_train (indices in
 * [0, n_items), strictly ascending inside a row; val NULL = every rating 1; row_ptr[0] may be non-zero).  Each row
 * starts from init ([n][factors], NULL: zeros) and gets n_iter >= 1 passes of update_user_thread
 * (MF_fastALS.cpp:243-322) against the model's current V, SV, Wi and reg, every pass recomputing the row's
 * predictions; an empty row keeps its init.  out: [n][factors], dense rows.  All arrays are host or device memory
 * as `space` says.  U, V, the S caches, Wi, the prediction-cache state and the timers stay exactly as they were.
 * With init = U[u], n_iter = 1 and u's train row the result is U[u] after eals_update_user_row(u), bit for bit. */
int eals_fold_in(eals_model* m, int32_t space, int32_t n, const int64_t* row_ptr, const int32_t* col_idx, const double* val,
                 const double* init, int32_t n_iter, double* out);
/* eals_recommend for arbitrary query vectors: Q is [n][factors] (finite, checked on the device) and row s stands in
 * for U[u], so score = predict's seq_dot(Q[s], V[i]) — bit-identical to eals_recommend when Q[s] == U[u] — with the
 * same order, padding, 1 <= k <= 1024, factors <= 256 and engines.  ex_ptr / ex_idx: an optional CSR of n rows of
 * items to leave out of row s's list (both or neither; validated like a history), e.g. the history a vector was
 * folded in from.  eals_recommend_stats reports the last eals_recommend or eals_recommend_vectors call. */
int eals_recommend_vectors(eals_model* m, int32_t space, int32_t n, const double* Q, const int64_t* ex_ptr, const int32_t* ex_idx,
                           int32_t k, int32_t* items, double* scores);

/* Similar items (which = EALS_BUF_V, catalogue V of n_items rows) or similar users (which = EALS_BUF_U, catalogue U
 * of n_users rows): for each of the n ids, the k other rows of the catalogue of highest cosine score, ordered by
 * score descending and id ascending.  With |y| = sqrt(seq_dot(y, y)) (predict's sequential fp64 sum of separately
 * rounded products, correctly rounded square root) and y^ = y / |y| per factor (a zero row stays zero), the score of
 * (q, r) is seq_dot(y^_q, y^_r) bit for bit.  Only the query's own row is left out: other rows with the same vector
 * stay and tie.  Slots that cannot be filled hold id -1 and score -inf.  ids may be any row in [0, n_Y) on any rank
 * (U and V are replicated).  out_ids: [n][k] int32, scores: [n][k] double or NULL; ids, out_ids and scores are host or
 * device memory as `space` says.  1 <= k <= 1024, factors <= 256, the engines of eals_recommend.  The model stays
 * exactly as it was; eals_recommend_stats reports the last call. */
int eals_similar(eals_model* m, int32_t which, int32_t space, int32_t n, const int32_t* ids, int32_t k, int32_t* out_ids,
                 double* scores);

/* Ranking metrics at k on a held-out test matrix.  test_ptr / test_idx: a CSR with one row per user (n_users + 1
 * offsets, the rules of eals_set_train; this model reads the rows of its own users).  For a test entry (u, g) the
 * rank is g's 0-based position in the list eals_recommend(u, k, exclude_seen) returns, or -1 when g is not in it (a
 * test item in u's train row is always -1 with exclude_seen).  Per user with n_u > 0 test items and H the hit ranks:
 * [0] hit rate (H non-empty), [1] precision |H| / k, [2] recall |H| / n_u, [3] NDCG sum_{h in H} ln 2 / ln(h + 2)
 * over the same sum for 0 .. min(k, n_u) - 1, [4] MAP (1 / min(k, n_u)) sum_{h in H} #{h' in H : h' <= h} / (h + 1),
 * [5] MRR 1 / (min H + 1).  sums[6]: the sums over this model's users with test items, in user order, *n_users their
 * number; per_user ([user_end - user_begin][6], 0 for users without test items) and ranks (one per test entry of
 * the owned rows, in CSR order) are optional.  1 <= k <= 1024; every rank is decided by exact fp64 comparisons
 * (tcgen05 filter for lists of >= 128 entries, the exact engine otherwise or with EALS_EVAL_SCALAR=1, both giving
 * the same result).  Arrays are host or device memory as `space` says.  The model stays exactly as it was;
 * eals_eval_stats reports this call like an evaluate. */
int eals_ranking_metrics(eals_model* m, int32_t space, const int64_t* test_ptr, const int32_t* test_idx, int32_t k,
                         int32_t exclude_seen, double sums[6], int64_t* n_users, double* per_user, int32_t* ranks);

/* Plumbing for the host layer. */
int eals_leading_dim(const eals_model* m);                 /* ld of U/V/SU/SV rows, in doubles   */
int eals_device_buffer(eals_model* m, int32_t which, void** dev_ptr, int64_t* bytes);
int eals_stream(eals_model* m, void** cuda_stream);        /* cudaStream_t the model enqueues on  */
/* Make the model enqueue on a caller-owned stream (e.g. the one the host's NCCL calls are ordered
 * against; NULL is the legacy default stream), or back on its own stream when restore_own != 0.
 * Synchronises the old stream first. */
int eals_set_stream(eals_model* m, void* cuda_stream, int32_t restore_own);
int eals_sync(eals_model* m);
/* 64-bit position-dependent checksums of the bit patterns of this model's U (out[0]) and V (out[1]) replicas,
 * computed on the device.  With several ranks every replica must give the same pair after every half-epoch
 * (the exchange is a copy; only the K x K Gram all-reduce involves arithmetic, and its result is the same
 * on all ranks) — the multi-GPU consistency check of bench.py and tests.  Synchronises. */
int eals_factor_hash(eals_model* m, uint64_t out[2]);
/* Fused exchange of the updated factor rows (one process per GPU, all on one NVLink box).
 * eals_ipc_handle writes the 64-byte CUDA IPC handle of this model's U or V replica
 * (which = EALS_BUF_U / EALS_BUF_V); after the host has exchanged the handles, eals_ipc_attach maps
 * the n_peers (<= 7) OTHER ranks' replicas (handles = n_peers x 64 bytes, in rank order with the own
 * rank left out).  From then on the sweep kernels store every finished row into all replicas
 * themselves, so no all-gather is needed after a sweep — only the all-reduce of the partial Gram,
 * which also orders the stores.  The same two calls with which = EALS_BUF_PC_USER / EALS_BUF_PC_ITEM
 * share the prediction caches (needs eals_params.n_ranks > 1): a sweep then leaves the prediction of
 * each nonzero with the rank that will start from it in the next half-epoch, and no rank has to
 * re-gather factor rows to rebuild it.  Handles must be exchanged again after eals_set_train.
 * eals_ipc_detach unmaps all peers (also done by eals_destroy). */
#define EALS_IPC_HANDLE_BYTES 64
int eals_ipc_handle(eals_model* m, int32_t which, void* handle_out);
int eals_ipc_attach(eals_model* m, int32_t which, int32_t n_peers, const void* handles);
int eals_ipc_detach(eals_model* m);
/* A prediction cache that has to grow in eals_set_train is not freed while peers may still map it:
 * eals_ipc_generation changes when that happened on this rank (then ALL ranks exchange handles and attach
 * again), eals_ipc_gc frees the retired buffers once every peer has re-attached.  With unchanged
 * generations on all ranks the existing mappings stay valid and no handle exchange is needed. */
int eals_ipc_generation(eals_model* m);
int eals_ipc_gc(eals_model* m);
int64_t eals_nnz(const eals_model* m);                     /* nonzeros of the owned user rows     */
int64_t eals_kernel_launches(const eals_model* m);         /* kernels launched so far             */
/* Device milliseconds of the most recent call of each kind: [0] user sweep, [1] user Gram,
 * [2] item sweep, [3] item Gram, [4] loss, [5] evaluate.  Synchronises. */
int eals_timings(eals_model* m, double ms[6]);
/* Device milliseconds and call counts of every call since the last reset, same six slots; each call
 * is bracketed by CUDA events on the model's stream, nothing synchronises until this query. */
int eals_timings_total(eals_model* m, double ms[6], int64_t calls[6], int32_t reset);
/* Accumulated device milliseconds of the sweep sub-phases since the last reset of
 * eals_timings_total: [0..2] user side heavy-row slab pipeline / one-CTA rows / warp rows,
 * [3..5] the same for the item side.  Query BEFORE eals_timings_total(reset=1). */
int eals_timings_detail(eals_model* m, double ms[6], int64_t calls[6]);

/* ---------------------------------------------------------------------------------------------------------
 * eals_group — N GPUs of one box behind ONE object, driven by ONE host thread like the reference's class
 * (MF_fastALS.h:52-55 ctor, MF_fastALS.cpp:112-161 buildModel).  Rank r lives on devices[r] (NULL: 0..N-1)
 * and owns a contiguous user range and item range, chosen by a per-row cost model (eals_partition); U and V
 * are replicated.  A half-epoch is: every rank's sweep (finished rows stored into ALL replicas by the
 * kernels themselves, over NVLink peer pointers), every rank's partial K x K Gram, and a one-shot
 * all-reduce over peer memory that adds the partials in rank order (all ranks end with bit-identical
 * S caches).  Everything is ordered by CUDA events between the ranks' streams; no call below synchronises
 * the host inside an epoch.  `devices` may repeat a GPU ("virtual ranks": the whole sharded path on one
 * GPU — how single-GPU CI covers it).  All other entry points mean what their eals_* namesakes mean, over
 * the whole matrix; evaluation outputs are indexed by GLOBAL user id and `means` are already divided by
 * n_users. */
typedef struct eals_group eals_group;
int eals_group_create(const eals_params* params, int32_t n_ranks, const int32_t* devices,
                      const int64_t* row_ptr, const int32_t* col_idx, const double* row_val,
                      const int64_t* col_ptr, const int32_t* row_idx, const double* col_val, eals_group** out);
int eals_group_destroy(eals_group* g);
int eals_group_size(const eals_group* g);
int eals_group_model(eals_group* g, int32_t rank, eals_model** out);        /* borrowed: timings, buffers, hashes */
int eals_group_bounds(const eals_group* g, int32_t* user_bounds, int32_t* item_bounds);   /* n_ranks + 1 each */
int eals_group_set_train(eals_group* g, int32_t input_space, const int64_t* row_ptr, const int32_t* col_idx,
                         const double* row_val, const int64_t* col_ptr, const int32_t* row_idx, const double* col_val);
int eals_group_init_factors(eals_group* g);
int eals_group_set_factors(eals_group* g, int32_t space, const double* U, const double* V);
int eals_group_get_factors(eals_group* g, int32_t space, double* U, double* V);
int eals_group_get_factor_row(eals_group* g, int32_t which, int32_t row, double* out);
int eals_group_get_S(eals_group* g, int32_t space, double* SU, double* SV);
int eals_group_set_item_weights(eals_group* g, int32_t space, const double* Wi);
int eals_group_get_item_weights(eals_group* g, int32_t space, double* Wi);
int eals_group_update_user(eals_group* g);                                  /* MF_fastALS.cpp:127-132 */
int eals_group_update_item(eals_group* g);                                  /* MF_fastALS.cpp:146-152 */
int eals_group_update_user_row(eals_group* g, int32_t u);                   /* update_user_thread(u)  */
int eals_group_update_item_row(eals_group* g, int32_t i);                   /* update_item_thread(i)  */
int eals_group_patch_SU(eals_group* g, const double* old_row, const double* new_row);
int eals_group_patch_SV(eals_group* g, int32_t i, const double* old_row, const double* new_row);
int eals_group_loss(eals_group* g, double* loss);
int eals_group_predict(eals_group* g, int32_t u, int32_t i, double* score);
int eals_group_evaluate(eals_group* g, const int32_t* gt_items, int32_t topk, int32_t mode, double means[3],
                        double* hr, double* ndcg, double* prec, int32_t* count_larger);
int eals_group_evaluate_user(eals_group* g, int32_t u, int32_t gt_item, int32_t topk, int32_t mode, double out[3]);
/* eals_recommend over the whole user range: each user is answered by the rank that owns it, results in input order. */
int eals_group_recommend(eals_group* g, int32_t space, int32_t n, const int32_t* users, int32_t k, int32_t exclude_seen,
                         int32_t* items, double* scores);
/* eals_fold_in / eals_recommend_vectors over the group: the queries go to the ranks in balanced contiguous slices
 * (V, SV and Wi are replicated), results in input order. */
int eals_group_fold_in(eals_group* g, int32_t space, int32_t n, const int64_t* row_ptr, const int32_t* col_idx,
                       const double* val, const double* init, int32_t n_iter, double* out);
int eals_group_recommend_vectors(eals_group* g, int32_t space, int32_t n, const double* Q, const int64_t* ex_ptr,
                                 const int32_t* ex_idx, int32_t k, int32_t* items, double* scores);
/* eals_similar over the group: the queries go to the ranks in balanced contiguous slices (U and V are replicated),
 * results in input order. */
int eals_group_similar(eals_group* g, int32_t which, int32_t space, int32_t n, const int32_t* ids, int32_t k, int32_t* out_ids,
                       double* scores);
/* eals_ranking_metrics over the whole matrix: each rank on the rows it owns, sums added in rank order.  means[6] are
 * divided by *n_users (0 when no user has test items); per_user is [n_users][6], ranks in test-entry order. */
int eals_group_ranking_metrics(eals_group* g, int32_t space, const int64_t* test_ptr, const int32_t* test_idx, int32_t k,
                               int32_t exclude_seen, double means[6], int64_t* n_users, double* per_user, int32_t* ranks);
int eals_group_sync(eals_group* g);
int eals_group_replicas_consistent(eals_group* g, int32_t* ok);             /* all U / V replicas bit-identical */
int eals_group_save_factors(eals_group* g, const char* path);
int eals_group_load_factors(eals_group* g, const char* path);
int64_t eals_group_kernel_launches(const eals_group* g);
/* Row ranges of (nearly) equal COST for n_ranks ranks: bounds[0] = 0 <= ... <= bounds[n_ranks] = n_rows.  The
 * cost of a row follows the kernel family its length selects (ns per row / per nonzero measured on B200).
 * `ptr` is the host offsets array of that orientation. */
int eals_partition(const int64_t* ptr, int32_t n_rows, int32_t n_ranks, int32_t* bounds);

#ifdef __cplusplus
}
#endif
#endif /* EALS_B200_H */
