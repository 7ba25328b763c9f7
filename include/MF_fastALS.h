// MF_fastALS.h — C++ drop-in host class over libeals_b200.so (include/eals_b200.h).
//
// Mirrors the public surface of the reference's class MF_fastALS (MF_fastALS.h:15-80): same
// constructor argument list (MF_fastALS.h:52-55), same method names and meanings, same stdout lines
// (MF_fastALS.cpp:134,155,179).  Every hot call is forwarded to the C ABI; nothing is computed on
// the CPU here apart from flattening the caller's SparseMat into CSR/CSC arrays.
//
// The class is a template over the caller's container types so that it works with the reference's
// own SparseMat / Rating (duck-typed: `n_r`, `n_c`, `rows[u].n`, `rows[u].spv_in[j]`,
// `rows[u].spv_do[j]`, `cols[i]...`; `Rating::itemId`) as well as with the small CSR-backed
// containers in eals_host_types.h.  A reference maintainer writes
//
//     #include "SparseMat.h"            // theirs
//     #include "Rating.h"               // theirs
//     #include "MF_fastALS.h"           // this file instead of theirs
//     using MF_fastALS = eals_b200::MF_fastALS_T<SparseMat, Rating>;
//
// and main.cpp:227-231 compiles unchanged (see INTEGRATION.md).  Differences from the reference, all
// deliberate (SURVEY.md §9 "Drop"): the object drives n_gpus GPUs of the box (trailing constructor arguments
// `device`, `n_gpus`, `devices`; default one GPU) through eals_group — users and items sharded, U / V
// replicated, the exchange inside the library; the object is non-copyable (the reference double-frees when
// copied, main.cpp:37 / MF_fastALS.cpp:664-673); inputs are copied to the device at construction,
// so the caller's arrays need not outlive the model; errors throw std::runtime_error with the
// library's message instead of being ignored; runOneIteration() refreshes the S caches.
#ifndef EALS_B200_MF_FASTALS_H
#define EALS_B200_MF_FASTALS_H

#include <algorithm>
#include <chrono>
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <iostream>
#include <stdexcept>
#include <string>
#include <vector>

#include "eals_b200.h"

namespace eals_b200 {

inline void check(int code, const char* what) {
  if (code != EALS_OK)
    throw std::runtime_error(std::string(what) + ": " + eals_last_error() + " (code " + std::to_string(code) + ")");
}

template <class SparseMatT, class RatingT>
class MF_fastALS_T {
 public:
  // public data members of the reference that callers read (MF_fastALS.h:19-29,48-49)
  int factors, maxIter;
  double reg, w0, init_mean, init_stdev;
  int itemCount, userCount, topK;
  double alpha;
  bool showprogress, showloss;
  std::vector<RatingT> testRatings;

  MF_fastALS_T(const SparseMatT& trainMatrix, const std::vector<RatingT>& testRatings_, int topK_,
               int threadNum, int factors_, int maxIter_, double w0_, double alpha_, double reg_,
               double init_mean_, double init_stdev_, bool showProgress, bool showLoss, int userCount_,
               int itemCount_, int device = 0, int n_gpus = 1, const int* devices = nullptr)
      : factors(factors_), maxIter(maxIter_), reg(reg_), w0(w0_), init_mean(init_mean_),
        init_stdev(init_stdev_), itemCount(itemCount_), userCount(userCount_), topK(topK_),
        alpha(alpha_), showprogress(showProgress), showloss(showLoss), testRatings(testRatings_) {
    (void)threadNum;  // accepted and ignored, as in the reference (MF_fastALS.cpp:30)
    eals_params p;
    eals_default_params(&p);
    p.n_users = userCount; p.n_items = itemCount; p.factors = factors; p.topk = topK;
    p.w0 = w0; p.alpha = alpha; p.reg = reg; p.init_mean = init_mean; p.init_stdev = init_stdev;
    p.device = device; p.input_space = EALS_HOST;
    mat_ = flatten(trainMatrix);
    const Flat& f = mat_;
    // rank r on devices[r]; default: `device`, device + 1, ...  (a repeated id = several ranks on one GPU)
    std::vector<int32_t> dev((size_t)std::max(1, n_gpus));
    for (size_t r = 0; r < dev.size(); r++) dev[r] = devices ? devices[r] : device + (int)r;
    check(eals_group_create(&p, (int32_t)dev.size(), dev.data(), f.row_ptr.data(), f.col_idx.data(), f.rv(),
                            f.col_ptr.data(), f.row_idx.data(), f.cv(), &g_), "eals_group_create");
    check(eals_group_init_factors(g_), "eals_group_init_factors");   // U.init, V.init, initS (MF_fastALS.cpp:85-90)
  }
  ~MF_fastALS_T() { eals_group_destroy(g_); }
  MF_fastALS_T(const MF_fastALS_T&) = delete;
  MF_fastALS_T& operator=(const MF_fastALS_T&) = delete;

  void setTrain(const SparseMatT& trainMatrix) {   // MF_fastALS.cpp:94-104
    mat_ = flatten(trainMatrix);
    upload_matrix();
  }
  // MF_fastALS.cpp:106-110, working: dense row-major [userCount][factors] / [itemCount][factors].
  void setUV(const double* U, const double* V) { check(eals_group_set_factors(g_, EALS_HOST, U, V), "eals_group_set_factors"); }
  // same from DenseMat-like objects exposing double** matrix
  template <class DenseMatT>
  void setUV(const DenseMatT& U, const DenseMatT& V) {
    std::vector<double> u((size_t)userCount * factors), v((size_t)itemCount * factors);
    for (int r = 0; r < userCount; r++) for (int c = 0; c < factors; c++) u[(size_t)r * factors + c] = U.matrix[r][c];
    for (int r = 0; r < itemCount; r++) for (int c = 0; c < factors; c++) v[(size_t)r * factors + c] = V.matrix[r][c];
    setUV(u.data(), v.data());
  }
  void getUV(double* U, double* V) { check(eals_group_get_factors(g_, EALS_HOST, U, V), "eals_group_get_factors"); }
  void getS(double* SU, double* SV) { check(eals_group_get_S(g_, EALS_HOST, SU, SV), "eals_group_get_S"); }

  // one half-epoch each (MF_fastALS.cpp:127-132, 146-152)
  void update_user() { check(eals_group_update_user(g_), "eals_group_update_user"); }
  void update_item() { check(eals_group_update_item(g_), "eals_group_update_item"); }

  void buildModel() {   // MF_fastALS.cpp:112-161
    double loss_pre = DBL_MAX;
    for (int iter = 0; iter < maxIter; iter++) {
      auto t0 = std::chrono::steady_clock::now();
      update_user();
      check(eals_group_sync(g_), "eals_group_sync");
      const double t_user = seconds_since(t0);
      std::cout << "Time of user_update: " << t_user << std::endl;
      t0 = std::chrono::steady_clock::now();
      update_item();
      check(eals_group_sync(g_), "eals_group_sync");
      const double t_item = seconds_since(t0);
      std::cout << "Time of item_update: " << t_item << std::endl;
      if (showloss) loss_pre = showLoss(iter, t_user + t_item, loss_pre);
    }
  }
  void runOneIteration() { update_user(); update_item(); }

  double showLoss(int iter, double time, double loss_pre) {   // MF_fastALS.cpp:175-182
    auto t0 = std::chrono::steady_clock::now();
    const double loss_cur = loss();
    const std::string symbol = loss_pre >= loss_cur ? "-" : "+";
    std::cout << "Iter=" << iter << " " << time << " " << symbol << " loss:" << loss_cur << " "
              << seconds_since(t0) << std::endl;
    return loss_cur;
  }
  double loss() { double l = 0; check(eals_group_loss(g_, &l), "eals_group_loss"); return l; }
  double predict(int u, int i) { double s = 0; check(eals_group_predict(g_, u, i, &s), "eals_group_predict"); return s; }

  // MF_fastALS.cpp:620-662 — {hit ratio, NDCG, reciprocal rank}; reproduces the reference's ranking
  // (int-truncating comparator) unless exact is set.
  std::vector<double> evaluate_for_user(int u, int gtItem, int topK_, bool exact = false) {
    std::vector<double> r(3);
    check(eals_group_evaluate_user(g_, u, gtItem, topK_, exact ? EALS_EVAL_EXACT : EALS_EVAL_REFERENCE, r.data()),
          "eals_group_evaluate_user");
    return r;
  }
  // evaluate_model (main.cpp:37-65) over all users at once: means of the three metrics.
  std::vector<double> evaluate(bool exact = false) {
    std::vector<int32_t> gt((size_t)userCount);
    for (int u = 0; u < userCount; u++) gt[u] = testRatings[u].itemId;
    std::vector<double> s(3);
    check(eals_group_evaluate(g_, gt.data(), topK, exact ? EALS_EVAL_EXACT : EALS_EVAL_REFERENCE, s.data(), nullptr,
                              nullptr, nullptr, nullptr), "eals_group_evaluate");   // means over ALL users (main.cpp:60-62)
    return s;
  }

  // Online update (MF_fastALS.cpp:223-242): add interaction (u, i) with rating 1 (= w_new), give a
  // brand-new item the weight w0 / itemCount (SV follows), then 10 alternating single-row updates.
  // The reference appends past the capacity of its SparseVec arrays and leaves SU / SV stale between
  // the row updates (SURVEY.md §9); here the entry goes to its sorted position and, with patch_S
  // (default), the S caches follow every row update as update_user_SU / update_item_SV intend.
  // patch_S = false reproduces the reference's arithmetic (stale caches).
  void updateModel(int u, int i, bool patch_S = true, int maxIterOnline = 10) {
    if (u < 0 || u >= userCount || i < 0 || i >= itemCount) throw std::out_of_range("updateModel: (u, i) outside the matrix");
    if (insert_entry(u, i)) upload_matrix();
    std::vector<double> Wi((size_t)itemCount);
    check(eals_group_get_item_weights(g_, EALS_HOST, Wi.data()), "eals_group_get_item_weights");
    if (Wi[(size_t)i] == 0.0) {   // a new item
      Wi[(size_t)i] = w0 / itemCount;
      check(eals_group_set_item_weights(g_, EALS_HOST, Wi.data()), "eals_group_set_item_weights");   // rebuilds SV too
    }
    std::vector<double> before((size_t)factors), after((size_t)factors);
    for (int it = 0; it < maxIterOnline; it++) {
      if (patch_S) check(eals_group_get_factor_row(g_, EALS_BUF_U, u, before.data()), "eals_group_get_factor_row");
      update_user_thread(u);
      if (patch_S) {
        check(eals_group_get_factor_row(g_, EALS_BUF_U, u, after.data()), "eals_group_get_factor_row");
        update_user_SU(before.data(), after.data());
        check(eals_group_get_factor_row(g_, EALS_BUF_V, i, before.data()), "eals_group_get_factor_row");
      }
      update_item_thread(i);
      if (patch_S) {
        check(eals_group_get_factor_row(g_, EALS_BUF_V, i, after.data()), "eals_group_get_factor_row");
        update_item_SV(i, before.data(), after.data());
      }
    }
  }

  // Top-k retrieval: for each user the k items of highest score (= predict(u, i) bit for bit), ties by item id,
  // the user's train items left out with exclude_seen.  Row-major [users.size()][k]; slots that cannot be filled
  // hold item -1 and score -inf.  1 <= k <= 1024.
  struct Recommendations { std::vector<int32_t> items; std::vector<double> scores; };
  Recommendations recommend(const std::vector<int>& users, int k, bool exclude_seen = true) {
    Recommendations r;
    std::vector<int32_t> u(users.begin(), users.end());
    r.items.resize(u.size() * (size_t)std::max(k, 0));
    r.scores.resize(r.items.size());
    check(eals_group_recommend(g_, EALS_HOST, (int32_t)u.size(), u.data(), k, exclude_seen ? 1 : 0, r.items.data(),
                               r.scores.data()), "eals_group_recommend");
    return r;
  }
  // Fold-in: user vectors for n histories (CSR over the items: row_ptr of n + 1 offsets, ascending col_idx, ratings
  // in val or all 1 when it is empty), n_iter passes of update_user_thread from init ([n][factors], empty: zeros)
  // against the current model, which stays as it is.  Row-major [n][factors].
  std::vector<double> fold_in(const std::vector<int64_t>& row_ptr, const std::vector<int32_t>& col_idx,
                              const std::vector<double>& val = {}, const std::vector<double>& init = {}, int n_iter = 10) {
    const int n = row_ptr.empty() ? 0 : (int)row_ptr.size() - 1;
    std::vector<double> out((size_t)n * factors);
    const int32_t none = 0;
    check(eals_group_fold_in(g_, EALS_HOST, n, row_ptr.data(), col_idx.empty() ? &none : col_idx.data(),
                             val.empty() ? nullptr : val.data(), init.empty() ? nullptr : init.data(), n_iter, out.data()),
          "eals_group_fold_in");
    return out;
  }
  // recommend() for query vectors Q ([n][factors] row-major, e.g. from fold_in), the items of row s of the CSR
  // ex_ptr / ex_idx left out of row s's list (ex_ptr empty: no exclusion).
  Recommendations recommend_vectors(const std::vector<double>& Q, int k, const std::vector<int64_t>& ex_ptr = {},
                                    const std::vector<int32_t>& ex_idx = {}) {
    const int n = (int)(Q.size() / (size_t)factors);
    Recommendations r;
    r.items.resize((size_t)n * (size_t)std::max(k, 0));
    r.scores.resize(r.items.size());
    const int32_t none = 0;
    check(eals_group_recommend_vectors(g_, EALS_HOST, n, Q.data(), ex_ptr.empty() ? nullptr : ex_ptr.data(),
                                       ex_ptr.empty() ? nullptr : (ex_idx.empty() ? &none : ex_idx.data()), k, r.items.data(),
                                       r.scores.data()), "eals_group_recommend_vectors");
    return r;
  }
  // Similar items / similar users: for each id the k other items (users) of highest cosine score, seq_dot of the rows
  // normalised by their norm sqrt(seq_dot(y, y)), ties by id ascending; only the query itself is left out.
  // Row-major [ids.size()][k]; slots that cannot be filled hold -1 and -inf.  1 <= k <= 1024.  The model is not touched.
  Recommendations similar_items(const std::vector<int>& items, int k) { return similar(EALS_BUF_V, items, k); }
  Recommendations similar_users(const std::vector<int>& users, int k) { return similar(EALS_BUF_U, users, k); }
  // Ranking metrics at k on a held-out test matrix (CSR over all users: row_ptr of userCount + 1 offsets, ascending
  // col_idx).  A test item's rank is its position in recommend({u}, k, exclude_seen), or -1; the means are over the
  // users with test items.  per_user: [userCount][6] (hit rate, precision, recall, NDCG, MAP, MRR), ranks: one per
  // test entry, both filled only when asked for.  1 <= k <= 1024.  The model is not touched.
  struct RankingMetrics {
    double hit_rate = 0, precision = 0, recall = 0, ndcg = 0, map = 0, mrr = 0;
    int64_t users = 0;
    std::vector<double> per_user;
    std::vector<int32_t> ranks;
  };
  RankingMetrics ranking_metrics(const std::vector<int64_t>& row_ptr, const std::vector<int32_t>& col_idx, int k,
                                 bool exclude_seen = true, bool want_per_user = false, bool want_ranks = false) {
    if ((int64_t)row_ptr.size() != (int64_t)userCount + 1) throw std::invalid_argument("ranking_metrics: row_ptr must have userCount + 1 offsets");
    RankingMetrics r;
    if (want_per_user) r.per_user.resize((size_t)userCount * 6);
    if (want_ranks) r.ranks.resize((size_t)(row_ptr.back() - row_ptr.front()));
    double means[6];
    const int32_t none = 0;
    check(eals_group_ranking_metrics(g_, EALS_HOST, row_ptr.data(), col_idx.empty() ? &none : col_idx.data(), k, exclude_seen ? 1 : 0,
                                     means, &r.users, want_per_user ? r.per_user.data() : nullptr,
                                     want_ranks && !r.ranks.empty() ? r.ranks.data() : nullptr),
          "eals_group_ranking_metrics");
    r.hit_rate = means[0]; r.precision = means[1]; r.recall = means[2]; r.ndcg = means[3]; r.map = means[4]; r.mrr = means[5];
    return r;
  }
  void update_user_thread(int u) { check(eals_group_update_user_row(g_, u), "eals_group_update_user_row"); }
  void update_item_thread(int i) { check(eals_group_update_item_row(g_, i), "eals_group_update_item_row"); }
  void update_user_SU(double* oldVector, double* uget) { check(eals_group_patch_SU(g_, oldVector, uget), "eals_group_patch_SU"); }
  void update_item_SV(int i, double* oldVector, double* vget) { check(eals_group_patch_SV(g_, i, oldVector, vget), "eals_group_patch_SV"); }

  // metric helpers (MF_fastALS.cpp:597-618)
  double getHitRatio(const std::vector<int>& rankList, int gtItem) {
    for (int item : rankList) if (item == gtItem) return 1;
    return 0;
  }
  double getNDCG(const std::vector<int>& rankList, int gtItem) {
    for (size_t i = 0; i < rankList.size(); i++) if (rankList[i] == gtItem) return std::log(2) / std::log(i + 2);
    return 0;
  }
  double getPrecision(const std::vector<int>& rankList, int gtItem) {
    for (size_t i = 0; i < rankList.size(); i++) if (rankList[i] == gtItem) return 1.0 / (i + 1);
    return 0;
  }

  // Factor checkpoint: U, V, Wi to / from a file (SURVEY.md §8 f4); load rebuilds the S caches on every rank.
  void save(const std::string& path) { check(eals_group_save_factors(g_, path.c_str()), "eals_group_save_factors"); }
  void load(const std::string& path) { check(eals_group_load_factors(g_, path.c_str()), "eals_group_load_factors"); }
  bool replicas_consistent() { int32_t ok = 0; check(eals_group_replicas_consistent(g_, &ok), "eals_group_replicas_consistent"); return ok != 0; }
  int n_gpus() const { return eals_group_size(g_); }

  eals_group* group() { return g_; }
  eals_model* handle(int rank = 0) { eals_model* m = nullptr; check(eals_group_model(g_, rank, &m), "eals_group_model"); return m; }

 private:
  Recommendations similar(int32_t which, const std::vector<int>& ids, int k) {
    Recommendations r;
    std::vector<int32_t> q(ids.begin(), ids.end());
    r.items.resize(q.size() * (size_t)std::max(k, 0));
    r.scores.resize(r.items.size());
    check(eals_group_similar(g_, which, EALS_HOST, (int32_t)q.size(), q.data(), k, r.items.data(), r.scores.data()),
          "eals_group_similar");
    return r;
  }
  struct Flat {
    std::vector<int64_t> row_ptr, col_ptr;
    std::vector<int32_t> col_idx, row_idx;
    std::vector<double> row_val, col_val;
    bool ones = true;   // every stored rating is exactly 1 (what the reference's loader writes)
    const double* rv() const { return ones ? nullptr : row_val.data(); }
    const double* cv() const { return ones ? nullptr : col_val.data(); }
  };
  // rows[u] / cols[i] -> offsets + indices + values, in the stored order (main.cpp:198-205 fills rows
  // ascending by item and cols ascending by user; eals_create verifies that).
  static Flat flatten(const SparseMatT& m) {
    Flat f;
    const int M = m.n_r, N = m.n_c;
    f.row_ptr.assign((size_t)M + 1, 0);
    f.col_ptr.assign((size_t)N + 1, 0);
    for (int u = 0; u < M; u++) f.row_ptr[u + 1] = f.row_ptr[u] + m.rows[u].n;
    for (int i = 0; i < N; i++) f.col_ptr[i + 1] = f.col_ptr[i] + m.cols[i].n;
    f.col_idx.resize((size_t)f.row_ptr[M]); f.row_val.resize((size_t)f.row_ptr[M]);
    f.row_idx.resize((size_t)f.col_ptr[N]); f.col_val.resize((size_t)f.col_ptr[N]);
    for (int u = 0; u < M; u++)
      for (int j = 0; j < m.rows[u].n; j++) {
        f.col_idx[(size_t)f.row_ptr[u] + j] = m.rows[u].spv_in[j];
        f.row_val[(size_t)f.row_ptr[u] + j] = m.rows[u].spv_do[j];
        f.ones &= m.rows[u].spv_do[j] == 1.0;
      }
    for (int i = 0; i < N; i++)
      for (int j = 0; j < m.cols[i].n; j++) {
        f.row_idx[(size_t)f.col_ptr[i] + j] = m.cols[i].spv_in[j];
        f.col_val[(size_t)f.col_ptr[i] + j] = m.cols[i].spv_do[j];
        f.ones &= m.cols[i].spv_do[j] == 1.0;
      }
    return f;
  }
  void upload_matrix() {
    const Flat& f = mat_;
    check(eals_group_set_train(g_, EALS_HOST, f.row_ptr.data(), f.col_idx.data(), f.rv(), f.col_ptr.data(),
                               f.row_idx.data(), f.cv()), "eals_group_set_train");
  }
  // (u, i) with rating 1 into the host copy of the matrix, both orientations, sorted position.  An entry that
  // is already there gets rating (= weight) 1, as trainMatrix.setValue(u, i, 1) / W.setValue(u, i, w_new) do
  // (MF_fastALS.cpp:224-226); false if nothing changed.
  bool insert_entry(int u, int i) {
    Flat& f = mat_;
    auto b = f.col_idx.begin() + f.row_ptr[u], e = f.col_idx.begin() + f.row_ptr[u + 1];
    auto at = std::lower_bound(b, e, (int32_t)i);
    if (at != e && *at == i) {
      const size_t k0 = (size_t)(at - f.col_idx.begin());
      if (f.row_val[k0] == 1.0) return false;
      f.row_val[k0] = 1.0;
      auto b3 = f.row_idx.begin() + f.col_ptr[i], e3 = f.row_idx.begin() + f.col_ptr[i + 1];
      f.col_val[(size_t)(std::lower_bound(b3, e3, (int32_t)u) - f.row_idx.begin())] = 1.0;
      f.ones = true;
      for (double v : f.row_val) f.ones = f.ones && v == 1.0;
      return true;
    }
    const size_t k = (size_t)(at - f.col_idx.begin());
    f.col_idx.insert(f.col_idx.begin() + k, (int32_t)i);
    f.row_val.insert(f.row_val.begin() + k, 1.0);
    for (size_t r = (size_t)u + 1; r < f.row_ptr.size(); r++) f.row_ptr[r]++;
    auto b2 = f.row_idx.begin() + f.col_ptr[i], e2 = f.row_idx.begin() + f.col_ptr[i + 1];
    const size_t k2 = (size_t)(std::lower_bound(b2, e2, (int32_t)u) - f.row_idx.begin());
    f.row_idx.insert(f.row_idx.begin() + k2, (int32_t)u);
    f.col_val.insert(f.col_val.begin() + k2, 1.0);
    for (size_t c = (size_t)i + 1; c < f.col_ptr.size(); c++) f.col_ptr[c]++;
    return true;
  }
  static double seconds_since(std::chrono::steady_clock::time_point t0) {
    return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  }

  eals_group* g_ = nullptr;
  Flat mat_;   // host copy of the train matrix (CSR + CSC), kept for updateModel
};

}  // namespace eals_b200
#endif
