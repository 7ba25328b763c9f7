"""Ranking metrics on a held-out test matrix: every rank equals g's position in a numpy top-k (the construction of
test_gpu_recommend.py: sequential-k scores, train items dropped, stable sort by (-score, item)), and the per-user
metrics equal a plain Python evaluation of the definitions in include/eals_b200.h."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import random_csr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_ARG = -1
NAMES = ("hit_rate", "precision", "recall", "ndcg", "map", "mrr")


def reference_scores(U, V):
    S = np.zeros((U.shape[0], V.shape[0]))
    for q in range(U.shape[1]):
        S = S + U[:, q:q + 1] * V[:, q]
    return S


def reference_ranks(S, rp, ci, tp, ti, k, exclude=True):
    M, N = S.shape
    ranks = np.full(int(tp[-1] - tp[0]), -1, np.int32)
    for u in range(M):
        a, b = int(tp[u] - tp[0]), int(tp[u + 1] - tp[0])
        if a == b:
            continue
        ok = np.ones(N, bool)
        if exclude:
            ok[ci[rp[u]:rp[u + 1]]] = False
        cand = np.nonzero(ok)[0]
        order = cand[np.lexsort((cand, -S[u, cand]))][:k]
        pos = {int(i): p for p, i in enumerate(order)}
        ranks[a:b] = [pos.get(int(g), -1) for g in ti[a:b]]
    return ranks


def reference_metrics(tp, ranks, k):
    M = len(tp) - 1
    gain = lambda r: math.log(2) / math.log(r + 2)
    per = np.zeros((M, 6))
    for u in range(M):
        a, b = int(tp[u] - tp[0]), int(tp[u + 1] - tp[0])
        n = b - a
        if n == 0:
            continue
        H = sorted(int(r) for r in ranks[a:b] if r >= 0)
        h, cap = len(H), min(k, n)
        dcg = idcg = ap = 0.0
        for r in H:
            dcg += gain(r)
        for j in range(cap):
            idcg += gain(j)
        for c, r in enumerate(H, 1):
            ap += c / (r + 1)
        per[u] = [1.0 if h else 0.0, h / k, h / n, dcg / idcg, ap / cap, 1.0 / (H[0] + 1) if h else 0.0]
    users = int((np.diff(tp) > 0).sum())
    return per, (per.sum(0) / users if users else per.sum(0)), users


def _model(M, N, K, seed=7, epochs=2, density=12):
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    rp, ci = random_csr(M, N, density, seed=seed, empty_frac=0.02)
    fals = MF_fastALS(SparseMat.from_csr(M, N, rp, ci), None, factors=K, showLoss=False, device=0)
    fals.run_epochs(epochs)
    return fals, rp, ci


def _test_matrix(M, N, seed, density=6, long_rows=()):
    """A seeded test CSR (rows may overlap the train rows; some are empty), with the listed rows made long."""
    from eals_cpp_b200.model import SparseMat
    tp, ti = random_csr(M, N, density, seed=seed, empty_frac=0.1)
    rows = [list(ti[tp[u]:tp[u + 1]]) for u in range(M)]
    rng = np.random.default_rng(seed)
    for u in long_rows:
        rows[u] = sorted(rng.choice(N, 150, replace=False).tolist())
    tp = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    ti = np.concatenate([np.array(r, np.int32) for r in rows])
    return SparseMat(M, N, tp, ti, None, None), tp, ti


def _check(fals, rp, ci, test, tp, ti, k, exclude=True, engine=None, S=None):
    got = fals.ranking_metrics(test, k, exclude_seen=exclude, per_user=True, ranks=True)
    if S is None:
        S = reference_scores(fals.U, fals.V)
    want = reference_ranks(S, rp, ci, tp, ti, k, exclude)
    assert np.array_equal(got["ranks"], want), (k, exclude, np.argwhere(got["ranks"] != want)[:5])
    per, means, users = reference_metrics(tp, want, k)
    np.testing.assert_allclose(got["per_user"], per, rtol=1e-13, atol=0)
    np.testing.assert_allclose([got[n] for n in NAMES], means, rtol=1e-12, atol=0)
    assert got["users"] == users
    if engine:
        assert fals.eval_stats()["engine"] == engine
    return got


def _same(a, b):
    assert np.array_equal(a["ranks"], b["ranks"])
    assert np.array_equal(a["per_user"].view(np.int64), b["per_user"].view(np.int64))
    assert [a[n] for n in NAMES] == [b[n] for n in NAMES] and a["users"] == b["users"]


@pytest.mark.gpu
@pytest.mark.parametrize("K", [8, 64, 128, 130, 200, 256])
def test_ranking_metrics_match_reference(K, monkeypatch):
    M, N = 300, 1000
    fals, rp, ci = _model(M, N, K)
    test, tp, ti = _test_matrix(M, N, seed=K, long_rows=(3, 4))
    S = reference_scores(fals.U, fals.V)
    for k in (1, 10, 100, 1024):
        for exclude in (True, False):
            tc = _check(fals, rp, ci, test, tp, ti, k, exclude, "tcgen05", S)
            monkeypatch.setenv("EALS_EVAL_SCALAR", "1")
            ex = _check(fals, rp, ci, test, tp, ti, k, exclude, "fp64", S)
            monkeypatch.delenv("EALS_EVAL_SCALAR")
            _same(tc, ex)


@pytest.mark.gpu
def test_short_list_runs_on_the_exact_engine():
    """Fewer than 128 test entries: the exact engine answers."""
    from eals_cpp_b200.model import SparseMat
    M, N, K = 200, 700, 32
    fals, rp, ci = _model(M, N, K, seed=2)
    _, tp, ti = _test_matrix(M, N, seed=5, density=3)
    keep = np.zeros(M, bool)
    keep[::9] = True                                   # a few users keep their test rows
    rows = [list(ti[tp[u]:tp[u + 1]]) if keep[u] else [] for u in range(M)]
    tp2 = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    ti2 = np.concatenate([np.array(r, np.int32) for r in rows])
    assert 0 < len(ti2) < 128
    _check(fals, rp, ci, SparseMat(M, N, tp2, ti2, None, None), tp2, ti2, 10, True, "fp64")


@pytest.mark.gpu
def test_ranks_equal_positions_in_recommend():
    M, N, K = 400, 1500, 64
    fals, rp, ci = _model(M, N, K, seed=3)
    test, tp, ti = _test_matrix(M, N, seed=4)
    for k in (10, 100):
        for exclude in (True, False):
            got = fals.ranking_metrics(test, k, exclude_seen=exclude, ranks=True)["ranks"]
            items = fals.recommend(np.arange(M), k, exclude_seen=exclude)[0]
            want = np.full(len(ti), -1, np.int32)
            for u in range(M):
                pos = {int(i): p for p, i in enumerate(items[u]) if i >= 0}
                want[tp[u]:tp[u + 1]] = [pos.get(int(g), -1) for g in ti[tp[u]:tp[u + 1]]]
            assert np.array_equal(got, want), (k, exclude)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["inflated", "ties", "all_equal", "many_blocks", "pair_cap", "hard_cap", "entry_chunks",
                                  "heavy_train"])
def test_edge_cases(case, monkeypatch):
    from eals_cpp_b200.model import SparseMat
    M, N, K = 400, 1500, 64
    fals, rp, ci = _model(M, N, K, seed=11)
    test, tp, ti = _test_matrix(M, N, seed=12, long_rows=(0, 1, 2))
    U, V = fals.U, fals.V
    engine = "tcgen05"
    if case == "inflated":
        fals.setUV(U * 40, V * 40)
    elif case == "ties":
        V[1::3] = V[0::3][:len(V[1::3])]               # duplicated rows: exact score ties, ordered by item id
        fals.setUV(U, V)
    elif case == "all_equal":
        fals.setUV(np.full_like(U, 0.125), np.full_like(V, 0.25))
        monkeypatch.setenv("EALS_EVAL_PAIR_HARD_CAP", "100000")   # every item is a candidate: the exact engine answers
        engine = "fp64"
    elif case == "many_blocks":
        monkeypatch.setenv("EALS_EVAL_FIRST_CHUNK", "128")
    elif case == "pair_cap":
        monkeypatch.setenv("EALS_EVAL_PAIR_CAP", "16")   # the second attempt has the exact size
    elif case == "hard_cap":
        monkeypatch.setenv("EALS_EVAL_PAIR_HARD_CAP", "1")       # any two candidate pairs overflow it
        engine = "fp64"
    elif case == "entry_chunks":
        monkeypatch.setenv("EALS_REC_LIST_BYTES", "200000")      # a few hundred entries per chunk
        engine = None                                  # a short last chunk may run on the exact engine
    elif case == "heavy_train":
        by_norm = np.argsort(-(V * V).sum(1), kind="stable")
        rows = [list(ci[rp[u]:rp[u + 1]]) for u in range(M)]
        for u in range(0, 40, 2):                      # heavy rows holding most of the high-norm items: large c_R
            rows[u] = sorted(set(rows[u]) | set(by_norm[:900].tolist()))
        rows[5] = []                                   # an empty train row with test items
        rp = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
        ci = np.concatenate([np.array(r, np.int32) for r in rows])
        fals.setTrain(SparseMat.from_csr(M, N, rp, ci))
        assert np.diff(rp)[0] > 512 and np.diff(tp)[5] > 0
    S = reference_scores(fals.U, fals.V)
    for k in (5, 50):
        for exclude in (True, False):
            tc = _check(fals, rp, ci, test, tp, ti, k, exclude, engine, S)
            monkeypatch.setenv("EALS_EVAL_SCALAR", "1")
            ex = _check(fals, rp, ci, test, tp, ti, k, exclude, "fp64", S)
            monkeypatch.delenv("EALS_EVAL_SCALAR")
            _same(tc, ex)
    overlap = sum(len(np.intersect1d(ti[tp[u]:tp[u + 1]], ci[rp[u]:rp[u + 1]])) for u in range(M))
    assert overlap > 0                                 # some test items are also train items: rank -1 with exclusion


@pytest.mark.gpu
def test_exclusion_follows_set_train_and_update_model():
    from eals_cpp_b200.model import SparseMat
    M, N, K = 300, 800, 32
    fals, rp, ci = _model(M, N, K, seed=5)
    test, tp, ti = _test_matrix(M, N, seed=6)
    rp2, ci2 = random_csr(M, N, 20, seed=8)
    fals.setTrain(SparseMat.from_csr(M, N, rp2, ci2))
    _check(fals, rp2, ci2, test, tp, ti, 20)
    u = int(np.nonzero(np.diff(tp) > 0)[0][0])
    got = fals.ranking_metrics(test, 20, ranks=True)["ranks"]
    e = tp[u] + int(np.argmax(got[tp[u]:tp[u + 1]]))   # a test item of u, ranked if any is
    g = int(ti[e])
    fals.updateModel(u, g)                             # g joins u's train row: from now on it is excluded
    rows = [list(ci2[rp2[v]:rp2[v + 1]]) for v in range(M)]
    rows[u] = sorted(set(rows[u]) | {g})
    rp3 = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    ci3 = np.concatenate([np.array(r, np.int32) for r in rows])
    got = _check(fals, rp3, ci3, test, tp, ti, 20)
    assert got["ranks"][e] == -1


@pytest.mark.gpu
def test_device_tensor_inputs():
    import torch
    from eals_cpp_b200.model import SparseMat
    M, N, K = 300, 900, 48
    fals, rp, ci = _model(M, N, K, seed=3)
    test, tp, ti = _test_matrix(M, N, seed=9)
    host = fals.ranking_metrics(test, 10, per_user=True, ranks=True)
    dt = SparseMat(M, N, torch.from_numpy(tp).cuda(), torch.from_numpy(ti).cuda(), None, None)
    _same(fals.ranking_metrics(dt, 10, per_user=True, ranks=True), host)


@pytest.mark.gpu
def test_argument_errors():
    from eals_cpp_b200._lib import EalsError
    from eals_cpp_b200.model import SparseMat
    M, N, K = 150, 300, 16
    fals, rp, ci = _model(M, N, K, epochs=1)
    test, tp, ti = _test_matrix(M, N, seed=2)
    bad_idx = ti.copy()
    bad_idx[3] = N
    u = int(np.nonzero(np.diff(tp) >= 2)[0][0])
    unsorted = ti.copy()
    unsorted[tp[u]], unsorted[tp[u] + 1] = ti[tp[u] + 1], ti[tp[u]]
    cases = [(test, 0), (test, 1025), (SparseMat(M, N, tp, bad_idx, None, None), 10),
             (SparseMat(M, N, tp, unsorted, None, None), 10), (SparseMat(M - 1, N, tp[:-1], ti, None, None), 10)]
    for t, k in cases:
        with pytest.raises(EalsError) as e:
            fals.ranking_metrics(t, k)
        assert e.value.code == ERR_ARG


@pytest.mark.gpu
@pytest.mark.parametrize("K", [16, 64])
def test_one_item_per_user_equals_evaluate(K):
    """One test item per user, no exclusion, factors without ties: hit, NDCG and MRR are evaluate's exact hr, ndcg and
    reciprocal rank bit for bit."""
    from eals_cpp_b200.model import SparseMat
    M, N = 400, 1200
    fals, rp, ci = _model(M, N, K, seed=13)
    gt = np.random.default_rng(2).integers(0, N, M).astype(np.int32)
    test = SparseMat(M, N, np.arange(M + 1, dtype=np.int64), gt, None, None)
    for k in (1, 10, 100):
        got = fals.ranking_metrics(test, k, exclude_seen=False, per_user=True)["per_user"]
        _, hr, ndcg, prec, _ = fals.evaluate(gt, topK=k, exact=True, per_user=True)
        for col, want in ((0, hr), (3, ndcg), (5, prec)):
            assert np.array_equal(got[:, col].view(np.int64), want.view(np.int64)), (k, col)


def _state(fals):
    return (fals.factor_hash(), fals.SU.tobytes(), fals.SV.tobytes(), np.float64(fals.loss()).tobytes())


@pytest.mark.gpu
@pytest.mark.parametrize("K", [64, 128, 200])
def test_model_untouched(K):
    M, N = 400, 1300
    fals, rp, ci = _model(M, N, K, seed=17)
    twin, _, _ = _model(M, N, K, seed=17)
    test, tp, ti = _test_matrix(M, N, seed=18)
    users = np.arange(M)
    gt = np.random.default_rng(4).integers(0, N, M).astype(np.int32)

    def retrieval():
        n0 = fals.kernel_launches()
        ev = fals.evaluate(gt, topK=10, per_user=True)
        n1 = fals.kernel_launches()
        rec = fals.recommend(users, 10)
        n2 = fals.kernel_launches()
        return ev, rec, (n1 - n0, n2 - n1)

    before, ret_before = _state(fals), retrieval()
    assert before == _state(twin)
    fals.ranking_metrics(test, 10, per_user=True, ranks=True)
    assert _state(fals) == before
    ret_after = retrieval()
    assert ret_after[2] == ret_before[2]
    for a, b in zip(ret_after[0] + ret_after[1], ret_before[0] + ret_before[1]):
        assert np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))
    fals.run_epochs(1)
    twin.run_epochs(1)
    assert _state(fals) == _state(twin)
    assert np.array_equal(fals.U.view(np.int64), twin.U.view(np.int64)) and np.array_equal(fals.V.view(np.int64), twin.V.view(np.int64))


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4, 8])
def test_group_equals_single_model(world):
    from eals_cpp_b200.model import GroupMF_fastALS, SparseMat
    M, N, K = 500, 900, 32
    fals, rp, ci = _model(M, N, K, seed=9)
    test, tp, ti = _test_matrix(M, N, seed=10, long_rows=(7,))
    g = GroupMF_fastALS(SparseMat.from_csr(M, N, rp, ci), None, factors=K, showLoss=False, devices=[0] * world)
    g.setUV(fals.U, fals.V)
    for k in (10, 100):
        for exclude in (True, False):
            a = g.ranking_metrics(test, k, exclude_seen=exclude, per_user=True, ranks=True)
            b = fals.ranking_metrics(test, k, exclude_seen=exclude, per_user=True, ranks=True)
            assert np.array_equal(a["ranks"], b["ranks"])
            assert np.array_equal(a["per_user"].view(np.int64), b["per_user"].view(np.int64))
            np.testing.assert_allclose([a[n] for n in NAMES], [b[n] for n in NAMES], rtol=1e-12, atol=0)
            assert a["users"] == b["users"]
    g.close()


def _ngpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.gpu
def test_one_process_per_gpu_ranking_metrics():
    """torch.distributed, one process per GPU: every rank gets the whole result.  With fewer than two GPUs NCCL
    cannot place two ranks on one device, so the same check runs through virtual ranks."""
    if _ngpus() < 2:
        test_group_equals_single_model(2)
        return
    world = min(_ngpus(), 4)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(29760 + world),
           os.path.join(ROOT, "tests", "dist_ranking_metrics_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "dist ranking metrics ok" in res.stdout
