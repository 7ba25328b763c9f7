"""Fold-in (user vectors for histories) and top-k for arbitrary query vectors.

fold_in runs the user CD kernels of a training sweep on a workspace matrix, so a pass from U[u] over u's train row is
update_user_thread(u) bit for bit ("bits": compared as int64 views).  recommend_vectors feeds the recommend engines
with query rows instead of U rows, so U[users] as queries gives recommend(users) bit for bit."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import random_csr
from test_gpu_recommend import _model, assert_same, reference_topk

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_ARG = -1


def bits_equal(a, b):
    a, b = np.ascontiguousarray(a, np.float64), np.ascontiguousarray(b, np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


def csr_of(rows):
    rp = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    ci = np.concatenate([np.asarray(r, np.int32) for r in rows] + [np.zeros(0, np.int32)])
    return rp, ci


def hist(N, rp, ci, val=None):
    """Histories as a SparseMat (only the row orientation is read)."""
    from eals_cpp_b200.model import SparseMat
    return SparseMat(len(rp) - 1, N, rp, ci, None, None, val)


def rows_of(rp, ci, users):
    return [ci[rp[u]:rp[u + 1]] for u in users]


def bucket_matrix(M, N, seed):
    """Rows of every length bucket: empty, 1..32, ..97..128 (warp kernels), 129..512 (one CTA per row) and heavy."""
    rng = np.random.default_rng(seed)
    lengths = [0, 1, 7, 32, 33, 64, 65, 96, 97, 128, 129, 256, 257, 384, 385, 512, 513, 700, 1100]
    rows = []
    for u in range(M):
        n = lengths[u] if u < len(lengths) else int(min(N, rng.geometric(1 / 12)))
        rows.append(np.sort(rng.choice(N, size=n, replace=False)))
    return csr_of(rows)


def _bucket_model(K, monkeypatch, **kw):
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    monkeypatch.setenv("EALS_HEAVY_MIN", "300")          # rows > 300 nonzeros through the slab pipeline
    M, N = 120, 1200
    rp, ci = bucket_matrix(M, N, seed=K)
    fals = MF_fastALS(SparseMat.from_csr(M, N, rp, ci), None, factors=K, showLoss=False, device=0, **kw)
    fals.run_epochs(2)
    return fals, rp, ci


@pytest.mark.parametrize("K", [8, 64, 129])
def test_one_pass_from_U_is_update_user_thread(K, monkeypatch):
    fals, rp, ci = _bucket_model(K, monkeypatch)
    users = np.arange(19)                                 # one row of every listed length, heavy ones included
    U = fals.U
    got = fals.fold_in(hist(fals.itemCount, *csr_of(rows_of(rp, ci, users))), init=U[users], n_iter=1)
    for u in users:
        fals.update_user_thread(int(u))
    assert bits_equal(got, fals.U[users])


@pytest.mark.parametrize("K", [16, 130])
def test_whole_matrix_pass_is_update_user(K, monkeypatch):
    monkeypatch.setenv("EALS_NO_PRED_CACHE", "1")        # the sweep recomputes every prediction, as fold-in does
    fals, rp, ci = _bucket_model(K, monkeypatch)
    got = fals.fold_in(hist(fals.itemCount, rp, ci), init=fals.U, n_iter=1)
    fals.update_user()
    assert bits_equal(got, fals.U)


@pytest.mark.parametrize("K", [8, 64, 129, 256])
def test_fold_in_matches_oracle(K, port):
    M, N, n = 150, 400, 90
    fals, _, _ = _model(M, N, K, seed=K, epochs=2)
    rng = np.random.default_rng(K)
    rp, ci = random_csr(n, N, 15, seed=K + 1, empty_frac=0.05)
    V, SV, Wi = fals.V, fals.SV, fals.Wi
    for val in (None, rng.uniform(0.5, 3.0, len(ci))):
        for init in (None, rng.standard_normal((n, K)) * 0.1):
            for n_iter in (1, 3, 10):
                got = fals.fold_in(hist(N, rp, ci, val), init=init, n_iter=n_iter)
                want = np.zeros((n, K)) if init is None else init.copy()
                for _ in range(n_iter):
                    port.update_user_sweep(rp, ci, val, want, V, np.zeros((K, K)), SV, Wi, fals.reg, patch_S=False)
                assert np.abs(got - want).max() < 1e-10, (val is None, init is None, n_iter)


def test_fold_in_converges_to_the_least_squares_solution():
    M, N, K = 100, 60, 8
    fals, _, _ = _model(M, N, K, seed=2, epochs=3)
    V, SV, Wi, reg = fals.V, fals.SV, fals.Wi, fals.reg
    h = np.array([3, 10, 11, 40, 59], np.int32)
    w = np.array([1.0, 2.0, 1.5, 1.0, 3.0])
    A = SV + reg * np.eye(K)
    b = np.zeros(K)
    for i, wi in zip(h, w):
        A += (wi - Wi[i]) * np.outer(V[i], V[i])
        b += wi * wi * V[i]                               # w_i r_i v_i with r_i = w_i (the rating is the weight)
    want = np.linalg.solve(A, b)
    got = fals.fold_in(hist(N, np.array([0, len(h)], np.int64), h, w), n_iter=400)[0]
    assert np.abs(got - want).max() <= 1e-9 * np.abs(want).max()


def test_no_side_effects_and_training_unchanged(monkeypatch):
    """fold_in and recommend_vectors leave factors, S caches, loss, timers and the prediction-cache state alone: a
    model that calls them between epochs (graph replay included) trains to the same bits as one that does not."""
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    monkeypatch.setenv("EALS_HEAVY_MIN", "64")
    M, N, K = 300, 500, 32
    rp, ci = random_csr(M, N, 20, seed=8, empty_frac=0.02)
    a = MF_fastALS(SparseMat.from_csr(M, N, rp, ci), None, factors=K, showLoss=False, device=0)
    b = MF_fastALS(SparseMat.from_csr(M, N, rp, ci), None, factors=K, showLoss=False, device=0)
    for m in (a, b):
        m.run_epochs(2)
    snap = lambda: (a.timings_detail(), a.timings_total(), a.factor_hash(), a.SU, a.SV)
    before = snap()
    big = [np.arange(0, N, 2)] * 3 + rows_of(rp, ci, range(200))   # heavy histories: the scratch has to grow
    h = hist(N, *csr_of(big))
    Q = a.fold_in(h)
    a.recommend_vectors(Q, 10, exclude=h)
    after = snap()
    assert before[:3] == after[:3] and bits_equal(before[3], after[3]) and bits_equal(before[4], after[4])
    assert a.loss() == b.loss()
    for m in (a, b):
        m.run_epochs(3)
    assert a.factor_hash() == b.factor_hash() and a.loss() == b.loss()


@pytest.mark.parametrize("case", ["plain", "inflated", "ties", "many_blocks", "overflow", "all_equal", "pair_chunks",
                                  "user_chunks"])
def test_recommend_vectors_of_U_equals_recommend(case, monkeypatch):
    M, N, K = 400, 1500, 64
    fals, rp, ci = _model(M, N, K, seed=11)
    U, V = fals.U, fals.V
    if case == "inflated":
        fals.setUV(U * 40, V * 40)
    elif case == "ties":
        V[1::3] = V[0::3][:len(V[1::3])]
        fals.setUV(U, V)
    elif case in ("all_equal", "pair_chunks"):
        fals.setUV(np.full_like(U, 0.125), np.full_like(V, 0.25))
    if case == "many_blocks":
        monkeypatch.setenv("EALS_EVAL_FIRST_CHUNK", "128")
    elif case == "overflow":
        monkeypatch.setenv("EALS_EVAL_PAIR_CAP", "16")
        monkeypatch.setenv("EALS_EVAL_PAIR_HARD_CAP", "64")
    elif case == "pair_chunks":
        monkeypatch.setenv("EALS_EVAL_PAIR_CAP", "16")
        monkeypatch.setenv("EALS_EVAL_PAIR_HARD_CAP", "400000")
    elif case == "user_chunks":
        monkeypatch.setenv("EALS_REC_LIST_BYTES", str(12 * 50 * 150))
    users = np.random.default_rng(4).permutation(M)
    U = fals.U
    train = hist(N, *csr_of(rows_of(rp, ci, users)))
    for k in (5, 50):
        for scalar in ("0", "1"):
            monkeypatch.setenv("EALS_EVAL_SCALAR", scalar)
            want = fals.recommend(users, k)
            st = fals.recommend_stats()
            got = fals.recommend_vectors(U[users], k, exclude=train)
            assert fals.recommend_stats()["engine"] == st["engine"]
            assert_same(got, want)
        monkeypatch.delenv("EALS_EVAL_SCALAR")


@pytest.mark.parametrize("n", [40, 300])                 # exact engine, tcgen05 engine
def test_arbitrary_queries_match_reference(n):
    import torch
    M, N, K = 200, 900, 48
    fals, rp, ci = _model(M, N, K, seed=6)
    rng = np.random.default_rng(n)
    Q = rng.standard_normal((n, K)) * 0.3
    Q[::7] = 0.0                                          # zero rows: every score +0.0, lowest item ids first
    Q[1::7] *= -1.0
    Q[2::7] *= 50.0
    Q[3::7] = fals.U[rng.integers(0, M, len(Q[3::7]))]
    erp, eci = random_csr(n, N, 30, seed=n, empty_frac=0.1)
    V = fals.V
    for k in (1, 10, 100):
        assert_same(fals.recommend_vectors(Q, k), reference_topk(Q, V, erp, eci, np.arange(n), k, exclude=False))
        assert_same(fals.recommend_vectors(Q, k, exclude=hist(N, erp, eci)),
                    reference_topk(Q, V, erp, eci, np.arange(n), k, exclude=True))
    zero = fals.recommend_vectors(np.zeros((n, K)), 10, exclude=hist(N, erp, eci))
    for s in range(n):
        ok = np.setdiff1d(np.arange(N), eci[erp[s]:erp[s + 1]])[:10]
        assert np.array_equal(zero[0][s], ok) and bits_equal(zero[1][s], np.zeros(10))
    dev = "cuda:0"
    ti, ts = fals.recommend_vectors(torch.from_numpy(Q).to(dev), 10,
                                    exclude=hist(N, torch.from_numpy(erp).to(dev), torch.from_numpy(eci).to(dev)))
    assert_same((ti, ts), reference_topk(Q, V, erp, eci, np.arange(n), 10, exclude=True))


@pytest.mark.parametrize("n", [3, 200])
def test_history_recommendations(n):
    """fold_in + recommend_vectors(exclude=history): an empty history with zero init folds to 0, whose top-k are the
    lowest item ids; no list contains an item of its history; device tensors give the same answer."""
    import torch
    M, N, K = 200, 700, 32
    fals, _, _ = _model(M, N, K, seed=3)
    rp, ci = random_csr(n, N, 25, seed=n, empty_frac=0.0)
    rp = np.concatenate([[0], rp]).astype(np.int64)      # history 0 is empty
    h = hist(N, rp, ci)
    Q = fals.fold_in(h)
    assert bits_equal(Q[0], np.zeros(K))
    items, scores = fals.recommend_vectors(Q, 20, exclude=h)
    assert np.array_equal(items[0], np.arange(20)) and bits_equal(scores[0], np.zeros(20))
    for s in range(n + 1):
        assert not set(items[s].tolist()) & set(ci[rp[s]:rp[s + 1]].tolist())
    dev = "cuda:0"
    hd = hist(N, torch.from_numpy(rp).to(dev), torch.from_numpy(ci).to(dev))
    Qd = fals.fold_in(hd, init=torch.zeros((n + 1, K), dtype=torch.float64, device=dev))
    assert bits_equal(Qd, Q)
    assert_same(fals.recommend_vectors(torch.from_numpy(Qd).to(dev), 20, exclude=hd), (items, scores))


def test_argument_errors():
    from eals_cpp_b200 import _lib
    from eals_cpp_b200._lib import EalsError
    M, N, K = 150, 300, 16
    fals, _, _ = _model(M, N, K, epochs=1)
    Q = np.zeros((2, K))
    good = hist(N, np.array([0, 1, 2], np.int64), np.array([4, 5], np.int32))
    bad_rows = [hist(N, np.array([0, 2, 3], np.int64), np.array([5, 4, 1], np.int32)),     # unsorted
                hist(N, np.array([0, 2, 2], np.int64), np.array([3, 3], np.int32)),        # duplicate
                hist(N, np.array([0, 1, 2], np.int64), np.array([0, N], np.int32)),        # out of range
                hist(N, np.array([0, 1, 2], np.int64), np.array([0, -1], np.int32))]
    calls = [lambda: fals.recommend_vectors(Q, 0), lambda: fals.recommend_vectors(Q, 1025),
             lambda: fals.fold_in(good, n_iter=0)]
    for v in (np.nan, np.inf, -np.inf):
        Qb = Q.copy()
        Qb[1, 3] = v
        calls.append(lambda Qb=Qb: fals.recommend_vectors(Qb, 5))
    for b in bad_rows:
        calls += [lambda b=b: fals.fold_in(b), lambda b=b: fals.recommend_vectors(Q, 5, exclude=b)]
    for call in calls:
        with pytest.raises(EalsError) as e:
            call()
        assert e.value.code == ERR_ARG and fals.lib.eals_last_error()
    items = np.zeros((2, 5), np.int32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = fals.lib.eals_recommend_vectors(fals.h, _lib.EALS_HOST, 2, p(Q), p(good.row_ptr), None, 5, p(items), None)
    assert rc == ERR_ARG and b"both" in fals.lib.eals_last_error()
    # the model still answers after every rejected call
    assert_same(fals.recommend_vectors(fals.U[:2], 5, exclude=hist(N, *csr_of([[], []]))), fals.recommend([0, 1], 5, exclude_seen=False))


@pytest.mark.parametrize("world", [2, 4, 8])
def test_group_equals_single_model(world):
    """The group's calls equal rank 0's own eals_fold_in / eals_recommend_vectors over all the queries."""
    from eals_cpp_b200.model import GroupMF_fastALS, SparseMat, _fold_in_call, _recommend_vectors_call
    M, N, K = 500, 900, 32
    fals, rp, ci = _model(M, N, K, seed=9)
    g = GroupMF_fastALS(SparseMat.from_csr(M, N, rp, ci), None, factors=K, showLoss=False, devices=[0] * world)
    g.setUV(fals.U, fals.V)
    hrp, hci = random_csr(301, N, 20, seed=world, empty_frac=0.05)
    val = np.random.default_rng(world).uniform(0.5, 2.0, len(hci))
    h = hist(N, hrp, hci, val)
    init = np.random.default_rng(1).standard_normal((301, K)) * 0.1
    r0 = g.rank_model(0)
    for ini in (None, init):
        Qs = _fold_in_call(g.lib.eals_fold_in, r0, K, "cuda:0", h, ini, 3)
        assert bits_equal(g.fold_in(h, init=ini, n_iter=3), Qs)
    for k in (10, 100):
        for ex in (h, None):
            want = _recommend_vectors_call(g.lib.eals_recommend_vectors, r0, K, "cuda:0", Qs, k, ex)
            assert_same(g.recommend_vectors(Qs, k, exclude=ex), want)
    g.close()


def _ngpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


def test_one_process_per_gpu_fold_in():
    """torch.distributed, one process per GPU: every rank gets the whole result.  With fewer than two GPUs NCCL
    cannot place two ranks on one device, so the same check runs through virtual ranks."""
    if _ngpus() < 2:
        test_group_equals_single_model(2)
        return
    world = min(_ngpus(), 4)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(29750 + world),
           os.path.join(ROOT, "tests", "dist_fold_in_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "dist fold_in ok" in res.stdout
