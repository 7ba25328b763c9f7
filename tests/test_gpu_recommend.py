"""Top-k retrieval (recommend): every result equals a numpy reference item for item and score bit for bit.

The reference builds the scores with acc = acc + U[:, k] * V[:, k] over k: numpy rounds the product and the
sum separately, the operation order of predict() (eval.cuh seq_dot), so its scores are bit-identical.  It then
drops the user's train items and sorts stably by (-score, item)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import random_csr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ERR_ARG = -1


def reference_topk(U, V, row_ptr, col_idx, users, k, exclude=True):
    users = np.asarray(users, np.int64)
    N, K = V.shape
    S = np.zeros((len(users), N))
    Uu = U[users]
    for q in range(K):
        S = S + Uu[:, q:q + 1] * V[:, q]
    items = np.full((len(users), k), -1, np.int32)
    scores = np.full((len(users), k), -np.inf)
    for t, u in enumerate(users):
        ok = np.ones(N, bool)
        if exclude:
            ok[col_idx[row_ptr[u]:row_ptr[u + 1]]] = False
        cand = np.nonzero(ok)[0]
        order = cand[np.lexsort((cand, -S[t, cand]))][:k]
        items[t, :len(order)] = order
        scores[t, :len(order)] = S[t, order]
    return items, scores


def assert_same(got, want):
    gi, gs = got
    wi, ws = want
    assert np.array_equal(gi, wi), np.argwhere(gi != wi)[:5]
    assert np.array_equal(gs.view(np.int64), ws.view(np.int64)), np.argwhere(gs.view(np.int64) != ws.view(np.int64))[:5]


def _model(M, N, K, seed=7, epochs=2, density=12):
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    rp, ci = random_csr(M, N, density, seed=seed, empty_frac=0.02)
    fals = MF_fastALS(SparseMat.from_csr(M, N, rp, ci), None, factors=K, showLoss=False, device=0)
    fals.run_epochs(epochs)
    return fals, rp, ci


def _check(fals, rp, ci, users, k, engine=None, exclude=True):
    got = fals.recommend(users, k, exclude_seen=exclude)
    assert_same(got, reference_topk(fals.U, fals.V, rp, ci, users, k, exclude))
    if engine:
        assert fals.recommend_stats()["engine"] == engine
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("K", [8, 64, 128, 130, 200, 256])
def test_recommend_matches_reference(K):
    M, N = 300, 1000                                   # catalogue not a multiple of 128
    fals, rp, ci = _model(M, N, K)
    for k in (1, 10, 100):
        _check(fals, rp, ci, np.arange(M), k, "tcgen05")
        _check(fals, rp, ci, np.arange(0, M, 7)[:40], k, "fp64")     # short list: exact engine


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["inflated", "ties", "many_blocks", "overflow", "all_equal", "pair_chunks", "user_chunks"])
def test_tcgen05_engine_equals_exact_engine(case, monkeypatch):
    M, N, K = 400, 1500, 64
    fals, rp, ci = _model(M, N, K, seed=11)
    U, V = fals.U, fals.V
    if case == "inflated":
        fals.setUV(U * 40, V * 40)
    elif case == "ties":
        V[1::3] = V[0::3][:len(V[1::3])]               # duplicated rows: exact score ties, ordered by item id
        fals.setUV(U, V)
    elif case == "all_equal":
        fals.setUV(np.full_like(U, 0.125), np.full_like(V, 0.25))
    elif case == "many_blocks":
        monkeypatch.setenv("EALS_EVAL_FIRST_CHUNK", "128")
    elif case == "overflow":
        monkeypatch.setenv("EALS_EVAL_PAIR_CAP", "16")
        monkeypatch.setenv("EALS_EVAL_PAIR_HARD_CAP", "64")
    elif case == "pair_chunks":
        # every item is a candidate: 400 users x 1372 items do not fit the hard cap, a chunk of 256 users does, so the
        # block is filtered and merged chunk by chunk (TMA map offset by the chunk's first position)
        fals.setUV(np.full_like(U, 0.125), np.full_like(V, 0.25))
        monkeypatch.setenv("EALS_EVAL_PAIR_CAP", "16")
        monkeypatch.setenv("EALS_EVAL_PAIR_HARD_CAP", "400000")
    elif case == "user_chunks":
        monkeypatch.setenv("EALS_REC_LIST_BYTES", str(12 * 50 * 150))   # k = 50: lists for 150 users at a time
    users = np.arange(M)
    for k in (5, 50):
        tc = _check(fals, rp, ci, users, k)
        st = fals.recommend_stats()
        assert st["engine"] == ("fp64" if case == "overflow" else "tcgen05")
        if case == "pair_chunks":
            assert "first_block" not in st           # only an unsplit first block is timed
        monkeypatch.setenv("EALS_EVAL_SCALAR", "1")
        ex = fals.recommend(users, k)
        assert fals.recommend_stats()["engine"] == "fp64"
        monkeypatch.delenv("EALS_EVAL_SCALAR")
        assert_same(tc, ex)


@pytest.mark.gpu
def test_early_out_leaves_users_behind(monkeypatch):
    """A few high-norm items that every user likes and a long tail of small ones: once the high-norm items are
    scored, |u| * max |v| over the tail is below every user's k-th score, and the users leave the working set
    long before the end of the catalogue."""
    M, N, K = 400, 3000, 32
    fals, rp, ci = _model(M, N, K, seed=4, epochs=1)
    rng = np.random.default_rng(5)
    U = rng.uniform(0.5, 1.0, (M, K))
    V = rng.uniform(-0.01, 0.01, (N, K))
    hot = rng.choice(N, 256, replace=False)
    V[hot] = rng.uniform(1.0, 2.0, (256, K))
    fals.setUV(U, V)
    monkeypatch.setenv("EALS_EVAL_FIRST_CHUNK", "128")      # block 1 = the next 128 items in norm order
    _check(fals, rp, ci, np.arange(M), 10, "tcgen05")
    assert fals.recommend_stats()["users_left_after_first_block"] < M


@pytest.mark.gpu
def test_exclusion_heavy_users_padding_and_updates():
    from eals_cpp_b200.model import SparseMat
    M, N, K = 260, 700, 32
    fals, rp, ci = _model(M, N, K, seed=5)
    V = fals.V
    by_norm = np.argsort(-(V * V).sum(1), kind="stable")
    rows = [list(ci[rp[u]:rp[u + 1]]) for u in range(M)]
    for u in range(10):                                # heavy users: seen most of the high-norm items
        rows[u] = sorted(set(rows[u]) | set(by_norm[:500].tolist()))
    rows[10] = sorted(set(range(N)) - {3, 400})        # seen >= N - k: padded with -1 / -inf
    rp2 = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    ci2 = np.concatenate([np.array(r, np.int32) for r in rows])
    fals.setTrain(SparseMat.from_csr(M, N, rp2, ci2))
    users = np.arange(M)
    items, scores = _check(fals, rp2, ci2, users, 20, "tcgen05")
    assert set(items[10, :2]) == {3, 400} and (items[10, 2:] == -1).all() and np.isneginf(scores[10, 2:]).all()
    _check(fals, rp2, ci2, users, 20, exclude=False)   # plain top-k
    # updateModel(u, i): the new interaction is excluded at once
    u = 20
    i = int(items[u, 0])
    fals.updateModel(u, i)
    rows[u] = sorted(set(rows[u]) | {i})
    rp3 = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    ci3 = np.concatenate([np.array(r, np.int32) for r in rows])
    it3, _ = _check(fals, rp3, ci3, users, 20)
    assert i not in it3[u]


@pytest.mark.gpu
def test_scores_equal_predict_and_device_tensors():
    import torch
    M, N, K = 200, 600, 48
    fals, rp, ci = _model(M, N, K, seed=3)
    items, scores = fals.recommend(np.arange(M), 10)
    rng = np.random.default_rng(0)
    for u, j in zip(rng.integers(0, M, 20), rng.integers(0, 10, 20)):
        assert fals.predict(int(u), int(items[u, j])) == scores[u, j]
    users = torch.arange(M - 1, -1, -1, dtype=torch.int32, device="cuda:0")
    di, ds = fals.recommend(users, 10)
    assert np.array_equal(di, items[::-1]) and np.array_equal(ds, scores[::-1])


@pytest.mark.gpu
def test_argument_errors():
    from eals_cpp_b200._lib import EalsError
    from eals_cpp_b200.model import GroupMF_fastALS, SparseMat
    import ctypes as C
    M, N, K = 150, 300, 16
    fals, rp, ci = _model(M, N, K, epochs=1)
    for users, k in (([0, M], 5), ([-1], 5), ([0], 0), ([0], 1025)):
        with pytest.raises(EalsError) as e:
            fals.recommend(users, k)
        assert e.value.code == ERR_ARG and fals.lib.eals_last_error()
    g = GroupMF_fastALS(SparseMat.from_csr(M, N, rp, ci), None, factors=K, showLoss=False, devices=[0, 0])
    h1 = g.rank_model(1)
    u0 = np.array([0], np.int32)                       # owned by rank 0
    out = np.zeros((1, 5), np.int32)
    rc = g.lib.eals_recommend(h1, 0, 1, u0.ctypes.data_as(C.c_void_p), 5, 1, out.ctypes.data_as(C.c_void_p), None)
    assert rc == ERR_ARG and b"outside" in g.lib.eals_last_error()
    g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4, 8])
def test_group_recommend_equals_single_model(world):
    from eals_cpp_b200.model import GroupMF_fastALS, SparseMat
    M, N, K = 500, 900, 32
    fals, rp, ci = _model(M, N, K, seed=9)
    g = GroupMF_fastALS(SparseMat.from_csr(M, N, rp, ci), None, factors=K, showLoss=False, devices=[0] * world)
    g.setUV(fals.U, fals.V)
    users = np.random.default_rng(1).permutation(M)
    for k in (10, 100):
        assert_same(g.recommend(users, k), fals.recommend(users, k))
    g.close()


def _ngpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.gpu
def test_one_process_per_gpu_recommend():
    """torch.distributed, one process per GPU: every rank gets the full result in input order.  With fewer than
    two GPUs NCCL cannot place two ranks on one device, so the same check runs through virtual ranks."""
    if _ngpus() < 2:
        test_group_recommend_equals_single_model(2)
        return
    world = min(_ngpus(), 4)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(29700 + world),
           os.path.join(ROOT, "tests", "dist_recommend_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "dist recommend ok" in res.stdout


@pytest.mark.gpu
def test_cpp_driver_recommend_matches_python(tmp_path):
    """eals_main --recommend (include/MF_fastALS.h over eals_group) writes what MF_fastALS.recommend returns on the
    same split and factors."""
    from eals_cpp_b200 import build
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    from test_gpu_driver import _ratings
    exe = build.build_host_example()
    data = tmp_path / "tiny.rating"
    split = _ratings(str(data))
    M = len(split)
    N = 1 + max(max(t + [g]) for t, g in split)
    ckpt, out = tmp_path / "f.eals", tmp_path / "rec.txt"
    res = subprocess.run([exe, "--data", str(data), "--factors", "8", "--iters", "2", "--save", str(ckpt),
                          "--recommend", "5", "--recommend-out", str(out)], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    rp = np.concatenate([[0], np.cumsum([len(t) for t, _ in split])]).astype(np.int64)
    ci = np.concatenate([np.array(t, np.int32) for t, _ in split])
    fals = MF_fastALS(SparseMat.from_csr(M, N, rp, ci), None, factors=8, showLoss=False, device=0)
    fals.load(str(ckpt))
    items, scores = fals.recommend(np.arange(M), 5)
    want = [(u, j) for u in range(M) for j in range(5) if items[u, j] >= 0]
    got = out.read_text().split("\n")[:-1]
    assert len(got) == len(want)
    for line, (u, j) in zip(got, want):
        a, b, c = line.split()
        assert (int(a), int(b)) == (u, items[u, j]) and float(c) == scores[u, j]
