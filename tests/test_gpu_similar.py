"""Similar items and similar users: every result equals a numpy reference item for item and score bit for bit.

The reference normalises each row with a sequential sum of squares (acc = acc + y_f * y_f, numpy rounding the product
and the sum separately, the order of eval.cuh seq_dot), np.sqrt and an IEEE division per factor (0 for a zero row),
scores with reference_topk's acc = acc + A[:, f] * B[:, f] loop, drops the query's own row and sorts by (-score, id).
"bits": scores compared as int64 views."""
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


def normalise(Y):
    acc = np.zeros(len(Y))
    for f in range(Y.shape[1]):
        acc = acc + Y[:, f] * Y[:, f]
    norm = np.sqrt(acc)
    out = np.zeros_like(Y)
    nz = norm != 0.0
    out[nz] = Y[nz] / norm[nz, None]
    return out


def reference_similar(Y, ids, k):
    """Top-k of the normalised rows for the normalised rows ids, each query's own row excluded."""
    Yh = normalise(Y)
    ids = np.asarray(ids, np.int32)
    n = len(ids)
    return reference_topk(Yh[ids], Yh, np.arange(n + 1, dtype=np.int64), ids, np.arange(n), k, exclude=True)


def catalogue(fals, which):
    return fals.V if which == "items" else fals.U


def similar(fals, which, ids, k):
    return fals.similar_items(ids, k) if which == "items" else fals.similar_users(ids, k)


@pytest.mark.parametrize("K", [8, 64, 128, 130, 200, 256])
def test_similar_matches_reference(K):
    M, N = 300, 1000                                      # neither catalogue a multiple of 128
    fals, _, _ = _model(M, N, K)
    for which in ("items", "users"):
        Y = catalogue(fals, which)
        full = np.random.default_rng(K).permutation(len(Y))
        for ids, engine in ((full, "tcgen05"), (full[:40], "fp64")):
            for k in (1, 10, 100):
                assert_same(similar(fals, which, ids, k), reference_similar(Y, ids, k))
                assert fals.recommend_stats()["engine"] == engine, (which, k, engine)


@pytest.mark.parametrize("case", ["duplicates", "zero_rows", "all_equal", "many_blocks", "overflow", "list_chunks"])
def test_tcgen05_engine_equals_exact_engine(case, monkeypatch):
    M, N, K = 400, 1500, 64
    fals, _, _ = _model(M, N, K, seed=11)
    U, V = fals.U, fals.V
    if case == "duplicates":                              # exact ties, ordered by id
        U[1::3] = U[0::3][:len(U[1::3])]
        V[1::3] = V[0::3][:len(V[1::3])]
    elif case == "zero_rows":                             # every score of a zero row is +0.0
        U[::5] = 0.0
        V[::5] = 0.0
    elif case == "all_equal":
        U, V = np.full_like(U, 0.125), np.full_like(V, 0.25)
    fals.setUV(U, V)
    if case == "many_blocks":
        monkeypatch.setenv("EALS_EVAL_FIRST_CHUNK", "128")
    elif case == "overflow":
        monkeypatch.setenv("EALS_EVAL_PAIR_CAP", "16")
        monkeypatch.setenv("EALS_EVAL_PAIR_HARD_CAP", "64")
    elif case == "list_chunks":
        monkeypatch.setenv("EALS_REC_LIST_BYTES", str(12 * 50 * 150))   # k = 50: lists for 150 queries at a time
    for which in ("items", "users"):
        Y = catalogue(fals, which)
        ids = np.arange(len(Y))
        for k in (5, 50):
            tc = similar(fals, which, ids, k)
            assert fals.recommend_stats()["engine"] == ("fp64" if case == "overflow" else "tcgen05")
            monkeypatch.setenv("EALS_EVAL_SCALAR", "1")
            ex = similar(fals, which, ids, k)
            assert fals.recommend_stats()["engine"] == "fp64"
            monkeypatch.delenv("EALS_EVAL_SCALAR")
            assert_same(tc, ex)
            assert_same(tc, reference_similar(Y, ids, k))
            if case == "duplicates":
                assert tc[0][0, 0] == 1 and tc[0][1, 0] == 0 and tc[1][0, 0] == tc[1][1, 0]
            if case in ("zero_rows", "all_equal"):
                q = 0                                     # a zero row (zero_rows) or any row (all_equal)
                want = np.arange(1, k + 1) if case == "all_equal" else np.arange(1, len(Y))[:k]
                assert np.array_equal(tc[0][q], want)
                assert case == "all_equal" or bits_equal(tc[1][q], np.zeros(k))


def test_edge_cases():
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    M, N, K = 150, 300, 16
    fals, _, _ = _model(M, N, K, seed=2)
    for which, nY in (("items", N), ("users", M)):
        Y = catalogue(fals, which)
        for ids in (np.full(200, 7, np.int32), np.full(3, 7, np.int32)):      # repeated ids: tcgen05, exact engine
            got = similar(fals, which, ids, 10)
            assert_same(got, reference_similar(Y, ids, 10))
            assert (got[0] == got[0][0]).all() and bits_equal(got[1], np.broadcast_to(got[1][0], got[1].shape))
        for k in (nY - 1, nY, nY + 5, 1024):              # k >= n_Y - 1: padding, and the query itself never listed
            ids = np.arange(nY)
            items, scores = similar(fals, which, ids, k)
            assert_same((items, scores), reference_similar(Y, ids, k))
            assert not (items == ids[:, None]).any()
            assert (items[:, nY - 1:] == -1).all() and np.isneginf(scores[:, nY - 1:]).all()
    # a one-row catalogue: nothing to list
    M1 = 130
    one = MF_fastALS(SparseMat.from_csr(M1, 1, np.arange(M1 + 1, dtype=np.int64), np.zeros(M1, np.int32)), None,
                     factors=K, showLoss=False, device=0)
    one.run_epochs(1)
    for ids in (np.zeros(M1, np.int32), np.zeros(1, np.int32)):
        items, scores = one.similar_items(ids, 5)
        assert (items == -1).all() and np.isneginf(scores).all()


def test_model_untouched(monkeypatch):
    """similar_users and similar_items leave factors, S caches, Wi, loss, timers and the prediction-cache state alone: a
    model that calls them between epochs (graph replay included) trains to the same bits as one that does not, and
    recommend and ranking_metrics answer as before: no state of the normalised catalogue is reused."""
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    monkeypatch.setenv("EALS_HEAVY_MIN", "64")
    M, N, K = 300, 500, 32
    rp, ci = random_csr(M, N, 20, seed=8, empty_frac=0.02)
    a = MF_fastALS(SparseMat.from_csr(M, N, rp, ci), None, factors=K, showLoss=False, device=0)
    b = MF_fastALS(SparseMat.from_csr(M, N, rp, ci), None, factors=K, showLoss=False, device=0)
    for m in (a, b):
        m.run_epochs(2)
    trp, tci = random_csr(M, N, 5, seed=9, empty_frac=0.1)
    test = SparseMat(M, N, trp, tci, None, None)
    users = np.arange(M)
    snap = lambda: (a.timings_detail(), a.timings_total(), a.factor_hash(), a.SU, a.SV, a.Wi)
    rec0 = [a.recommend(users, k) for k in (10, 100)] + [a.recommend(users[:40], 10)]
    rm0 = a.ranking_metrics(test, 10, per_user=True, ranks=True)
    before = snap()
    a.similar_users(users, 10)
    a.similar_items(np.arange(N), 10)
    a.similar_users(users, 100)
    after = snap()
    assert before[:3] == after[:3]
    assert all(bits_equal(x, y) for x, y in zip(before[3:], after[3:]))
    rec1 = [a.recommend(users, k) for k in (10, 100)] + [a.recommend(users[:40], 10)]
    for x, y in zip(rec0, rec1):
        assert_same(x, y)
    rm1 = a.ranking_metrics(test, 10, per_user=True, ranks=True)
    assert np.array_equal(rm0["ranks"], rm1["ranks"]) and bits_equal(rm0["per_user"], rm1["per_user"])
    assert a.loss() == b.loss()
    for m in (a, b):
        m.run_epochs(3)
    assert a.factor_hash() == b.factor_hash() and a.loss() == b.loss()


def test_argument_errors():
    import torch
    from eals_cpp_b200 import _lib
    from eals_cpp_b200._lib import EalsError
    M, N, K = 150, 300, 16
    fals, _, _ = _model(M, N, K, epochs=1)
    dev = "cuda:0"
    calls = []
    for call, nY in ((fals.similar_items, N), (fals.similar_users, M)):
        for bad in ([0, nY], [-1]):
            calls += [lambda c=call, b=bad: c(b, 5), lambda c=call, b=bad: c(torch.tensor(b, dtype=torch.int32, device=dev), 5)]
        calls += [lambda c=call: c([0], 0), lambda c=call: c([0], 1025)]
    for call in calls:
        with pytest.raises(EalsError) as e:
            call()
        assert e.value.code == ERR_ARG and fals.lib.eals_last_error()
    with pytest.raises(EalsError) as e:
        fals.similar_items(torch.tensor([3, N + 7], dtype=torch.int32, device=dev), 5)
    assert f"item {N + 7} (position 1)".encode() in fals.lib.eals_last_error()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    ids, out = np.array([0, 1], np.int32), np.zeros((2, 5), np.int32)
    H = _lib.EALS_HOST
    fn, h, err = fals.lib.eals_similar, fals.h, fals.lib.eals_last_error
    assert fn(h, _lib.BUF_SU, H, 2, p(ids), 5, p(out), None) == ERR_ARG and b"which" in err()
    assert fn(h, _lib.BUF_V, 5, 2, p(ids), 5, p(out), None) == ERR_ARG and b"space" in err()
    assert fn(h, _lib.BUF_V, H, 2, None, 5, p(out), None) == ERR_ARG and b"null" in err()
    assert fn(h, _lib.BUF_U, H, 2, p(ids), 5, None, None) == ERR_ARG and b"null" in err()
    assert fn(h, _lib.BUF_U, H, -1, p(ids), 5, p(out), None) == ERR_ARG
    # scores are optional, and the model still answers after every rejected call
    assert fals.lib.eals_similar(fals.h, _lib.BUF_V, H, 2, p(ids), 5, p(out), None) == 0
    items, _ = fals.similar_items(ids, 5)
    assert np.array_equal(out, items)


def test_device_tensors():
    import torch
    M, N, K = 200, 600, 48
    fals, _, _ = _model(M, N, K, seed=3)
    dev = "cuda:0"
    for which, nY in (("items", N), ("users", M)):
        ids = np.random.default_rng(1).permutation(nY).astype(np.int32)
        want = similar(fals, which, ids, 10)
        assert_same(similar(fals, which, torch.from_numpy(ids).to(dev), 10), want)
        assert_same(similar(fals, which, torch.from_numpy(ids).to(dev).to(torch.int64), 10), want)
        assert_same(similar(fals, which, ids.tolist(), 10), want)


@pytest.mark.parametrize("world", [2, 4, 8])
def test_group_equals_single_model(world):
    from eals_cpp_b200.model import GroupMF_fastALS, SparseMat
    M, N, K = 500, 900, 32
    fals, rp, ci = _model(M, N, K, seed=9)
    g = GroupMF_fastALS(SparseMat.from_csr(M, N, rp, ci), None, factors=K, showLoss=False, devices=[0] * world)
    g.setUV(fals.U, fals.V)
    rng = np.random.default_rng(world)
    for k in (10, 100):
        for ids in (rng.permutation(N), rng.permutation(N)[:97]):
            assert_same(g.similar_items(ids, k), fals.similar_items(ids, k))
        for ids in (rng.permutation(M), rng.permutation(M)[:61]):
            assert_same(g.similar_users(ids, k), fals.similar_users(ids, k))
    g.close()


def _ngpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


def test_one_process_per_gpu_similar():
    """torch.distributed, one process per GPU: every rank gets the whole result.  With fewer than two GPUs NCCL cannot
    place two ranks on one device, so the same check runs through virtual ranks."""
    if _ngpus() < 2:
        test_group_equals_single_model(2)
        return
    world = min(_ngpus(), 4)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(29800 + world),
           os.path.join(ROOT, "tests", "dist_similar_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "dist similar ok" in res.stdout


def test_cpp_driver_similar_matches_python(tmp_path):
    """eals_main --similar-items (include/MF_fastALS.h over eals_group) writes what MF_fastALS.similar_items returns on
    the same split and factors."""
    from eals_cpp_b200 import build
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    from test_gpu_driver import _ratings
    exe = build.build_host_example()
    data = tmp_path / "tiny.rating"
    split = _ratings(str(data))
    M = len(split)
    N = 1 + max(max(t + [g]) for t, g in split)
    ckpt, out = tmp_path / "f.eals", tmp_path / "sim.txt"
    res = subprocess.run([exe, "--data", str(data), "--factors", "8", "--iters", "2", "--save", str(ckpt),
                          "--similar-items", "5", "--similar-out", str(out)], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    rp = np.concatenate([[0], np.cumsum([len(t) for t, _ in split])]).astype(np.int64)
    ci = np.concatenate([np.array(t, np.int32) for t, _ in split])
    fals = MF_fastALS(SparseMat.from_csr(M, N, rp, ci), None, factors=8, showLoss=False, device=0)
    fals.load(str(ckpt))
    items, scores = fals.similar_items(np.arange(N), 5)
    want = [(i, j) for i in range(N) for j in range(5) if items[i, j] >= 0]
    got = out.read_text().split("\n")[:-1]
    assert len(got) == len(want) > 0
    for line, (i, j) in zip(got, want):
        a, b, c = line.split()
        assert (int(a), int(b)) == (i, items[i, j]) and float(c) == scores[i, j]
