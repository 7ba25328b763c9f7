"""eval_stats() and recommend_stats() describe the last call, whichever engine answered it."""
import numpy as np
import pytest

from test_gpu_recommend import _model, assert_same, reference_topk


@pytest.mark.gpu
def test_eval_stats_describe_the_last_evaluate(monkeypatch):
    """After the exact engine (pair-list overflow, evaluate_for_user, EALS_EVAL_SCALAR=1) the candidate and pair
    counts are zero, not those of an earlier evaluate on the tensor-core filter."""
    M, N, K = 300, 200, 16
    fals, _, _ = _model(M, N, K, seed=3)
    U, V = fals.U, fals.V
    order = np.argsort(-(U @ V.T), axis=1, kind="stable")
    gt = order[:, 5].astype(np.int32)                  # about 5 larger scores: every user is a close call

    def filtered():
        fals.evaluate(gt, 10)
        st = fals.eval_stats()
        assert st["engine"] == "tcgen05" and st["candidates"] > 0 and st["pairs_rescored"] > 0, st

    def exact():
        st = fals.eval_stats()
        assert st["engine"] == "fp64" and st["candidates"] == 0 and st["pairs_rescored"] == 0, st
        assert "first_block" not in st

    filtered()
    # all scores equal: every item is a candidate of every user, the pair list overflows, the exact engine answers
    fals.setUV(np.zeros_like(U), V)
    monkeypatch.setenv("EALS_EVAL_PAIR_CAP", "1000")
    monkeypatch.setenv("EALS_EVAL_PAIR_HARD_CAP", "5000")
    fals.evaluate(gt, 10)
    exact()
    monkeypatch.delenv("EALS_EVAL_PAIR_CAP")
    monkeypatch.delenv("EALS_EVAL_PAIR_HARD_CAP")
    fals.setUV(U, V)
    filtered()
    fals.evaluate_for_user(0, int(gt[0]), 10)
    exact()
    filtered()
    monkeypatch.setenv("EALS_EVAL_SCALAR", "1")
    fals.evaluate(gt, 10)
    exact()


def _chunks(n, k, list_bytes):
    """The users of one recommend call per chunk, as the library balances them."""
    max_per = min(n, max(1, list_bytes // (12 * k)))
    n_chunks = -(-n // max_per)
    per = -(-n // n_chunks)
    return [np.arange(s, min(n, s + per)) for s in range(0, n, per)]


@pytest.mark.gpu
def test_recommend_stats_combine_the_chunks(monkeypatch):
    """Several chunks in one call: pairs and users left after the first block are summed over the chunks, the first
    block is chunk 0's, and engine and seed are those of tcgen05 only if every chunk ran there."""
    M, N, K, k = 400, 1500, 32, 5
    fals, rp, ci = _model(M, N, K, seed=11)
    list_bytes = 12 * k * 150                          # lists for 150 users at a time: three chunks of ~134
    monkeypatch.setenv("EALS_REC_LIST_BYTES", str(list_bytes))
    monkeypatch.setenv("EALS_EVAL_FIRST_CHUNK", "128")      # the first block leaves users behind
    # one block of the all-zero users (every item a candidate) exceeds the hard cap, no block of the others does
    monkeypatch.setenv("EALS_EVAL_PAIR_HARD_CAP", "90000")
    chunks = _chunks(M, k, list_bytes)
    assert len(chunks) == 3
    users = np.arange(M)

    def per_chunk():
        out = []
        for c in chunks:
            assert_same(fals.recommend(c, k), reference_topk(fals.U, fals.V, rp, ci, c, k))
            out.append(fals.recommend_stats())
        return out

    for zero_last in (False, True):
        if zero_last:
            U = fals.U
            U[chunks[-1]] = 0
            fals.setUV(U, fals.V)
        alone = per_chunk()
        assert [s["engine"] for s in alone] == ["tcgen05", "tcgen05", "fp64" if zero_last else "tcgen05"]
        assert_same(fals.recommend(users, k), reference_topk(fals.U, fals.V, rp, ci, users, k))
        st = fals.recommend_stats()
        assert st["engine"] == ("fp64" if zero_last else "tcgen05")
        assert st["seed_items"] == (0 if zero_last else alone[0]["seed_items"]) and alone[0]["seed_items"] == 128
        assert st["pairs_rescored"] == sum(s["pairs_rescored"] for s in alone)
        assert st["users_left_after_first_block"] == sum(s["users_left_after_first_block"] for s in alone)
        assert st["users_left_after_first_block"] > 0
        assert ("first_block" in st) == ("first_block" in alone[0])
        if "first_block" in st:
            fb, fb0 = st["first_block"], alone[0]["first_block"]
            assert (fb["users"], fb["items"]) == (fb0["users"], fb0["items"]) == (len(chunks[0]), 128)
