"""Pins the CPU oracle (oracle/eals_oracle.c, a C restatement) to the reference.

Anchors (SURVEY.md §8c — the reference ships no unit tests or vectors of its own besides
Outputs.txt, whose input file yelp.rating is not distributed):
  1. the committed fixtures in tests/golden/*.npz, produced by tests/golden/make_golden.py from the
     reference's own unmodified translation units;
  2. the reference's values on seeded inputs from K = 8 to 200 and at the full c1 size, stored in
     tests/golden/reference_vectors.json (see tests/reference_vectors.py);
  3. live, when oracle/_ref/libeals_ref.so was built from the reference's sources: its driver order.
The restatement follows the reference's operation order and is compiled with -ffp-contract=off, so
agreement is BIT-EXACT except through libm `pow` in the item weights (same libm here: also exact).
"""
import os

import numpy as np
import pytest

import reference_vectors
from conftest import random_csr
from oracle import bindings
from oracle.bindings import PortModel, Reference, csr_to_csc

GOLD = os.path.join(os.path.dirname(__file__), "golden")
have_ref = pytest.mark.skipif(not bindings.reference_available(), reason="compiled reference not available")

# SURVEY.md §8 row a2: first values of DenseMat::init(0, 0.01), probed from the reference
KAT_INIT = [-0.0012196578414159691, -0.010868180442613574, 0.0068428994379655488, -0.01075189149518029,
            0.00033269476420492392, 0.0074483559772278241, 0.0003360612264682257, -0.005266372061852982]


def test_init_stream_known_answers(port):
    got = port.normal_fill(8, 0.0, 0.01)
    assert got.tolist() == KAT_INIT
    gold = np.load(os.path.join(GOLD, "dense_init.npz"))["init"]
    assert np.array_equal(port.normal_fill(gold.size, 0.0, 0.01).reshape(gold.shape), gold)


@pytest.mark.parametrize("name", ["tiny_k8", "tiny_k64"])
def test_port_reproduces_golden_run(port, name):
    g = np.load(os.path.join(GOLD, f"{name}.npz"))
    M, N = int(g["row_ptr"].size - 1), int(g["Wi"].size)
    K = g["SU0"].shape[0]
    m = PortModel(M, N, g["row_ptr"], g["col_idx"], factors=K, port=port)
    assert np.array_equal(m.Wi, g["Wi"])
    assert np.array_equal(m.U[:4], g["U0_head"])
    assert np.array_equal(m.SU, g["SU0"]) and np.array_equal(m.SV, g["SV0"])
    losses = [m.loss()]
    for it in range(len(g["losses"]) - 1):
        m.update_user()
        if it == 0:
            assert np.array_equal(m.U, g["U_after_first_user_sweep"])
        m.update_item()
        if it == 0:
            assert np.array_equal(m.V, g["V_after_first_item_sweep"])
        losses.append(m.loss())
    assert np.array_equal(np.asarray(losses), g["losses"])
    assert np.array_equal(m.U, g["U_final"]) and np.array_equal(m.V, g["V_final"])
    assert np.array_equal(m.SU, g["SU_final"]) and np.array_equal(m.SV, g["SV_final"])
    mean, hr, ndcg, prec, _ = m.evaluate(g["test_items"], 10, compat=True)
    assert np.array_equal(hr, g["eval_hr"]) and np.array_equal(ndcg, g["eval_ndcg"])
    assert np.array_equal(prec, g["eval_prec"]) and np.array_equal(mean, g["eval_mean"])
    if "U_scaled" in g.files:      # non-zero truncated scores: the int-comparator heap order
        m.U[:], m.V[:] = g["U_scaled"], g["V_scaled"]
        mean, hr, ndcg, prec, _ = m.evaluate(g["test_items"], 10, compat=True)
        assert np.array_equal(hr, g["eval2_hr"]) and np.array_equal(ndcg, g["eval2_ndcg"])
        assert np.array_equal(prec, g["eval2_prec"]) and np.array_equal(mean, g["eval2_mean"])
        assert hr.sum() != g["eval_hr"].sum()


@pytest.mark.parametrize("K,M,N,dens,weighted", reference_vectors.SMALL_CASES)
def test_port_matches_live_reference(port, K, M, N, dens, weighted):
    """Against the values the reference's own object computed on these seeded inputs (stored, see
    tests/reference_vectors.py): factors, S caches, item weights and loss after initialisation and every
    half-epoch of two epochs, and the top-5 evaluation on trained and on inflated factors — bit for bit."""
    want = reference_vectors.load()["small"][reference_vectors.case_id(K, M, N, dens, weighted)]
    reference_vectors.assert_same(reference_vectors.small_case(port, K, M, N, dens, weighted), want)


def test_port_matches_live_reference_at_the_headline_size(port):
    """BASELINE.json configs[0] in full (yelp-shaped: 25677 x 25815, 669k interactions, K = 64, the synthetic
    stand-in bench.py calls c1): one whole epoch of the restatement against the reference's own object — factors,
    S caches and loss bit for bit (stored, see tests/reference_vectors.py).  This is the size the CPU baseline of
    bench.py is quoted on."""
    want = reference_vectors.load()["headline_c1"]
    reference_vectors.assert_same(reference_vectors.headline_case(port), want)


@have_ref
def test_buildmodel_call_order_matches_our_sweep_drivers(port):
    """ref_harness's half-epoch drivers repeat buildModel()'s call order: the real buildModel()
    must land on the same factors."""
    row_ptr, col_idx = random_csr(150, 100, 8, seed=77)
    a = Reference(150, 100, row_ptr, col_idx, factors=16)
    b = Reference(150, 100, row_ptr, col_idx, factors=16)
    a.build_model(3)
    for _ in range(3):
        b.update_user(); b.update_item()
    assert np.array_equal(a.U, b.U) and np.array_equal(a.V, b.V)
    assert np.array_equal(a.SU, b.SU) and np.array_equal(a.SV, b.SV)


def test_csc_orientation_matches_reference_append_order():
    """cols[i] lists users ascending (main.cpp:198-205 appends in (u asc, i asc) order)."""
    row_ptr, col_idx = random_csr(60, 40, 7, seed=5)
    col_ptr, row_idx, _, order = csr_to_csc(60, 40, row_ptr, col_idx)
    want = [[] for _ in range(40)]
    for u in range(60):
        for p in range(row_ptr[u], row_ptr[u + 1]):
            want[col_idx[p]].append(u)
    for i in range(40):
        assert row_idx[col_ptr[i]:col_ptr[i + 1]].tolist() == want[i]


def test_empty_rows_keep_initial_factors(port):
    row_ptr = np.array([0, 0, 2, 2, 3], np.int64)
    col_idx = np.array([0, 2, 1], np.int32)
    m = PortModel(4, 4, row_ptr, col_idx, factors=4, port=port)     # item 3 has no ratings either
    U0, V0 = m.U.copy(), m.V.copy()
    m.update_user(); m.update_item()
    assert np.array_equal(m.U[[0, 2]], U0[[0, 2]]) and np.array_equal(m.V[3], V0[3])
    assert not np.array_equal(m.U[1], U0[1])
    assert m.Wi[3] == 0.0


def test_parallel_init_stream_is_the_sequential_stream(monkeypatch):
    """eals_init_factors generates the reference's normal stream in parallel chunks (LCG skip-ahead + the real
    std::normal_distribution per chunk).  Exercised WITHOUT a GPU through the stand-alone export
    eals_debug_init_stream: several chunk sizes, lengths that end inside a chunk and inside a pair, against the
    oracle's sequential loop (itself pinned to the compiled reference above)."""
    import ctypes as C
    from eals_cpp_b200 import _lib
    from oracle.bindings import Port
    lib = _lib.load()
    port = Port()
    for chunk, n in ((8, 1), (8, 2), (8, 37), (64, 4096), (1000, 250_001), (1 << 16, 400_000)):
        monkeypatch.setenv("EALS_INIT_CHUNK", str(chunk))
        out = np.empty(n)
        assert lib.eals_debug_init_stream(C.c_double(0.0), C.c_double(0.01), out.ctypes.data_as(C.c_void_p), C.c_int64(n)) == 0
        want = port.normal_fill(n, 0.0, 0.01)
        assert np.array_equal(out, want), (chunk, n)
    monkeypatch.setenv("EALS_INIT_CHUNK", "4096")
    out = np.empty(100_003)
    lib.eals_debug_init_stream(C.c_double(1.5), C.c_double(2.0), out.ctypes.data_as(C.c_void_p), C.c_int64(len(out)))
    assert np.array_equal(out, port.normal_fill(len(out), 1.5, 2.0))


def _ratings_with_ties(path, M=90, N=60, seed=8):
    """`user item score timestamp` lines with MANY tied timestamps (also for the newest rating of a user) and
    duplicate (u, i) pairs: which of the tied ratings becomes the test item is decided by libstdc++'s unstable
    std::sort (main.cpp:122-124) and is part of the reference's behaviour."""
    rng = np.random.default_rng(seed)
    with open(path, "w") as f:
        for u in range(M):
            n = int(rng.integers(4, 40))
            items = rng.integers(0, N, size=n)
            ts = rng.integers(1, 6, size=n)              # only 5 distinct timestamps
            for it, t in zip(items, ts):
                f.write(f"{u}\t{it}\t{float(rng.integers(1, 6))}\t{t}\n")


def _reference_transcript(tmp_path):
    """What the reference's own driver (main.cpp, the run.sh defaults) prints on tmp_path/yelp.rating, stored (see
    tests/reference_vectors.py): its 20 losses, the final <hr, ndcg, prec>, the counts and its lines with the
    numbers masked."""
    want = reference_vectors.load()["transcript_ties"]
    assert reference_vectors.file_digest(tmp_path / "yelp.rating") == want["ratings_sha256"], "not the stored input"
    assert len(want["losses"]) == 20
    return want["losses"], want["metrics"], want["counts"], want["lines"]


def test_loader_split_matches_the_reference_binary_with_tied_timestamps(tmp_path):
    """Our loader (host/eals_main.cpp --dump-split, no GPU) against what the reference's own main.cpp printed on
    the same file, ties and duplicates included: same counts, and the oracle trained on OUR split reproduces the
    reference binary's 20 printed losses and its final metrics (which depend on every tie decision)."""
    import subprocess as sp
    from eals_cpp_b200 import build
    _ratings_with_ties(str(tmp_path / "yelp.rating"))
    losses, metrics, counts, _ = _reference_transcript(tmp_path)
    exe = build.build_host_example()
    split = tmp_path / "split.txt"
    res = sp.run([exe, "--data", str(tmp_path / "yelp.rating"), "--dump-split", str(split)], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    lines = open(split).read().split("\n")
    M, N = (int(x) for x in lines[0].split())
    rows, gt = [], []
    for u in range(M):
        v = [int(x) for x in lines[1 + u].split()]
        gt.append(v[0]); rows.append(v[1:])
    assert (M, N) == (counts["#Users"], counts["#items"]) and sum(len(r) for r in rows) == counts["#Ratings"]
    assert f"#Ratings\t{counts['#Ratings']}" in res.stdout
    row_ptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    col_idx = np.concatenate([np.array(r, np.int32) for r in rows])
    port = PortModel(M, N, row_ptr, col_idx, factors=64)               # main.cpp:133-144 defaults
    for it in range(20):
        port.update_user(); port.update_item()
        assert abs(port.loss() - losses[it]) <= 2e-6 * abs(losses[it]), it   # printed with 6 significant digits
    want = port.evaluate(np.array(gt, np.int32), 10, compat=True)[0]
    assert np.allclose(want, metrics, rtol=2e-6, atol=1e-9)
