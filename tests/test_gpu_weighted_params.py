"""Training parity with weighted ratings, non-default hyperparameters and the documented switches (DESIGN.md §6b).

The rest of the parity suite trains all-ones ratings with the default w0 / alpha / reg / init.  Here one seeded
matrix (``weighted_matrix``) reaches every CD kernel family on both sides with non-unit ratings: user rows on both
sides of every length-bucket edge, a row of more than 32 slabs of 256 (several reduction groups at either slab
size), item columns of one-CTA and slab length, empty users and unrated items.  Ratings are uniform in [0.5, 5)
with planted exact 1.0 values and a few large ones (25).

Bounds are the suite's: factors 1e-10 absolute, scaled by max(1, max|oracle|) because weighted factors grow
well past 1; loss 1e-10 relative; S caches 1e-11 relative to their largest entry; initial factors bit for bit.
Bit-identity checks compare int64 views."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import random_csr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# user rows on both sides of every edge of kBucketMax (eals_b200.cu), ~700, and one row over 32 x 256 nonzeros
ROW_LENGTHS = [1, 31, 32, 33, 64, 65, 96, 97, 128, 129, 256, 257, 384, 385, 512, 513, 700, 9000]
N_EMPTY = 6                                  # users ROW_LENGTHS..+N_EMPTY rate nothing
ITEM_COLS = {41: 50, 43: 100, 57: 200, 61: 450, 3: 1300, 17: 2600, 29: 5100}   # item -> raters
N_UNRATED = 40                               # the last items are rated by nobody
M_USERS, N_ITEMS = 5200, 9500
USER_CTA, USER_SLAB = ROW_LENGTHS.index(257), ROW_LENGTHS.index(9000)
ITEM_CTA, ITEM_SLAB = 57, 17

H1 = dict(w0=1.5, alpha=0.4, reg=0.3, init_mean=0.02, init_stdev=0.05)
H2 = dict(w0=40.0, alpha=1.0, reg=1e-4)
H3 = dict(alpha=0.0)                         # pow(0, 0) = 1: unrated items weigh as much as rated ones


def csr(rows):
    row_ptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    col_idx = np.concatenate([np.array(sorted(r), np.int32) for r in rows] + [np.zeros(0, np.int32)])
    return row_ptr, col_idx


def ratings(n, seed):
    """Uniform in [0.5, 5), every 7th exactly 1.0, about 30 of value 25."""
    rng = np.random.default_rng(seed)
    val = rng.uniform(0.5, 5.0, n)
    val[::7] = 1.0
    val[rng.choice(n, size=min(n, 30), replace=False)] = 25.0
    return val


def weighted_rows(seed=0):
    rng = np.random.default_rng(seed)
    rateable = N_ITEMS - N_UNRATED
    rows = [set(rng.choice(rateable, size=n, replace=False).tolist()) for n in ROW_LENGTHS]
    rows += [set() for _ in range(N_EMPTY)]
    first = len(rows)
    rows += [set(rng.choice(rateable, size=int(min(40, rng.geometric(1 / 4))), replace=False).tolist())
             for _ in range(first, M_USERS)]
    for c, n in ITEM_COLS.items():           # the exact-length users above keep their lengths
        for u in rng.choice(np.arange(first, M_USERS), size=n, replace=False):
            rows[u].add(c)
    return rows


def weighted_matrix(seed=0):
    """(M, N, row_ptr, col_idx, val) of the matrix described in the module docstring."""
    row_ptr, col_idx = csr(weighted_rows(seed))
    return M_USERS, N_ITEMS, row_ptr, col_idx, ratings(len(col_idx), seed + 100)


def grown_matrix(seed=0):
    """The same users with about 12 more ratings for 900 of them: more nonzeros, so device buffers grow."""
    rows = weighted_rows(seed)
    rng = np.random.default_rng(seed + 7)
    for u in rng.choice(np.arange(len(ROW_LENGTHS) + N_EMPTY, M_USERS), size=900, replace=False):
        rows[u].update(rng.choice(N_ITEMS - N_UNRATED, size=12, replace=False).tolist())
    row_ptr, col_idx = csr(rows)
    return M_USERS, N_ITEMS, row_ptr, col_idx, ratings(len(col_idx), seed + 200)


def bits_equal(a, b):
    a, b = np.ascontiguousarray(a, np.float64), np.ascontiguousarray(b, np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


def check_factors(got, want, what):
    bound = 1e-10 * max(1.0, float(np.abs(want).max()))
    err = float(np.abs(got - want).max())
    assert err <= bound, f"{what}: max |diff| {err:.3e} > {bound:.3e}"


def check_S(got, want, what, rel=1e-11):
    err, bound = float(np.abs(got - want).max()), rel * float(np.abs(want).max())
    assert err <= bound, f"{what}: max |diff| {err:.3e} > {bound:.3e}"


def check_loss(got, want, what):
    assert abs(got - want) <= 1e-10 * abs(want), f"{what}: loss {got!r} vs oracle {want!r}"


def models(matrix, K, weighted=True, **hp):
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    from oracle.bindings import PortModel
    M, N, row_ptr, col_idx, val = matrix
    val = val if weighted else None
    fals = MF_fastALS(SparseMat.from_csr(M, N, row_ptr, col_idx, val), None, factors=K, showLoss=False,
                      debug_sync=True, **hp)
    return fals, PortModel(M, N, row_ptr, col_idx, val, factors=K, **hp)


def train_and_check(fals, port, epochs=2, what=""):
    """U after every user half-epoch, V after every item half-epoch, the loss after every epoch, then S."""
    for it in range(epochs):
        fals.update_user(); port.update_user()
        check_factors(fals.U, port.U, f"{what} U after user sweep {it}")
        fals.update_item(); port.update_item()
        check_factors(fals.V, port.V, f"{what} V after item sweep {it}")
        check_loss(fals.loss(), port.loss(), f"{what} epoch {it}")
    check_S(fals.SU, port.SU, f"{what} SU")
    check_S(fals.SV, port.SV, f"{what} SV")


def set_port_matrix(port, M, N, row_ptr, col_idx, val):
    from oracle.bindings import csr_to_csc
    port.row_ptr = np.ascontiguousarray(row_ptr, np.int64)
    port.col_idx = np.ascontiguousarray(col_idx, np.int32)
    port.val = None if val is None else np.ascontiguousarray(val, np.float64)
    port.col_ptr, port.row_idx, port.cval, _ = csr_to_csc(M, N, port.row_ptr, port.col_idx, port.val)


@pytest.fixture(scope="module")
def matrix():
    return weighted_matrix()


def test_weighted_matrix_reaches_every_kernel_family(matrix):
    """The builder itself: every bucket edge on the user side, >1 reduction group at slab 256, one-CTA and slab
    columns on the item side, empty users, unrated items and the planted rating values."""
    M, N, row_ptr, col_idx, val = matrix
    lens = np.diff(row_ptr)
    assert lens[:len(ROW_LENGTHS)].tolist() == ROW_LENGTHS
    assert max(ROW_LENGTHS) > 32 * 256 and N > max(ROW_LENGTHS)
    assert (lens == 0).sum() >= N_EMPTY
    col_lens = np.bincount(col_idx, minlength=N)
    assert (col_lens[N - N_UNRATED:] == 0).all()
    assert col_lens[ITEM_CTA] > 128 and col_lens[ITEM_CTA] <= 512
    assert all(col_lens[c] >= n for c, n in ITEM_COLS.items()) and col_lens.max() > 5000
    assert (val == 1.0).any() and (val == 25.0).any() and val.min() >= 0.5


# ---- B. weighted parity -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [1, 8, 40, 128, 200, 256])
def test_weighted_sweeps_match_oracle(K, matrix):
    """Two weighted epochs through warp, one-CTA and slab rows on both sides (K = 1 and 8 leave a partial 16-factor
    block, 40 is not a multiple of 16, 200 and 256 take the LD = 256 kernels), the cached loss stream, then the
    single-row API on a one-CTA row and a slab row of either side."""
    fals, port = models(matrix, K)
    assert bits_equal(fals.U, port.U) and bits_equal(fals.V, port.V)
    train_and_check(fals, port, what=f"K={K}")
    for i in (ITEM_CTA, ITEM_SLAB):          # item rows read SU only: the oracle's SV patch does not matter
        fals.update_item_thread(i); port.update_item(i, i + 1)
    check_factors(fals.V, port.V, "V after update_item_thread")
    fals.refresh_S(); port.init_S()
    for u in (USER_CTA, USER_SLAB):
        fals.update_user_thread(u); port.update_user(u, u + 1)
    check_factors(fals.U, port.U, "U after update_user_thread")


@pytest.mark.parametrize("mode", ["nocache", "refresh2"])
def test_weighted_prediction_cache_modes(mode, matrix, monkeypatch):
    """The recompute-every-sweep path and the periodic cache refresh on the weighted matrix."""
    monkeypatch.setenv(*{"nocache": ("EALS_NO_PRED_CACHE", "1"), "refresh2": ("EALS_PRED_REFRESH_EVERY", "2")}[mode])
    fals, port = models(matrix, 40)
    train_and_check(fals, port, epochs=3, what=mode)


def test_weighted_update_model_on_a_heavy_row(matrix):
    """updateModel on the slab user: once a new entry (rating 1), once overwriting a non-unit rating with 1."""
    M, N, row_ptr, col_idx, val = matrix
    fals, port = models(matrix, 40)
    fals.update_user(); port.update_user(); port.SU = port.p.gram_plain(port.U)
    fals.update_item(); port.update_item(); port.SV = port.p.gram_weighted(port.V, port.Wi)
    u = USER_SLAB
    row = col_idx[row_ptr[u]:row_ptr[u + 1]]
    rated = np.bincount(col_idx, minlength=N) > 0
    new = int(next(i for i in range(N) if rated[i] and i not in set(row.tolist())))
    k = int(row_ptr[u] + np.flatnonzero(val[row_ptr[u]:row_ptr[u + 1]] != 1.0)[0])
    rp, ci, v = row_ptr, col_idx, val
    for i in (new, int(col_idx[k])):
        fals.updateModel(u, i)
        a, b = int(rp[u]), int(rp[u + 1])
        pos = a + int(np.searchsorted(ci[a:b], i))
        if pos < b and ci[pos] == i:
            v = v.copy(); v[pos] = 1.0
        else:
            ci, v = np.insert(ci, pos, np.int32(i)), np.insert(v, pos, 1.0)
            rp = rp.copy(); rp[u + 1:] += 1
        set_port_matrix(port, M, N, rp, ci, v)
        for _ in range(10):
            port.update_user(u, u + 1)
            port.update_item(i, i + 1)
        check_factors(fals.U, port.U, f"U after updateModel({u}, {i})")
        check_factors(fals.V, port.V, f"V after updateModel({u}, {i})")
        check_S(fals.SU, port.SU, "SU after updateModel", rel=1e-10)
        check_S(fals.SV, port.SV, "SV after updateModel", rel=1e-10)


# ---- C. bit identity ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [64, 200])
def test_all_ones_values_equal_no_values_bit_for_bit(K, matrix):
    """val = 1.0 everywhere and val = None both make the kernels compute w*w and w - Wi with w = 1."""
    M, N, row_ptr, col_idx, _ = matrix
    ones = (M, N, row_ptr, col_idx, np.ones(len(col_idx)))
    a, _ = models(ones, K)
    b, _ = models(ones, K, weighted=False)
    for _ in range(2):
        a.update_user(); b.update_user()
        a.update_item(); b.update_item()
    assert bits_equal(a.U, b.U) and bits_equal(a.V, b.V)
    assert bits_equal(a.SU, b.SU) and bits_equal(a.SV, b.SV)
    assert a.loss() == b.loss()


def test_graph_replay_with_weights_across_set_train(matrix):
    """run_epochs(graph=True) equals the same epochs run call by call, also after setTrain switches unit ->
    weighted -> unit -> weighted (the last with more nonzeros, so the value buffers are reallocated): a replayed
    graph must not read a stale or freed value pointer."""
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    M, N, rp, ci, val = matrix
    _, _, rp2, ci2, val2 = grown_matrix()
    K = 32
    sm = SparseMat.from_csr(M, N, rp, ci, val)
    a = MF_fastALS(sm, None, factors=K, showLoss=False)
    b = MF_fastALS(sm, None, factors=K, showLoss=False)
    for step, nxt in enumerate([None, SparseMat.from_csr(M, N, rp, ci), SparseMat.from_csr(M, N, rp, ci, val),
                                SparseMat.from_csr(M, N, rp2, ci2), SparseMat.from_csr(M, N, rp2, ci2, val2)]):
        if nxt is not None:
            a.setTrain(nxt); b.setTrain(nxt)
        for _ in range(2):
            a.update_user(); a.update_item()
        b.run_epochs(2, graph=True)
        assert bits_equal(a.U, b.U) and bits_equal(a.V, b.V), step
        assert a.loss() == b.loss(), step
    # ... and the call-by-call model followed the last (weighted, grown) matrix
    from oracle.bindings import PortModel
    port = PortModel(M, N, rp2, ci2, val2, factors=K)
    port.U[:], port.V[:], port.Wi[:] = a.U, a.V, a.Wi
    port.init_S()
    a.update_user(); port.update_user()
    a.update_item(); port.update_item()
    check_factors(a.U, port.U, "U")
    check_factors(a.V, port.V, "V")


def _device_mat(sm):
    import torch
    from eals_cpp_b200.model import SparseMat
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to("cuda:0")
    return SparseMat(sm.M, sm.N, d(sm.row_ptr), d(sm.col_idx), d(sm.col_ptr), d(sm.row_idx), d(sm.row_val),
                     d(sm.col_val))


def test_device_resident_weighted_matrix_equals_host(matrix):
    """A model created from torch CUDA tensors with row_val / col_val, and a setTrain from device tensors, give the
    same bits as the host-array model."""
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    M, N, rp, ci, val = matrix
    _, _, rp2, ci2, val2 = grown_matrix()
    K = 48
    host = SparseMat.from_csr(M, N, rp, ci, val)
    dev = _device_mat(host)
    assert dev.on_device
    a = MF_fastALS(host, None, factors=K, showLoss=False, device=0)
    b = MF_fastALS(dev, None, factors=K, showLoss=False, device=0)
    for nxt in (None, SparseMat.from_csr(M, N, rp2, ci2, val2)):
        if nxt is not None:
            a.setTrain(nxt); b.setTrain(_device_mat(nxt))
        for _ in range(2):
            a.update_user(); b.update_user()
            a.update_item(); b.update_item()
        assert bits_equal(a.U, b.U) and bits_equal(a.V, b.V)
        assert bits_equal(a.SU, b.SU) and bits_equal(a.SV, b.SV)
        assert a.loss() == b.loss()


# ---- D. hyperparameters -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hp", [H1, H2, H3], ids=["H1", "H2", "H3"])
def test_hyperparameters_match_oracle(hp, matrix):
    """w0 and alpha reach the item weights, init_mean / init_stdev the initial factors, reg the three solves and the
    loss."""
    fals, port = models(matrix, 40, **hp)
    assert bits_equal(fals.U, port.U) and bits_equal(fals.V, port.V)
    assert np.allclose(fals.Wi, port.Wi, rtol=1e-15, atol=0)
    check_S(fals.SU, port.SU, "initial SU")
    check_S(fals.SV, port.SV, "initial SV")
    train_and_check(fals, port, what=str(hp))


def test_fold_in_uses_the_model_reg(matrix, port):
    """fold_in under H1 equals the oracle's user sweep with reg = 0.3."""
    fals, _ = models(matrix, 40, **H1)
    fals.update_user(); fals.update_item()
    assert fals.reg == H1["reg"]
    N, K, n = fals.itemCount, 40, 80
    rp, ci = random_csr(n, N, 20, seed=5, empty_frac=0.05)
    val = ratings(len(ci), 6)
    from eals_cpp_b200.model import SparseMat
    got = fals.fold_in(SparseMat(n, N, rp, ci, None, None, val), n_iter=3)
    want = np.zeros((n, K))
    V, SV, Wi = fals.V, fals.SV, fals.Wi
    for _ in range(3):
        port.update_user_sweep(rp, ci, val, want, V, np.zeros((K, K)), SV, Wi, H1["reg"], patch_S=False)
    check_factors(got, want, "fold_in")


# ---- E. weighted multi-rank ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 4, 8])
def test_weighted_group_matches_oracle(world, matrix):
    """Virtual ranks on GPU 0 with weights and H1: every rank trains on its slice of the values."""
    run_group_weighted([0] * world, matrix)


def run_group_weighted(devices, matrix, K=40):
    from eals_cpp_b200.model import GroupMF_fastALS, SparseMat
    M, N, rp, ci, val = matrix
    fals = GroupMF_fastALS(SparseMat.from_csr(M, N, rp, ci, val), None, factors=K, showLoss=False, devices=devices,
                           **H1)
    from oracle.bindings import PortModel
    port = PortModel(M, N, rp, ci, val, factors=K, **H1)
    world = len(devices)
    assert bits_equal(fals.U, port.U) and bits_equal(fals.V, port.V)

    def check_ranks(what, rel=1e-11):
        assert fals.replicas_consistent(), what
        for r in range(world):
            U, V = fals.rank_factors(r)
            check_factors(U, port.U, f"{what}: U of rank {r}")
            check_factors(V, port.V, f"{what}: V of rank {r}")
            SU, SV = fals.rank_S(r)
            check_S(SU, port.SU, f"{what}: SU of rank {r}", rel)
            check_S(SV, port.SV, f"{what}: SV of rank {r}", rel)

    train_and_check(fals, port, what=f"world {world}")
    check_ranks("trained")
    _, _, rp2, ci2, val2 = grown_matrix()
    fals.setTrain(SparseMat.from_csr(M, N, rp2, ci2, val2))
    set_port_matrix(port, M, N, rp2, ci2, val2)
    train_and_check(fals, port, what=f"world {world} after growing setTrain")
    check_ranks("after setTrain")
    # overwrite a non-unit rating of a user owned by the last rank
    u = next(u for u in range(M - 1, -1, -1) if (val2[rp2[u]:rp2[u + 1]] != 1.0).any())
    assert u >= fals.user_bounds[world - 1]
    k = int(rp2[u] + np.flatnonzero(val2[rp2[u]:rp2[u + 1]] != 1.0)[0])
    i = int(ci2[k])
    port.SU = port.p.gram_plain(port.U); port.SV = port.p.gram_weighted(port.V, port.Wi)
    fals.updateModel(u, i)
    v3 = val2.copy(); v3[k] = 1.0
    set_port_matrix(port, M, N, rp2, ci2, v3)
    for _ in range(10):
        port.update_user(u, u + 1)
        port.update_item(i, i + 1)
    check_ranks("after updateModel", rel=1e-10)
    fals.close()


# ---- F. switches, one process each --------------------------------------------------------------------------------
def run_switch_worker(env, out):
    clean = {k: v for k, v in os.environ.items() if not k.startswith("EALS_")}
    res = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "switch_parity_worker.py"), str(out)],
                         capture_output=True, text=True, timeout=900, env=dict(clean, **env))
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert res.stdout.strip().splitlines()[-1].startswith("ok"), res.stdout[-3000:]
    return dict(np.load(out))


@pytest.fixture(scope="module")
def switch_defaults(tmp_path_factory):
    return run_switch_worker({}, tmp_path_factory.mktemp("switch_defaults") / "single.npz")


def same_bits(a, b):
    return all(bits_equal(a[k], b[k]) for k in ("U", "V", "SU", "SV"))


@pytest.mark.parametrize("env", [
    {"EALS_SLAB": "256"},
    {"EALS_SLAB": "256", "EALS_HEAVY_BATCH_NNZ": "3000"},
    {"EALS_SLAB": "256", "EALS_HEAVY_MIN": "128"},
    {"EALS_HEAVY_MIN": "32"},
    {"EALS_HEAVY_MIN": "128"},
], ids=lambda e: ",".join(f"{k}={v}" for k, v in e.items()))
def test_slab_switches_match_oracle(env, switch_defaults, tmp_path):
    """Slab width 256 (heavy_step_kernel<..., 256>: rows of 513, ~700 and 9000 end in a partial slab), several
    heavy batches, and lower slab thresholds (rows of 129 and 257 become one- and two-slab heavy rows).  The worker
    checks the oracle; a different reduction order must show in at least one bit, or the switch did not act."""
    got = run_switch_worker(env, tmp_path / "out.npz")
    assert not same_bits(got, switch_defaults)


@pytest.mark.parametrize("wpb", ["1", "3"])
def test_warp_rows_per_block_is_bit_identical(wpb, switch_defaults, tmp_path):
    """EALS_WARP_WPB caps the row-warps of a warp-kernel CTA; a row's arithmetic does not depend on the CTA it runs
    in, so the result is bit-identical and nothing observable changes (not even the launch count).  That the cap
    reaches the launch was confirmed during development with a temporary stderr print of the warps per block."""
    got = run_switch_worker({"EALS_WARP_WPB": wpb}, tmp_path / "out.npz")
    assert same_bits(got, switch_defaults)


# ---- G. weighted, one process per GPU -----------------------------------------------------------------------------
def _ngpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.mark.parametrize("gather", ["1", "0"])
@pytest.mark.parametrize("partition", ["cost", "nnz"])
def test_weighted_one_process_per_gpu(partition, gather, matrix):
    """torch.distributed with weights and H1: both partitions, with and without the chunked upload plus all-gather
    of the values (``_device_matrix``), and a weighted setTrain.  With fewer than 2 GPUs NCCL cannot place two ranks
    on one device, so the scenario runs through virtual ranks instead."""
    world = 2
    if _ngpus() < world:
        run_group_weighted([0] * world, matrix)
        return
    env = dict(os.environ, EALS_CHECK_REPLICAS="1", EALS_GATHER_UPLOAD=gather)
    env.pop("EALS_PARTITION", None)
    if partition == "nnz":
        env["EALS_PARTITION"] = "nnz"
    port = 29800 + 10 * (partition == "nnz") + int(gather)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "dist_weighted_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "dist weighted ok" in res.stdout and f"partition {partition}" in res.stdout, res.stdout[-3000:]
