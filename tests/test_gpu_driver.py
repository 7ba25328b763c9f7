"""The C++ drop-in path end to end on a GPU: eals_main (host/eals_main.cpp over include/MF_fastALS.h
over the C ABI) reads a ratings file like the reference's main.cpp:73-205, trains, evaluates and runs
one online update; its printed losses and metrics must match the CPU oracle on the same split."""
import os
import re
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ratings(path, M=120, N=80, seed=4):
    """`user item score timestamp` lines, users contiguous from 0, unique timestamps per user (the
    reference's std::sort is unstable on ties), a few duplicate (u, i) pairs to exercise the dedup."""
    rng = np.random.default_rng(seed)
    lines, split = [], []
    for u in range(M):
        n = int(rng.integers(3, 25))
        items = rng.integers(0, N, size=n)
        ts = rng.permutation(10_000)[:n] + 1
        for it, t in zip(items, ts):
            lines.append(f"{u}\t{it}\t{float(rng.integers(1, 6))}\t{t}")
        order = np.argsort(ts)
        test_item = int(items[order[-1]])
        train = sorted(set(int(x) for x in items[order[:-1]]))        # newest -> test, the rest deduplicated
        split.append((train, test_item))
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")
    return split


@pytest.mark.parametrize("devices", [None, "0,0,0"])
def test_cpp_driver_trains_evaluates_and_updates_online(tmp_path, devices):
    """devices=None: one GPU.  "0,0,0": the C++ class drives THREE ranks (eals_group; here all on GPU 0, on a
    multi-GPU box `--gpus N` spreads them) — users and items sharded, the exchange inside the library — and must
    print the same losses, metrics and online update."""
    from eals_cpp_b200 import build
    from oracle.bindings import PortModel, csr_to_csc
    exe = build.build_host_example()
    data = tmp_path / "tiny.rating"
    split = _ratings(str(data))
    M = len(split)
    N = 1 + max(max(t + [g]) for t, g in split)
    K, iters = 8, 3
    ckpt = tmp_path / "factors.eals"
    cmd = [exe, "--data", str(data), "--factors", str(K), "--iters", str(iters), "--online", "3,5", "--save", str(ckpt)]
    if devices:
        cmd += ["--devices", devices]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    out = res.stdout
    if devices:
        assert "replicas consistent: yes" in res.stderr
    assert os.path.getsize(ckpt) == 32 + 8 * (M * K + N * K + N)
    assert f"#Users\t{M}" in out and f"#items\t{N}" in out          # main.cpp:212-216 lines
    losses = [float(x) for x in re.findall(r"Iter=\d+ \S+ [-+] loss:(\S+)", out)]
    assert len(losses) == iters

    row_ptr = np.concatenate([[0], np.cumsum([len(t) for t, _ in split])]).astype(np.int64)
    col_idx = np.concatenate([np.array(t, np.int32) for t, _ in split])
    gt = np.array([g for _, g in split], np.int32)
    port = PortModel(M, N, row_ptr, col_idx, factors=K)
    for it in range(iters):
        port.update_user(); port.SU = port.p.gram_plain(port.U)
        port.update_item(); port.SV = port.p.gram_weighted(port.V, port.Wi)
        assert abs(losses[it] - port.loss()) <= 1e-5 * abs(port.loss())   # printed with 6 significant digits
    hr, ndcg, prec = [float(x) for x in re.search(r"<hr, ndcg, prec>: \t(\S+)\t(\S+)\t(\S+)", out).groups()]
    want = port.evaluate(gt, 10, compat=True)[0]
    assert np.allclose([hr, ndcg, prec], want, atol=5e-6)

    # online update of (3, 5): same schedule on the oracle (S caches patched after every row)
    u, i = 3, 5
    before = float(port.U[u] @ port.V[i])
    rows = [list(col_idx[row_ptr[r]:row_ptr[r + 1]]) for r in range(M)]
    if i not in rows[u]:
        rows[u] = sorted(rows[u] + [i])
    port.row_ptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    port.col_idx = np.concatenate([np.array(r, np.int32) for r in rows])
    port.col_ptr, port.row_idx, port.cval, _ = csr_to_csc(M, N, port.row_ptr, port.col_idx, None)
    if port.Wi[i] == 0.0:
        port.Wi[i] = 10.0 / N
        port.SV = port.p.gram_weighted(port.V, port.Wi)
    for _ in range(10):   # the oracle's row sweeps patch SU / SV themselves (MF_fastALS.cpp:127-132, 146-152)
        port.update_user(u, u + 1)
        port.update_item(i, i + 1)
    m = re.search(r"online \(3,5\): predict (\S+) -> (\S+) loss:(\S+)", out)
    got_before, got_after, got_loss = (float(x) for x in m.groups())
    assert abs(got_before - before) < 1e-10
    assert abs(got_after - float(port.U[u] @ port.V[i])) < 1e-10
    assert abs(got_loss - port.loss()) <= 1e-10 * abs(port.loss())


def test_cpp_driver_transcript_equals_the_reference_binary(tmp_path):
    """Same ratings file (tied timestamps, duplicates), what the reference's OWN driver (main.cpp + the five TUs,
    unmodified) printed (stored, see tests/reference_vectors.py) against ours with the run.sh defaults (K=64,
    20 iterations, top-10): every printed loss and the final <hr, ndcg, prec> line agree to the 6 significant
    digits the reference prints."""
    from reference_vectors import transcript_shape
    from test_oracle import _ratings_with_ties, _reference_transcript
    from eals_cpp_b200 import build
    _ratings_with_ties(str(tmp_path / "yelp.rating"))
    losses, metrics, counts, ref_lines = _reference_transcript(tmp_path)
    exe = build.build_host_example()
    res = subprocess.run([exe], cwd=str(tmp_path), capture_output=True, text=True, timeout=600)   # default --data yelp.rating
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    out = res.stdout
    for key in ("#Users", "#items", "#Ratings"):
        assert f"{key}\t{counts[key]}" in out
    ours = [float(x) for x in re.findall(r"Iter=\d+ \S+ [-+] loss:(\S+)", out)]
    assert len(ours) == 20
    assert ours == pytest.approx(losses, rel=2e-6)
    got = [float(x) for x in re.search(r"<hr, ndcg, prec>: \t(\S+)\t(\S+)\t(\S+)", out).groups()]
    assert got == pytest.approx(metrics, rel=2e-6, abs=1e-9)
    # the same lines in the same order (timings aside): a transcript diff is empty up to the numbers' noise
    assert transcript_shape(out)[:len(ref_lines)] == ref_lines
