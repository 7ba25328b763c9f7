"""The reference's values on the seeded inputs of the reference comparisons in test_oracle.py and
test_gpu_driver.py, stored in tests/golden/reference_vectors.json so that those comparisons run on any
checkout: the repository does not ship the reference's sources (oracle/Makefile builds it only where they are).

Every array comparison here is bit for bit, so an array is stored as the SHA-256 digest of its dtype, shape and
bytes: the same check as np.array_equal, in a few bytes.  Scalars are stored as JSON numbers, which keep a
float64 exactly.

The values were recorded from the C restatement (oracle/eals_oracle.c) and the C++ driver (host/eals_main.cpp)
at a commit where both had been checked against the compiled reference on exactly these inputs: factors, S
caches, losses and evaluation bit for bit, the driver's transcript to the six digits the reference prints.
Rerun `python tests/reference_vectors.py` only when these inputs change on purpose (the transcript needs a GPU).
"""
import hashlib
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "reference_vectors.json")

# (K, M, N, density, weighted ratings): every factor-count regime of the restatement
SMALL_CASES = [(8, 120, 90, 6, False), (20, 200, 310, 15, True), (64, 90, 40, 12, False),
               (129, 70, 50, 9, False), (200, 60, 45, 8, True)]


def digest(a) -> str:
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def file_digest(path) -> str:
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def case_id(K, M, N, dens, weighted) -> str:
    return f"K{K}_M{M}_N{N}_d{dens}" + ("_weighted" if weighted else "")


def load() -> dict:
    with open(GOLDEN) as f:
        return json.load(f)


def assert_same(got: dict, want: dict) -> None:
    """Checkpoint by checkpoint, in the order they were taken: the first difference names where the run left."""
    assert list(got) == list(want)
    for key in want:
        assert got[key] == want[key], f"differs from the reference at {key}"


def _eval(m, gt, topK, tag, out):
    mean, hr, ndcg, prec, _ = m.evaluate(gt, topK, compat=True)
    out[f"{tag}_mean"] = [float(x) for x in mean]
    out[f"{tag}_hr"], out[f"{tag}_ndcg"], out[f"{tag}_prec"] = digest(hr), digest(ndcg), digest(prec)


def small_case(port, K, M, N, dens, weighted) -> dict:
    """Initialisation, two epochs (factors and S caches after every half-epoch, loss after every epoch) and the
    reference-compatible evaluation at top-5, on the trained factors and on inflated ones (non-zero truncated
    scores for the ranking)."""
    from conftest import random_csr
    from oracle.bindings import PortModel
    row_ptr, col_idx = random_csr(M, N, dens, seed=K * 7 + M, empty_frac=0.08)
    val = np.random.default_rng(K).uniform(0.5, 2.5, len(col_idx)) if weighted else None
    gt = np.random.default_rng(K + 1).integers(0, N, M).astype(np.int32)
    m = PortModel(M, N, row_ptr, col_idx, val, factors=K, port=port)
    out = {"U0": digest(m.U), "V0": digest(m.V), "Wi": digest(m.Wi), "SU0": digest(m.SU), "SV0": digest(m.SV),
           "loss0": m.loss()}
    for e in (1, 2):
        m.update_user()
        out[f"U{e}"], out[f"SU{e}"] = digest(m.U), digest(m.SU)
        m.update_item()
        out[f"V{e}"], out[f"SV{e}"] = digest(m.V), digest(m.SV)
        out[f"loss{e}"] = m.loss()
    _eval(m, gt, 5, "eval", out)
    rng = np.random.default_rng(3)
    U = m.U * 25.0 + rng.normal(0, 0.6, m.U.shape)
    V = m.V * 25.0 + rng.normal(0, 0.6, m.V.shape)
    m.U[:], m.V[:] = U, V
    _eval(m, gt, 5, "eval_inflated", out)
    return out


def headline_case(port) -> dict:
    """The c1 workload in full (25677 x 25815, K = 64): the matrix, initialisation and one whole epoch."""
    from eals_cpp_b200 import datasets
    from oracle.bindings import PortModel
    d = datasets.powerlaw_csr(**datasets.WORKLOADS["c1"])
    K = datasets.WORKLOADS["c1"]["K"]
    out = {"row_ptr": digest(d.row_ptr), "col_idx": digest(d.col_idx)}
    m = PortModel(d.M, d.N, d.row_ptr, d.col_idx, factors=K, port=port)
    out.update(U0=digest(m.U), V0=digest(m.V), Wi=digest(m.Wi))
    m.update_user()
    out.update(U1=digest(m.U), SU1=digest(m.SU))
    m.update_item()
    out.update(V1=digest(m.V), SV1=digest(m.SV), loss1=m.loss())
    return out


def transcript_shape(text: str) -> list:
    """The transcript's lines with every number masked: timings aside, the same lines in the same order."""
    return [re.sub(r"[-+]?\d+(\.\d+)?(e[-+]?\d+)?", "#", l) for l in text.strip().split("\n") if l.strip()]


def parse_transcript(text: str):
    losses = [float(x) for x in re.findall(r"Iter=\d+ \S+ [-+] loss:(\S+)", text)]
    metrics = [float(x) for x in re.search(r"<hr, ndcg, prec>: \t(\S+)\t(\S+)\t(\S+)", text).groups()]
    counts = {k: int(re.search(k + r"\t(\d+)", text).group(1)) for k in ("#Users", "#items", "#Ratings")}
    return losses, metrics, counts


def transcript_case() -> dict:
    """The driver with the reference's defaults (K = 64, 20 iterations, top-10) on the ratings file with tied
    timestamps and duplicates of test_oracle._ratings_with_ties."""
    from eals_cpp_b200 import build
    from test_oracle import _ratings_with_ties
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "yelp.rating")
        _ratings_with_ties(path)
        res = subprocess.run([build.build_host_example()], cwd=d, capture_output=True, text=True, timeout=600, check=True)
        losses, metrics, counts = parse_transcript(res.stdout)
        return {"ratings_sha256": file_digest(path), "counts": counts, "losses": losses, "metrics": metrics,
                "lines": transcript_shape(res.stdout)}


def record(path=GOLDEN) -> None:
    from oracle.bindings import Port
    port = Port()
    out = {"small": {case_id(*c): small_case(port, *c) for c in SMALL_CASES},
           "headline_c1": headline_case(port),
           "transcript_ties": transcript_case()}
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    sys.path[:0] = [os.path.dirname(HERE)]
    record(*sys.argv[1:])
