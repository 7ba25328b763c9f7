"""Fold-in benchmark on the c4 model (10M users x 2M items, K = 128) after 5 trained epochs.

Workload: 1M histories, the train rows of users 0 .. 1M-1, folded in from zero init.  Reports
  * fold_in at n_iter 1 and 10: seconds of the ABI call with device inputs and outputs (host clock after a
    synchronise; first and second call) and the rate nnz * K * n_iter / s;
  * recommend_vectors(U[users], exclude = the users' train rows) against recommend(users), top-10, for the same 1M
    users, run alternately (--rounds times each) in this one process, and whether their results are identical;
  * the latency of fold_in + recommend_vectors(top-10, exclude = the history) for a single history (exact engine):
    median and max over --single calls, the history being one train row of median length.
The card name and power limit are read in the same run and printed beside the numbers, as one JSON line.

    python tools/fold_in_bench.py [--workload c4] [--epochs 5] [--histories 1000000] [--rounds 3] [--single 50]"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c4")
    ap.add_argument("--epochs", type=int, default=5)
    ap.add_argument("--histories", type=int, default=1_000_000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--single", type=int, default=50)
    args = ap.parse_args()
    import torch
    import bench
    from recommend_bench import card
    from eals_cpp_b200 import _lib
    from eals_cpp_b200._lib import check
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    spec, sm, _ = bench.build_workload(args.workload, 0)
    M, N, K = spec["M"], spec["N"], spec["K"]
    U0, V0 = bench.random_factors(M, N, K, 0)
    fals = MF_fastALS(sm, None, factors=K, showLoss=False, init=False, device=0)
    fals.setUV(U0, V0)
    del U0, V0
    for _ in range(args.epochs):
        fals.update_user(); fals.update_item()
    fals.sync()
    dev = "cuda:0"
    n = min(args.histories, M)
    rp = sm.row_ptr[:n + 1].contiguous()                  # device tensors: offsets into the whole index array
    ci = sm.col_idx
    nnz = int(rp[-1] - rp[0])
    h = SparseMat(n, N, rp, ci, None, None)
    out = {"workload": args.workload, "users": M, "items": N, "factors": K, "epochs": args.epochs, "card": card(),
           "histories": n, "history_nnz": nnz}

    def timed(fn):
        torch.cuda.synchronize(); fals.sync()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize(); fals.sync()
        return time.perf_counter() - t0, r

    Q = torch.empty((n, K), dtype=torch.float64, device=dev)
    for n_iter in (1, 10):
        call = lambda: check(fals.lib.eals_fold_in(fals.h, _lib.EALS_DEVICE, n, C.c_void_p(rp.data_ptr()),
                                                   C.c_void_p(ci.data_ptr()), None, None, n_iter, C.c_void_p(Q.data_ptr())))
        secs = [timed(call)[0] for _ in range(2)]
        out[f"fold_in_iter{n_iter}"] = {"first_call_s": secs[0], "second_call_s": secs[1],
                                        "nnz_K_iter_per_s": nnz * K * n_iter / secs[1]}

    users = torch.arange(n, dtype=torch.int32, device=dev)
    Uq = fals.device_tensor(_lib.BUF_U)[:n, :K].contiguous()
    rec_s, vec_s = [], []
    same = True
    for _ in range(args.rounds):
        t, (ri, rs) = timed(lambda: fals.recommend(users, 10))
        rec_s.append(t)
        t, (vi, vs) = timed(lambda: fals.recommend_vectors(Uq, 10, exclude=h))
        vec_s.append(t)
        same = same and np.array_equal(ri, vi) and np.array_equal(rs.view(np.int64), vs.view(np.int64))
    out["top10"] = {"recommend_s": rec_s, "recommend_vectors_s": vec_s, "identical": bool(same),
                    "engine": fals.recommend_stats()["engine"]}
    del Uq, ri, rs, vi, vs

    lens = np.diff(rp.cpu().numpy())
    u = int(np.argsort(lens, kind="stable")[len(lens) // 2])
    one = SparseMat(1, N, rp[u:u + 2].contiguous(), ci, None, None)
    lat = []
    for _ in range(args.single + 1):
        t, _ = timed(lambda: fals.recommend_vectors(fals.fold_in(one), 10, exclude=one))
        lat.append(t)
    lat = lat[1:]                                          # the first call sizes the workspace
    out["single_history"] = {"history_len": int(lens[u]), "calls": len(lat), "median_s": float(np.median(lat)),
                             "max_s": float(np.max(lat)), "engine": fals.recommend_stats()["engine"]}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
