"""C5 retrieval benchmark: recommend() (top-10 and top-100, seen items excluded) for ALL users of the c4 matrix
(10M users x 2M items, K = 128) on the factors after 5 trained epochs — trained factors, not random ones: how well
the tcgen05 filter and the early-out work depends on the score distribution.

Prints one JSON line: seconds of the first and second call per k (host clock after a synchronise), the engine
and the library's stats, the first item block's tensor rate against the sustained bf16 peak bench.py uses, the
card name and power limit read in this run, and a 64-user sample compared item for item and bit for bit with
the exact fp64 engine (EALS_EVAL_SCALAR=1).

    python tools/recommend_bench.py [--workload c4] [--epochs 5] [--gpus N]
--gpus N runs through eals_group (GroupMF_fastALS) over GPUs 0..N-1."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power = out[0].split(", ")
        return {"name": name, "power_limit": power}
    except Exception as e:          # the measurement stands without the label, but says so
        return {"name": None, "power_limit": None, "error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c4")
    ap.add_argument("--epochs", type=int, default=5)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--ks", default="10,100")
    args = ap.parse_args()
    import torch
    import bench
    from eals_cpp_b200.model import GroupMF_fastALS, MF_fastALS
    spec, sm, _ = bench.build_workload(args.workload, 0)
    M, N, K = spec["M"], spec["N"], spec["K"]
    U0, V0 = bench.random_factors(M, N, K, 0)
    if args.gpus > 1:
        host = lambda a: a.cpu().numpy() if hasattr(a, "cpu") else a
        from eals_cpp_b200.model import SparseMat
        hsm = SparseMat(M, N, host(sm.row_ptr), host(sm.col_idx), host(sm.col_ptr), host(sm.row_idx))
        fals = GroupMF_fastALS(hsm, None, factors=K, showLoss=False, devices=list(range(args.gpus)), init=False)
        fals.setUV(U0.cpu().numpy(), V0.cpu().numpy())
    else:
        fals = MF_fastALS(sm, None, factors=K, showLoss=False, init=False, device=0)
        fals.setUV(U0, V0)
    del U0, V0
    for _ in range(args.epochs):
        fals.update_user(); fals.update_item()
    fals.sync()
    peaks, _ = bench.measured_peaks()
    peak = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
    out = {"workload": args.workload, "users": M, "items": N, "factors": K, "epochs": args.epochs, "gpus": args.gpus,
           "card": card(), "bf16_peak_tflops_sustained": peak, "runs": {}}
    users = np.arange(M, dtype=np.int32)
    rng = np.random.default_rng(0)
    sample = np.sort(rng.choice(M, 64, replace=False)).astype(np.int32)
    stats_model = fals if args.gpus == 1 else None
    for k in (int(x) for x in args.ks.split(",")):
        secs = []
        for _ in range(2):
            fals.sync(); t0 = time.perf_counter()
            items, scores = fals.recommend(users, k)
            fals.sync(); secs.append(time.perf_counter() - t0)
        run = {"first_call_s": secs[0], "second_call_s": secs[1]}
        if stats_model is not None:
            st = stats_model.recommend_stats()
            run.update(st)
            if "first_block" in st:
                run["first_block"]["frac_of_bf16_peak"] = st["first_block"]["tflops"] / peak
        os.environ["EALS_EVAL_SCALAR"] = "1"
        si, ss = fals.recommend(sample, k)
        del os.environ["EALS_EVAL_SCALAR"]
        run["sample_users"] = len(sample)
        run["sample_item_mismatches"] = int((si != items[sample]).sum())
        run["sample_score_bit_mismatches"] = int((ss.view(np.int64) != scores[sample].view(np.int64)).sum())
        out["runs"][f"top{k}"] = run
        del items, scores
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
