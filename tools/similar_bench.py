"""Similar-items / similar-users benchmark on the c4 model (10M users x 2M items, K = 128) after 5 trained epochs, the
model tools/recommend_bench.py builds: trained factors, not random ones, because how well the tcgen05 filter and the
early-out work depends on the score distribution.

Runs, each called twice (first and second call, seconds on the host clock after a synchronise):
    similar_items for all 2M items at k = 10 and k = 100, for 1 item and for 10,000 items at k = 10;
    similar_users for 1M users at k = 10.
Per call the library's stats (engine, pairs re-scored, queries left after the first block, the first block's shape,
time and tensor rate against the sustained bf16 peak bench.py uses), and a 64-query sample of the call compared item
for item and bit for bit with the exact fp64 engine (EALS_EVAL_SCALAR=1).  The card name and power limit are read in
the same run.  Prints one JSON line and, with --out, writes it to that file (rewritten after every run).

    python tools/similar_bench.py [--workload c4] [--epochs 5] [--out FILE]"""
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
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import bench
    from eals_cpp_b200.model import MF_fastALS
    spec, sm, _ = bench.build_workload(args.workload, 0)
    M, N, K = spec["M"], spec["N"], spec["K"]
    U0, V0 = bench.random_factors(M, N, K, 0)
    fals = MF_fastALS(sm, None, factors=K, showLoss=False, init=False, device=0)
    fals.setUV(U0, V0)
    del U0, V0
    for _ in range(args.epochs):
        fals.update_user(); fals.update_item()
    fals.sync()
    peaks, _ = bench.measured_peaks()
    peak = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
    out = {"workload": args.workload, "users": M, "items": N, "factors": K, "epochs": args.epochs,
           "card": card(), "bf16_peak_tflops_sustained": peak, "runs": {}}
    rng = np.random.default_rng(0)
    runs = [("items_all_top10", fals.similar_items, np.arange(N, dtype=np.int32), 10),
            ("items_all_top100", fals.similar_items, np.arange(N, dtype=np.int32), 100),
            ("items_1_top10", fals.similar_items, rng.choice(N, 1).astype(np.int32), 10),
            ("items_10000_top10", fals.similar_items, np.sort(rng.choice(N, 10000, replace=False)).astype(np.int32), 10),
            ("users_1M_top10", fals.similar_users, np.sort(rng.choice(M, 1000000, replace=False)).astype(np.int32), 10)]
    for name, call, ids, k in runs:
        secs = []
        for _ in range(2):
            fals.sync(); t0 = time.perf_counter()
            got, scores = call(ids, k)
            fals.sync(); secs.append(time.perf_counter() - t0)
        run = {"queries": len(ids), "k": k, "first_call_s": secs[0], "second_call_s": secs[1]}
        st = fals.recommend_stats()
        run.update(st)
        if "first_block" in st:
            run["first_block"]["frac_of_bf16_peak"] = st["first_block"]["tflops"] / peak
        sample = np.sort(rng.choice(len(ids), min(64, len(ids)), replace=False))
        os.environ["EALS_EVAL_SCALAR"] = "1"
        si, ss = call(ids[sample], k)
        del os.environ["EALS_EVAL_SCALAR"]
        run["sample_queries"] = len(sample)
        run["sample_item_mismatches"] = int((si != got[sample]).sum())
        run["sample_score_bit_mismatches"] = int((ss.view(np.int64) != scores[sample].view(np.int64)).sum())
        out["runs"][name] = run
        print(name, json.dumps(run), file=sys.stderr, flush=True)
        del got, scores
        if args.out:                # after every run, so that a partial result survives an interrupted one
            with open(args.out, "w") as f:
                f.write(json.dumps(out) + "\n")
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
