"""Ranking-metrics benchmark on c4 (10M users x 2M items, K = 128): a held-out split, 5 trained epochs on the rest,
then ranking_metrics(test, k) for k = 10 and 100 against the route without it, recommend(users, k) plus a lookup of
each test item in its user's list.

Split (seeded, on the device): for each user with at least 2 nonzeros, max(1, n // 10) of its n nonzeros, chosen at
random, go to the test matrix; the train matrix keeps the rest.  Prints one JSON line: per k the first and second
call's seconds (host clock after a synchronise), eval_stats() with the first item block's tensor rate against the
sustained bf16 peak bench.py uses, the same metrics on a 1M-user subset timed against recommend + lookup (the two
run alternately, twice each, and their ranks compared), a 64-user sample checked against recommend + lookup, and
the card name and power limit read in this run.

    python tools/ranking_metrics_bench.py [--workload c4] [--epochs 5] [--ks 10,100] [--subset 1000000]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def split(rp, ci, seed=0):
    """(train_ptr, train_idx, test_ptr, test_idx) of the held-out split, torch tensors on rp's device."""
    import torch
    dev = rp.device
    M = rp.numel() - 1
    lens = rp[1:] - rp[:-1]
    n_test = torch.where(lens >= 2, torch.clamp(lens // 10, min=1), torch.zeros_like(lens))
    row = torch.repeat_interleave(torch.arange(M, device=dev), lens)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    key = row.to(torch.float64) + torch.rand(row.numel(), generator=g, device=dev, dtype=torch.float64)
    order = torch.argsort(key)                         # rows stay contiguous, random order inside each
    del key
    pos = torch.arange(row.numel(), device=dev) - rp[:-1][row]   # position inside the row, in the shuffled order
    mask = torch.zeros(row.numel(), dtype=torch.bool, device=dev)
    mask[order[pos < n_test[row]]] = True
    del order, pos, row
    zero = torch.zeros(1, dtype=torch.int64, device=dev)
    test_ptr = torch.cat([zero, torch.cumsum(n_test, 0)])
    train_ptr = torch.cat([zero, torch.cumsum(lens - n_test, 0)])
    return train_ptr, ci[~mask].contiguous(), test_ptr, ci[mask].contiguous()


def recommend_ranks(fals, users, test_ptr, test_idx, k):
    """Ranks by the route without ranking_metrics: recommend(users, k) and each test item looked up in its list."""
    import torch
    dev = test_ptr.device
    u = torch.from_numpy(users.astype(np.int32)).to(dev)
    items, _ = fals.recommend(u, k)
    items = torch.from_numpy(items).to(dev)
    ul = u.to(torch.int64)
    lens = test_ptr[ul + 1] - test_ptr[ul]
    slot = torch.repeat_interleave(torch.arange(len(users), device=dev), lens)
    start = torch.repeat_interleave(test_ptr[ul], lens)
    first = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), torch.cumsum(lens, 0)[:-1]])
    ent = start + torch.arange(slot.numel(), device=dev) - torch.repeat_interleave(first, lens)
    hit = items[slot] == test_idx[ent].unsqueeze(1)
    rank = torch.where(hit.any(1), hit.to(torch.int32).argmax(1), torch.full_like(slot, -1))
    torch.cuda.synchronize()
    return ent.cpu().numpy(), rank.to(torch.int32).cpu().numpy()


def subset_matrix(M, N, test_ptr, test_idx, users):
    """The test matrix with only the rows of `users` (ascending) kept."""
    import torch
    from eals_cpp_b200.model import SparseMat
    dev = test_ptr.device
    keep = torch.zeros(M, dtype=torch.bool, device=dev)
    keep[torch.from_numpy(users.astype(np.int64)).to(dev)] = True
    lens = torch.where(keep, test_ptr[1:] - test_ptr[:-1], torch.zeros(M, dtype=torch.int64, device=dev))
    ent_keep = torch.repeat_interleave(keep, test_ptr[1:] - test_ptr[:-1])
    ptr = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), torch.cumsum(lens, 0)])
    return SparseMat(M, N, ptr, test_idx[ent_keep].contiguous(), None, None), ent_keep.nonzero().reshape(-1).cpu().numpy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c4")
    ap.add_argument("--epochs", type=int, default=5)
    ap.add_argument("--ks", default="10,100")
    ap.add_argument("--subset", type=int, default=1_000_000)
    args = ap.parse_args()
    import torch
    import bench
    from recommend_bench import card
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    spec, sm, _ = bench.build_workload(args.workload, 0)
    M, N, K = spec["M"], spec["N"], spec["K"]
    t0 = time.perf_counter()
    trp, tci, tp, ti = split(sm.row_ptr, sm.col_idx)
    del sm
    train = SparseMat.from_csr_device(M, N, trp, tci)
    test = SparseMat(M, N, tp, ti, None, None)
    torch.cuda.synchronize()
    split_s = time.perf_counter() - t0
    U0, V0 = bench.random_factors(M, N, K, 0)
    fals = MF_fastALS(train, None, factors=K, showLoss=False, init=False, device=0)
    fals.setUV(U0, V0)
    del U0, V0
    for _ in range(args.epochs):
        fals.update_user(); fals.update_item()
    fals.sync()
    peaks, _ = bench.measured_peaks()
    peak = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
    test_users = int(((tp[1:] - tp[:-1]) > 0).sum())
    out = {"workload": args.workload, "users": M, "items": N, "factors": K, "epochs": args.epochs, "card": card(),
           "train_nnz": int(trp[-1]), "test_nnz": int(tp[-1]), "test_users": test_users, "split_s": split_s,
           "bf16_peak_tflops_sustained": peak, "runs": {}}
    rng = np.random.default_rng(0)
    has_test = ((tp[1:] - tp[:-1]) > 0).cpu().numpy()
    subset = np.sort(rng.choice(np.nonzero(has_test)[0], min(args.subset, int(has_test.sum())), replace=False))
    sample = np.sort(rng.choice(subset, 64, replace=False))
    sub_test, sub_ent = subset_matrix(M, N, tp, ti, subset)
    for k in (int(x) for x in args.ks.split(",")):
        run = {}
        secs = []
        for _ in range(2):
            fals.sync(); t0 = time.perf_counter()
            res = fals.ranking_metrics(test, k, ranks=True)
            fals.sync(); secs.append(time.perf_counter() - t0)
            st = fals.eval_stats()
        run.update({"first_call_s": secs[0], "second_call_s": secs[1], "stats": st,
                    **{n: res[n] for n in ("hit_rate", "precision", "recall", "ndcg", "map", "mrr", "users")}})
        if "first_block" in st:
            st["first_block"]["frac_of_bf16_peak"] = st["first_block"]["tflops"] / peak
        ranks_all = res.pop("ranks")
        # 64-user sample: recommend + lookup
        ent, rk = recommend_ranks(fals, sample, tp, ti, k)
        run["sample_users"], run["sample_entries"] = len(sample), int(len(ent))
        run["sample_rank_mismatches"] = int((ranks_all[ent] != rk).sum())
        # the 1M-user subset, the two routes alternately
        t_rm, t_rec = [], []
        for _ in range(2):
            fals.sync(); t0 = time.perf_counter()
            sub = fals.ranking_metrics(sub_test, k, ranks=True)
            fals.sync(); t_rm.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            ent, rk = recommend_ranks(fals, subset, tp, ti, k)
            t_rec.append(time.perf_counter() - t0)
        run["subset"] = {"users": len(subset), "entries": int(len(sub_ent)), "ranking_metrics_s": t_rm, "recommend_lookup_s": t_rec,
                         "rank_mismatches": int((sub["ranks"] != rk).sum()) if len(rk) == len(sub["ranks"]) else -1,
                         "stats": fals.eval_stats()}
        out["runs"][f"k{k}"] = run
        print(json.dumps({f"k{k}": run}), file=sys.stderr, flush=True)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
