"""Worker for the one-process-per-GPU ranking-metrics test: run under torch.distributed.run with N ranks (one per GPU).
Every rank builds the same matrices and factors, calls the collective ranking_metrics and checks the WHOLE result
against a single-rank model of its own: per-user values and ranks bit for bit, means within 1e-12."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import torch
    import torch.distributed as dist
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    from conftest import random_csr
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    M, N, K = 600, 800, 32
    rp, ci = random_csr(M, N, 12, seed=9, empty_frac=0.02)
    tp, ti = random_csr(M, N, 6, seed=10, empty_frac=0.1)
    sm, test = SparseMat.from_csr(M, N, rp, ci), SparseMat(M, N, tp, ti, None, None)
    rng = np.random.default_rng(3)
    U0, V0 = rng.standard_normal((M, K)) * 0.3, rng.standard_normal((N, K)) * 0.3
    fals = MF_fastALS(sm, None, factors=K, showLoss=False, device=local)
    assert fals.world == dist.get_world_size() > 1
    fals.setUV(U0, V0)
    single = MF_fastALS(sm, None, factors=K, showLoss=False, device=local, distributed=False)
    single.setUV(U0, V0)
    names = ("hit_rate", "precision", "recall", "ndcg", "map", "mrr")
    for k in (10, 100):
        for exclude in (True, False):
            a = fals.ranking_metrics(test, k, exclude_seen=exclude, per_user=True, ranks=True)
            b = single.ranking_metrics(test, k, exclude_seen=exclude, per_user=True, ranks=True)
            assert np.array_equal(a["ranks"], b["ranks"]), (rank, k, exclude)
            assert np.array_equal(a["per_user"].view(np.int64), b["per_user"].view(np.int64)), (rank, k, exclude)
            np.testing.assert_allclose([a[n] for n in names], [b[n] for n in names], rtol=1e-12, atol=0)
            assert a["users"] == b["users"]
    dist.barrier()
    if rank == 0:
        print(f"dist ranking metrics ok: world {fals.world}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
