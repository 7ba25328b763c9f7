"""Worker for the one-process-per-GPU similar test: run under torch.distributed.run with N ranks (one per GPU).  Every
rank builds the same matrix and factors, calls the collective similar_items and similar_users and checks the WHOLE
result against its own rank-local ABI call over all the queries (U and V are the same on every rank)."""
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
    from eals_cpp_b200 import _lib
    from eals_cpp_b200.model import MF_fastALS, SparseMat, _similar_call
    M, N, K = 600, 800, 32
    rp, ci = random_csr(M, N, 12, seed=9, empty_frac=0.02)
    rng = np.random.default_rng(3)
    U0, V0 = rng.standard_normal((M, K)) * 0.3, rng.standard_normal((N, K)) * 0.3
    fals = MF_fastALS(SparseMat.from_csr(M, N, rp, ci), None, factors=K, showLoss=False, device=local)
    assert fals.world == dist.get_world_size() > 1
    fals.setUV(U0, V0)
    dev = f"cuda:{local}"
    items, users = rng.permutation(N)[:517].astype(np.int32), rng.permutation(M)[:333].astype(np.int32)
    for k in (10, 100):
        for call, which, ids in ((fals.similar_items, _lib.BUF_V, items), (fals.similar_users, _lib.BUF_U, users)):
            gi, gs = call(ids, k)
            wi, ws = _similar_call(fals.lib.eals_similar, fals.h, which, dev, ids, k)
            assert np.array_equal(gi, wi) and np.array_equal(gs.view(np.int64), ws.view(np.int64)), (rank, k, which)
    dist.barrier()
    if rank == 0:
        print(f"dist similar ok: world {fals.world}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
