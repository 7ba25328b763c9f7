"""Worker for the one-process-per-GPU recommend test: run under torch.distributed.run with N ranks (one per GPU).
Every rank builds the same matrix and factors, calls the collective recommend and checks the WHOLE result against
a single-rank model of its own."""
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
    sm = SparseMat.from_csr(M, N, rp, ci)
    rng = np.random.default_rng(3)
    U0, V0 = rng.standard_normal((M, K)) * 0.3, rng.standard_normal((N, K)) * 0.3
    fals = MF_fastALS(sm, None, factors=K, showLoss=False, device=local)
    assert fals.world == dist.get_world_size() > 1
    fals.setUV(U0, V0)
    single = MF_fastALS(sm, None, factors=K, showLoss=False, device=local, distributed=False)
    single.setUV(U0, V0)
    users = rng.permutation(M)
    for k in (10, 100):
        gi, gs = fals.recommend(users, k)
        wi, ws = single.recommend(users, k)
        assert np.array_equal(gi, wi) and np.array_equal(gs.view(np.int64), ws.view(np.int64)), (rank, k)
    dist.barrier()
    if rank == 0:
        print(f"dist recommend ok: world {fals.world}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
