"""Worker for the one-process-per-GPU fold-in test: run under torch.distributed.run with N ranks (one per GPU).
Every rank builds the same matrix and factors, calls the collective fold_in and recommend_vectors and checks the
WHOLE result against its own rank-local ABI call over all the queries (V, SV and Wi are the same on every rank)."""
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
    from eals_cpp_b200.model import MF_fastALS, SparseMat, _fold_in_call, _recommend_vectors_call
    M, N, K = 600, 800, 32
    rp, ci = random_csr(M, N, 12, seed=9, empty_frac=0.02)
    rng = np.random.default_rng(3)
    U0, V0 = rng.standard_normal((M, K)) * 0.3, rng.standard_normal((N, K)) * 0.3
    fals = MF_fastALS(SparseMat.from_csr(M, N, rp, ci), None, factors=K, showLoss=False, device=local)
    assert fals.world == dist.get_world_size() > 1
    fals.setUV(U0, V0)
    hrp, hci = random_csr(333, N, 15, seed=4, empty_frac=0.05)
    h = SparseMat(333, N, hrp, hci, None, None)
    dev = f"cuda:{local}"
    Q = fals.fold_in(h, n_iter=3)
    assert np.array_equal(Q.view(np.int64), _fold_in_call(fals.lib.eals_fold_in, fals.h, K, dev, h, None, 3).view(np.int64)), rank
    for k in (10, 100):
        gi, gs = fals.recommend_vectors(Q, k, exclude=h)
        wi, ws = _recommend_vectors_call(fals.lib.eals_recommend_vectors, fals.h, K, dev, Q, k, h)
        assert np.array_equal(gi, wi) and np.array_equal(gs.view(np.int64), ws.view(np.int64)), (rank, k)
    dist.barrier()
    if rank == 0:
        print(f"dist fold_in ok: world {fals.world}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
