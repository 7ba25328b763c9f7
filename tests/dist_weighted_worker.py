"""Worker for test_weighted_one_process_per_gpu: run under torch.distributed.run with one rank per GPU.
Every rank builds the weighted matrix of test_gpu_weighted_params.py, trains it with the non-default
hyperparameters H1 and checks its replica against the CPU oracle, before and after a weighted setTrain to a
matrix with more nonzeros.  EALS_PARTITION and EALS_GATHER_UPLOAD pick the partition and the upload path."""
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
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    from oracle.bindings import PortModel
    from test_gpu_weighted_params import (H1, check_factors, check_loss, check_S, grown_matrix, set_port_matrix,
                                          weighted_matrix)
    M, N, rp, ci, val = weighted_matrix()
    K = 40
    fals = MF_fastALS(SparseMat.from_csr(M, N, rp, ci, val), None, factors=K, showLoss=False, device=local, **H1)
    assert fals.world == dist.get_world_size() and fals.world > 1
    port = PortModel(M, N, rp, ci, val, factors=K, **H1)

    def train(what):
        for it in range(2):
            fals.update_user(); port.update_user()
            fals.update_item(); port.update_item()
            check_loss(fals.loss(), port.loss(), f"rank {rank} {what} epoch {it}")   # ends in a collective
            check_factors(fals.U, port.U, f"rank {rank} {what} U epoch {it}")
            check_factors(fals.V, port.V, f"rank {rank} {what} V epoch {it}")
            fals.barrier()            # replica reads are local: nobody sweeps on while another rank still reads
        check_S(fals.SU, port.SU, f"rank {rank} {what} SU")
        check_S(fals.SV, port.SV, f"rank {rank} {what} SV")
        assert fals.replicas_consistent(), (rank, what)

    train("first matrix")
    _, _, rp2, ci2, val2 = grown_matrix()
    fals.setTrain(SparseMat.from_csr(M, N, rp2, ci2, val2))
    set_port_matrix(port, M, N, rp2, ci2, val2)
    train("after weighted setTrain")
    dist.barrier()
    if rank == 0:
        part = "nnz" if os.environ.get("EALS_PARTITION") == "nnz" else "cost"
        print(f"dist weighted ok: world {fals.world}, partition {part}, "
              f"gather_upload {os.environ.get('EALS_GATHER_UPLOAD', '1')}, bounds {fals.user_bounds}")
    fals.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
