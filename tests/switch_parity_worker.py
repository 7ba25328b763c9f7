"""Worker for the switch tests of test_gpu_weighted_params.py: one process per setting, because EALS_WARP_WPB is read
once per process.

    python switch_parity_worker.py OUT.npz

Trains the weighted matrix for two epochs at K = 40 on one model, checks every half-epoch against the CPU oracle,
writes U, V, SU, SV and the kernel-launch count to OUT.npz and prints a final ``ok`` line."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main(out):
    import torch
    torch.cuda.set_device(0)
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    from oracle.bindings import PortModel
    from test_gpu_weighted_params import check_factors, check_loss, check_S, weighted_matrix
    M, N, rp, ci, val = weighted_matrix()
    K = 40
    sm = SparseMat.from_csr(M, N, rp, ci, val)
    fals = MF_fastALS(sm, None, factors=K, showLoss=False, device=0)
    port = PortModel(M, N, rp, ci, val, factors=K)
    for it in range(2):
        fals.update_user(); port.update_user()
        check_factors(fals.U, port.U, f"U after user sweep {it}")
        fals.update_item(); port.update_item()
        check_factors(fals.V, port.V, f"V after item sweep {it}")
        check_loss(fals.loss(), port.loss(), f"epoch {it}")
    SU, SV = fals.SU, fals.SV
    check_S(SU, port.SU, "SU")
    check_S(SV, port.SV, "SV")
    launches = fals.kernel_launches()
    np.savez(out, U=fals.U, V=fals.V, SU=SU, SV=SV, launches=np.int64(launches))
    fals.close()
    switches = " ".join(f"{k}={v}" for k, v in sorted(os.environ.items()) if k.startswith("EALS_")) or "defaults"
    print(f"ok: {switches}, launches {launches}")


if __name__ == "__main__":
    main(sys.argv[1])
