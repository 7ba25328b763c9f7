"""Worker for the switch tests of test_gpu_weighted_params.py: one process per setting, because several switches
(EALS_WARP_WPB, EALS_ROUTE_INLINE, EALS_COPY_FAN, EALS_PEER_FENCE) are read once per process.

    python switch_parity_worker.py single|group OUT.npz

Trains the weighted matrix for two epochs at K = 40 (``single``: one model; ``group``: 4 virtual ranks on GPU 0),
checks every half-epoch against the CPU oracle, writes U, V, SU, SV and the kernel-launch count to OUT.npz and
prints a final ``ok`` line."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main(mode, out):
    import torch
    torch.cuda.set_device(0)
    from eals_cpp_b200.model import GroupMF_fastALS, MF_fastALS, SparseMat
    from oracle.bindings import PortModel
    from test_gpu_weighted_params import check_factors, check_loss, check_S, weighted_matrix
    M, N, rp, ci, val = weighted_matrix()
    K = 40
    sm = SparseMat.from_csr(M, N, rp, ci, val)
    if mode == "single":
        fals = MF_fastALS(sm, None, factors=K, showLoss=False, device=0)
    else:
        fals = GroupMF_fastALS(sm, None, factors=K, showLoss=False, devices=[0] * 4)
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
    if mode == "group":
        assert fals.replicas_consistent()
        for r in range(4):
            SUr, SVr = fals.rank_S(r)
            assert np.array_equal(SUr, SU) and np.array_equal(SVr, SV), r
    launches = fals.kernel_launches()
    np.savez(out, U=fals.U, V=fals.V, SU=SU, SV=SV, launches=np.int64(launches))
    fals.close()
    switches = " ".join(f"{k}={v}" for k, v in sorted(os.environ.items()) if k.startswith("EALS_")) or "defaults"
    print(f"ok: {mode}, {switches}, launches {launches}")


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
