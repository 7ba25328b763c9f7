"""ranking_metrics' C ABI without a GPU: the symbols are bound, null arguments are rejected before any device work,
and without a device the call cannot run: there is no model to call it on."""
import ctypes as C

import numpy as np
import pytest

NAMES = ("eals_ranking_metrics", "eals_group_ranking_metrics")


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def test_ranking_metrics_symbols_are_bound():
    from eals_cpp_b200 import _lib
    lib = _lib.load()
    for name in NAMES:
        assert hasattr(lib, name) and name in _lib.SIGNATURES


def test_ranking_metrics_rejects_null_arguments():
    from eals_cpp_b200 import _lib
    lib = _lib.load()
    tp, ti = np.array([0, 1], np.int64), np.zeros(1, np.int32)
    sums, n = np.zeros(6), C.c_int64()
    H = _lib.EALS_HOST
    for fn in (lib.eals_ranking_metrics, lib.eals_group_ranking_metrics):
        assert fn(None, H, _p(tp), _p(ti), 10, 1, _p(sums), C.byref(n), None, None) == _lib.ERR_ARG
        assert b"null" in lib.eals_last_error()


def test_ranking_metrics_needs_a_device():
    """The call takes a model, and without a device eals_create already fails with EALS_ERR_CUDA, so it cannot reach
    a CPU path."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("box has a GPU")
    from eals_cpp_b200._lib import EalsError
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    sm = SparseMat.from_csr(2, 2, np.array([0, 1, 2], np.int64), np.array([0, 1], np.int32))
    with pytest.raises(EalsError) as e:
        MF_fastALS(sm, None, factors=8, device=0).ranking_metrics(sm, 1)
    assert e.value.code == -2                              # EALS_ERR_CUDA
