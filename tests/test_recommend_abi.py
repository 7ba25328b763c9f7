"""recommend's C ABI without a GPU: the symbols are bound, arguments are checked before any device work, and
without a device the call cannot run: there is no model to call it on."""
import ctypes as C

import numpy as np
import pytest


def test_recommend_symbols_are_bound():
    from eals_cpp_b200 import _lib
    lib = _lib.load()
    for name in ("eals_recommend", "eals_group_recommend", "eals_recommend_stats"):
        assert hasattr(lib, name) and name in _lib.SIGNATURES


def test_recommend_rejects_bad_arguments_without_a_device():
    from eals_cpp_b200 import _lib
    lib = _lib.load()
    users = np.zeros(1, np.int32)
    items = np.zeros((1, 4), np.int32)
    up, ip = users.ctypes.data_as(C.c_void_p), items.ctypes.data_as(C.c_void_p)
    assert lib.eals_recommend(None, _lib.EALS_HOST, 1, up, 4, 1, ip, None) == -1
    assert lib.eals_group_recommend(None, _lib.EALS_HOST, 1, up, 4, 1, ip, None) == -1
    assert lib.eals_recommend_stats(None, None) == -1
    assert b"null" in lib.eals_last_error()


def test_recommend_needs_a_device():
    """eals_recommend takes a model, and without a device eals_create already fails with EALS_ERR_CUDA, so no
    recommend call can reach a CPU path."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("box has a GPU")
    from eals_cpp_b200._lib import EalsError
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    sm = SparseMat.from_csr(2, 2, np.array([0, 1, 2], np.int64), np.array([0, 1], np.int32))
    with pytest.raises(EalsError) as e:
        MF_fastALS(sm, None, factors=8, device=0).recommend([0], 1)
    assert e.value.code == -2                              # EALS_ERR_CUDA
