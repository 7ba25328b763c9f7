"""similar_items' and similar_users' C ABI without a GPU: the symbols are bound, arguments are checked before any device
work, and without a device the calls cannot run: there is no model to call them on."""
import ctypes as C

import numpy as np
import pytest

NAMES = ("eals_similar", "eals_group_similar")


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def test_similar_symbols_are_bound():
    from eals_cpp_b200 import _lib
    lib = _lib.load()
    for name in NAMES:
        assert hasattr(lib, name) and name in _lib.SIGNATURES


def test_similar_rejects_null_arguments_without_a_device():
    from eals_cpp_b200 import _lib
    lib = _lib.load()
    ids = np.zeros(2, np.int32)
    out = np.zeros((2, 4), np.int32)
    H = _lib.EALS_HOST
    for fn in (lib.eals_similar, lib.eals_group_similar):
        for which in (_lib.BUF_U, _lib.BUF_V):
            assert fn(None, which, H, 2, _p(ids), 4, _p(out), None) == -1
            assert b"null" in lib.eals_last_error()


def test_similar_needs_a_device():
    """Both calls take a model, and without a device eals_create already fails with EALS_ERR_CUDA, so neither can
    reach a CPU path."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("box has a GPU")
    from eals_cpp_b200._lib import EalsError
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    sm = SparseMat.from_csr(2, 2, np.array([0, 1, 2], np.int64), np.array([0, 1], np.int32))
    for call in (lambda m: m.similar_items([0], 1), lambda m: m.similar_users([0], 1)):
        with pytest.raises(EalsError) as e:
            call(MF_fastALS(sm, None, factors=8, device=0))
        assert e.value.code == -2                          # EALS_ERR_CUDA
