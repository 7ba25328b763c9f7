"""fold_in's and recommend_vectors' C ABI without a GPU: the symbols are bound, arguments are checked before any
device work, and without a device the calls cannot run: there is no model to call them on."""
import ctypes as C

import numpy as np
import pytest

NAMES = ("eals_fold_in", "eals_recommend_vectors", "eals_group_fold_in", "eals_group_recommend_vectors")


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def test_fold_in_symbols_are_bound():
    from eals_cpp_b200 import _lib
    lib = _lib.load()
    for name in NAMES:
        assert hasattr(lib, name) and name in _lib.SIGNATURES


def test_fold_in_rejects_bad_arguments_without_a_device():
    from eals_cpp_b200 import _lib
    lib = _lib.load()
    rp, ci = np.array([0, 1], np.int64), np.zeros(1, np.int32)
    out, Q = np.zeros((1, 8)), np.zeros((1, 8))
    items = np.zeros((1, 4), np.int32)
    H = _lib.EALS_HOST
    for fold_in in (lib.eals_fold_in, lib.eals_group_fold_in):
        assert fold_in(None, H, 1, _p(rp), _p(ci), None, None, 1, _p(out)) == -1
        assert b"null" in lib.eals_last_error()
    for rec in (lib.eals_recommend_vectors, lib.eals_group_recommend_vectors):
        assert rec(None, H, 1, _p(Q), None, None, 4, _p(items), None) == -1
        assert b"null" in lib.eals_last_error()


def test_fold_in_needs_a_device():
    """Both calls take a model, and without a device eals_create already fails with EALS_ERR_CUDA, so neither can
    reach a CPU path."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("box has a GPU")
    from eals_cpp_b200._lib import EalsError
    from eals_cpp_b200.model import MF_fastALS, SparseMat
    sm = SparseMat.from_csr(2, 2, np.array([0, 1, 2], np.int64), np.array([0, 1], np.int32))
    with pytest.raises(EalsError) as e:
        MF_fastALS(sm, None, factors=8, device=0).fold_in(sm)
    assert e.value.code == -2                              # EALS_ERR_CUDA
    with pytest.raises(EalsError) as e:
        MF_fastALS(sm, None, factors=8, device=0).recommend_vectors(np.zeros((1, 8)), 1)
    assert e.value.code == -2
