"""ctypes declarations for libeals_b200.so (include/eals_b200.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``eals_cpp_b200.build.build_library``.
There is no fallback: if the shared object is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libeals_b200.so")

EALS_HOST, EALS_DEVICE = 0, 1
BUF_U, BUF_V, BUF_SU, BUF_SV, BUF_WI, BUF_LOSS_TERMS, BUF_PC_USER, BUF_PC_ITEM = range(8)
EVAL_REFERENCE, EVAL_EXACT = 0, 1
ERR_ARG = -1
FLAG_SYNC_EACH_CALL = 1


class EalsParams(C.Structure):
    _fields_ = [
        ("struct_bytes", C.c_int32), ("n_users", C.c_int32), ("n_items", C.c_int32),
        ("factors", C.c_int32), ("topk", C.c_int32),
        ("w0", C.c_double), ("alpha", C.c_double), ("reg", C.c_double),
        ("init_mean", C.c_double), ("init_stdev", C.c_double),
        ("device", C.c_int32), ("input_space", C.c_int32),
        ("user_begin", C.c_int32), ("user_end", C.c_int32),
        ("item_begin", C.c_int32), ("item_end", C.c_int32),
        ("flags", C.c_int32), ("reserved", C.c_int32),
        ("n_ranks", C.c_int32), ("rank", C.c_int32),
        ("user_bounds", C.c_int32 * 9), ("item_bounds", C.c_int32 * 9),
    ]


class EalsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libeals_b200 error {code}: {msg}")
        self.code = code


# name -> (restype, argtypes); every symbol include/eals_b200.h declares
_P = C.c_void_p
SIGNATURES = {
    "eals_abi_version": (C.c_int, []),
    "eals_last_error": (C.c_char_p, []),
    "eals_default_params": (None, [C.POINTER(EalsParams)]),
    "eals_create": (C.c_int, [C.POINTER(EalsParams), _P, _P, _P, _P, _P, _P, C.POINTER(_P)]),
    "eals_destroy": (C.c_int, [_P]),
    "eals_set_train": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "eals_init_factors": (C.c_int, [_P]),
    "eals_debug_init_stream": (C.c_int, [C.c_double, C.c_double, _P, C.c_int64]),
    "eals_init_seconds": (C.c_int, [_P, C.POINTER(C.c_double)]),
    "eals_set_factors": (C.c_int, [_P, C.c_int32, _P, _P]),
    "eals_get_factors": (C.c_int, [_P, C.c_int32, _P, _P]),
    "eals_save_factors": (C.c_int, [_P, C.c_char_p]),
    "eals_load_factors": (C.c_int, [_P, C.c_char_p]),
    "eals_get_factor_row": (C.c_int, [_P, C.c_int32, C.c_int32, _P]),
    "eals_set_item_weights": (C.c_int, [_P, C.c_int32, _P]),
    "eals_get_item_weights": (C.c_int, [_P, C.c_int32, _P]),
    "eals_refresh_S": (C.c_int, [_P]),
    "eals_get_S": (C.c_int, [_P, C.c_int32, _P, _P]),
    "eals_update_user": (C.c_int, [_P]),
    "eals_update_item": (C.c_int, [_P]),
    "eals_run_epochs": (C.c_int, [_P, C.c_int32, C.c_int32]),
    "eals_sweep_users": (C.c_int, [_P]),
    "eals_sweep_items": (C.c_int, [_P]),
    "eals_gram_users": (C.c_int, [_P]),
    "eals_gram_items": (C.c_int, [_P]),
    "eals_update_user_row": (C.c_int, [_P, C.c_int32]),
    "eals_update_item_row": (C.c_int, [_P, C.c_int32]),
    "eals_patch_SU": (C.c_int, [_P, _P, _P]),
    "eals_patch_SV": (C.c_int, [_P, C.c_int32, _P, _P]),
    "eals_loss_terms": (C.c_int, [_P, _P]),
    "eals_loss": (C.c_int, [_P, C.POINTER(C.c_double)]),
    "eals_predict": (C.c_int, [_P, C.c_int32, C.c_int32, C.POINTER(C.c_double)]),
    "eals_evaluate": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "eals_evaluate_user": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
    "eals_eval_stats": (C.c_int, [_P, _P]),
    "eals_recommend": (C.c_int, [_P, C.c_int32, C.c_int32, _P, C.c_int32, C.c_int32, _P, _P]),
    "eals_recommend_stats": (C.c_int, [_P, _P]),
    "eals_fold_in": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, _P, C.c_int32, _P]),
    "eals_recommend_vectors": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, C.c_int32, _P, _P]),
    "eals_ranking_metrics": (C.c_int, [_P, C.c_int32, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "eals_leading_dim": (C.c_int, [_P]),
    "eals_device_buffer": (C.c_int, [_P, C.c_int32, C.POINTER(_P), C.POINTER(C.c_int64)]),
    "eals_stream": (C.c_int, [_P, C.POINTER(_P)]),
    "eals_set_stream": (C.c_int, [_P, _P, C.c_int32]),
    "eals_sync": (C.c_int, [_P]),
    "eals_factor_hash": (C.c_int, [_P, _P]),
    "eals_ipc_handle": (C.c_int, [_P, C.c_int32, _P]),
    "eals_ipc_attach": (C.c_int, [_P, C.c_int32, C.c_int32, _P]),
    "eals_ipc_detach": (C.c_int, [_P]),
    "eals_ipc_generation": (C.c_int, [_P]),
    "eals_ipc_gc": (C.c_int, [_P]),
    "eals_nnz": (C.c_int64, [_P]),
    "eals_kernel_launches": (C.c_int64, [_P]),
    "eals_timings": (C.c_int, [_P, _P]),
    "eals_timings_total": (C.c_int, [_P, _P, _P, C.c_int32]),
    "eals_timings_detail": (C.c_int, [_P, _P, _P]),
    # eals_group: N ranks in one process (multi-GPU behind the C ABI; virtual ranks on one GPU)
    "eals_group_create": (C.c_int, [C.POINTER(EalsParams), C.c_int32, _P, _P, _P, _P, _P, _P, _P, C.POINTER(_P)]),
    "eals_group_destroy": (C.c_int, [_P]),
    "eals_group_size": (C.c_int, [_P]),
    "eals_group_model": (C.c_int, [_P, C.c_int32, C.POINTER(_P)]),
    "eals_group_bounds": (C.c_int, [_P, _P, _P]),
    "eals_group_set_train": (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "eals_group_init_factors": (C.c_int, [_P]),
    "eals_group_set_factors": (C.c_int, [_P, C.c_int32, _P, _P]),
    "eals_group_get_factors": (C.c_int, [_P, C.c_int32, _P, _P]),
    "eals_group_get_factor_row": (C.c_int, [_P, C.c_int32, C.c_int32, _P]),
    "eals_group_get_S": (C.c_int, [_P, C.c_int32, _P, _P]),
    "eals_group_set_item_weights": (C.c_int, [_P, C.c_int32, _P]),
    "eals_group_get_item_weights": (C.c_int, [_P, C.c_int32, _P]),
    "eals_group_update_user": (C.c_int, [_P]),
    "eals_group_update_item": (C.c_int, [_P]),
    "eals_group_update_user_row": (C.c_int, [_P, C.c_int32]),
    "eals_group_update_item_row": (C.c_int, [_P, C.c_int32]),
    "eals_group_patch_SU": (C.c_int, [_P, _P, _P]),
    "eals_group_patch_SV": (C.c_int, [_P, C.c_int32, _P, _P]),
    "eals_group_loss": (C.c_int, [_P, C.POINTER(C.c_double)]),
    "eals_group_predict": (C.c_int, [_P, C.c_int32, C.c_int32, C.POINTER(C.c_double)]),
    "eals_group_evaluate": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "eals_group_evaluate_user": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
    "eals_group_recommend": (C.c_int, [_P, C.c_int32, C.c_int32, _P, C.c_int32, C.c_int32, _P, _P]),
    "eals_group_fold_in": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, _P, C.c_int32, _P]),
    "eals_group_recommend_vectors": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, C.c_int32, _P, _P]),
    "eals_group_ranking_metrics": (C.c_int, [_P, C.c_int32, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "eals_group_sync": (C.c_int, [_P]),
    "eals_group_replicas_consistent": (C.c_int, [_P, C.POINTER(C.c_int32)]),
    "eals_group_save_factors": (C.c_int, [_P, C.c_char_p]),
    "eals_group_load_factors": (C.c_int, [_P, C.c_char_p]),
    "eals_group_kernel_launches": (C.c_int64, [_P]),
    "eals_partition": (C.c_int, [_P, C.c_int32, C.c_int32, _P]),
}

_lib = None


def load() -> C.CDLL:
    """dlopen the in-tree library and attach signatures.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError(
                f"{LIB_PATH} not built — run `python -c 'import __graft_entry__ as g; g.build()'`. "
                "eals_cpp_b200 has no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(code: int) -> None:
    if code != 0:
        raise EalsError(code, load().eals_last_error().decode(errors="replace"))
