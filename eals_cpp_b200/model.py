"""Host-side mirror of the reference's ``MF_fastALS`` class (MF_fastALS.h:15-80) over the C ABI.

This is plumbing, not the product: every number comes out of libeals_b200.so (hand-written sm_100a
kernels).  Python is used here because the tests and bench.py are Python and because the
multi-GPU launch model is one process per GPU under ``torch.distributed``; the C++ drop-in class
of the same name is ``include/MF_fastALS.h``.  Names, argument order and print formats follow the
reference:

    fals = MF_fastALS(trainMatrix, testRatings, topK, threadNum, factors, maxIter, w0, alpha, reg,
                      init_mean, init_stdev, showProgress, showLoss, userCount, itemCount)
    fals.buildModel()                        # MF_fastALS.cpp:112-161
    fals.loss()                              # :184-206
    fals.evaluate()                          # evaluate_model, main.cpp:37-65
    fals.evaluate_for_user(u, gtItem, topK)  # :620-662

Multi-GPU (SURVEY.md §8e): every rank holds full replicas of U and V and owns a contiguous,
nnz-balanced user range and item range.  After each half-epoch the updated rows are exchanged
(one broadcast per owner, straight into the replica — the all-gather of variable-size shards) and
the partial K x K Grams are all-reduced.
"""
from __future__ import annotations

import ctypes as C
import os
import sys
import time
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import EalsParams, check


# --------------------------------------------------------------------------------------------------
# SparseMat: the train matrix in both orientations (SparseMat.h:15-42 holds rows[] and cols[]).
# --------------------------------------------------------------------------------------------------
@dataclass
class SparseMat:
    """Dual CSR/CSC container.  Arrays are numpy (host) or torch CUDA tensors (device):
    ``row_ptr`` int64 [M+1], ``col_idx`` int32 [nnz] ascending per row (main.cpp:198-205 order),
    ``col_ptr`` int64 [N+1], ``row_idx`` int32 [nnz] ascending per column; ``row_val``/``col_val``
    fp64 or None (all ratings 1, which is what the reference's loader stores)."""
    M: int
    N: int
    row_ptr: object
    col_idx: object
    col_ptr: object
    row_idx: object
    row_val: object = None
    col_val: object = None

    @property
    def on_device(self) -> bool:
        return not isinstance(self.row_ptr, np.ndarray)

    @property
    def nnz(self) -> int:
        return int(self.row_ptr[-1])

    @staticmethod
    def from_csr(M, N, row_ptr, col_idx, val=None) -> "SparseMat":
        """Build the column orientation from a host CSR (stable sort by column keeps users
        ascending inside a column, as the reference's append order does)."""
        row_ptr = np.ascontiguousarray(row_ptr, np.int64)
        col_idx = np.ascontiguousarray(col_idx, np.int32)
        rows = np.repeat(np.arange(M, dtype=np.int32), np.diff(row_ptr))
        order = np.argsort(col_idx, kind="stable")
        col_ptr = np.zeros(N + 1, np.int64)
        np.cumsum(np.bincount(col_idx, minlength=N), out=col_ptr[1:])
        row_val = col_val = None
        if val is not None:
            row_val = np.ascontiguousarray(val, np.float64)
            col_val = np.ascontiguousarray(row_val[order])
        return SparseMat(M, N, row_ptr, col_idx, col_ptr, np.ascontiguousarray(rows[order]), row_val, col_val)

    @staticmethod
    def from_csr_device(M, N, row_ptr, col_idx) -> "SparseMat":
        """Same, for torch CUDA tensors (all-ones ratings)."""
        from .datasets import csr_to_csc_device
        col_ptr, row_idx, _ = csr_to_csc_device(M, N, row_ptr, col_idx)
        return SparseMat(M, N, row_ptr.contiguous(), col_idx.contiguous(), col_ptr, row_idx)


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    return C.c_void_p(a.data_ptr())          # torch tensor


def partition_by_nnz(ptr, world: int) -> list[int]:
    """Contiguous row ranges with (nearly) equal nonzero counts: bounds[r]..bounds[r+1] is rank r's
    range.  ``ptr`` is the host offsets array of that orientation."""
    ptr = np.asarray(ptr)
    n = len(ptr) - 1
    total = int(ptr[-1])
    bounds = [0]
    for r in range(1, world):
        b = int(np.searchsorted(ptr, total * r / world, side="left"))
        bounds.append(min(max(b, bounds[-1]), n))
    bounds.append(n)
    return bounds


def partition_by_cost(ptr, world: int) -> list[int]:
    """Contiguous row ranges of (nearly) equal COST: the library's per-row cost model (eals_partition — ns per
    row / per nonzero by kernel family, measured on B200).  Balancing nonzeros alone left ranks waiting in the
    Gram all-reduce: a nonzero costs 0.37 ns in the slab pipeline and 0.84 ns in a row of <= 32 nonzeros."""
    ptr = np.ascontiguousarray(ptr, np.int64)
    bounds = np.zeros(world + 1, np.int32)
    check(_lib.load().eals_partition(_ptr(ptr), len(ptr) - 1, world, _ptr(bounds)))
    return [int(b) for b in bounds]


def exchange_rows(full, bounds, rank: int, group=None) -> None:
    """All-gather of variable-size shards: rows bounds[r]:bounds[r+1] of the replicated matrix
    ``full`` (a torch tensor [n][ld], CPU for gloo or CUDA for nccl) are sent from rank r into
    every other replica, in place."""
    import torch.distributed as dist
    world = len(bounds) - 1
    for r in range(world):
        if bounds[r + 1] > bounds[r]:
            src = dist.get_global_rank(group, r) if group is not None else r
            dist.broadcast(full[bounds[r]:bounds[r + 1]], src=src, group=group)


def allreduce_sum(t, group=None) -> None:
    import torch.distributed as dist
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)


def gather_full_array(host, n: int, rank: int, world: int, device, buf=None, group=None):
    """Every rank needs the FULL array ``host[:n]`` (a numpy array every rank holds in host memory) on
    its device.  Rank r copies only the r-th 1/world chunk from the host and an all-gather completes the
    array on every rank (NCCL over NVLink for CUDA tensors; gloo on CPU in the tests): the host-to-device
    bytes of a rank shrink by ``world``.  Returns (tensor of n elements, the padded buffer to reuse)."""
    import torch
    import torch.distributed as dist
    dt = torch.from_numpy(np.empty(0, host.dtype)).dtype
    per = max(1, (n + world - 1) // world)
    if buf is None or buf.numel() < per * world or buf.dtype != dt or str(buf.device) != str(torch.device(device)):
        buf = torch.empty(per * world, dtype=dt, device=device)
    full = buf[:per * world]
    lo, hi = min(rank * per, n), min((rank + 1) * per, n)
    chunk = full[rank * per:(rank + 1) * per]
    if hi > lo:
        chunk[:hi - lo].copy_(torch.from_numpy(np.ascontiguousarray(host[lo:hi])), non_blocking=True)
    dist.all_gather_into_tensor(full, chunk, group=group)
    return full[:max(n, 1)], buf


def insert_interaction(sm: "SparseMat", u: int, i: int):
    """The host arrays of ``sm`` with the entry (u, i), rating 1, added at its sorted position in both
    orientations (what ``trainMatrix.setValue(u, i, 1)`` / ``W.setValue(u, i, w_new)`` of
    MF_fastALS.cpp:224-226 mean).  An entry that is already there has its rating (= weight) overwritten
    with 1, as setValue does; None if nothing changes (entry present with rating 1)."""
    rp, ci, cp, ri, rv, cv = sm.row_ptr, sm.col_idx, sm.col_ptr, sm.row_idx, sm.row_val, sm.col_val
    a, b = int(rp[u]), int(rp[u + 1])
    k = a + int(np.searchsorted(ci[a:b], i))
    a2, b2 = int(cp[i]), int(cp[i + 1])
    k2 = a2 + int(np.searchsorted(ri[a2:b2], u))
    if k < b and ci[k] == i:
        if rv is None or rv[k] == 1.0:
            return None
        rv, cv = rv.copy(), cv.copy()
        rv[k] = 1.0
        cv[k2] = 1.0
        return SparseMat(sm.M, sm.N, rp, ci, cp, ri, rv, cv)
    ci = np.insert(ci, k, np.int32(i)); ri = np.insert(ri, k2, np.int32(u))
    rp = rp.copy(); rp[u + 1:] += 1
    cp = cp.copy(); cp[i + 1:] += 1
    if rv is not None:
        rv = np.insert(rv, k, 1.0); cv = np.insert(cv, k2, 1.0)
    return SparseMat(sm.M, sm.N, rp, ci, cp, ri, rv, cv)


def _recommend_call(fn, handle, users, k, exclude_seen):
    """One eals_recommend / eals_group_recommend call.  ``users``: a sequence, a numpy array or a torch tensor
    (a CUDA tensor stays on the device: inputs and outputs then live there).  Returns torch tensors for a CUDA
    input, numpy arrays otherwise."""
    k = int(k)
    if not isinstance(users, np.ndarray) and hasattr(users, "is_cuda") and users.is_cuda:
        import torch
        u = users.to(torch.int32).contiguous()
        n = u.numel()
        items = torch.empty((n, k), dtype=torch.int32, device=u.device)
        scores = torch.empty((n, k), dtype=torch.float64, device=u.device)
        torch.cuda.current_stream(u.device).synchronize()
        check(fn(handle, _lib.EALS_DEVICE, n, _ptr(u), k, int(bool(exclude_seen)), _ptr(items), _ptr(scores)))
        return items, scores
    u = np.ascontiguousarray(users.cpu().numpy() if hasattr(users, "cpu") else users, np.int32).reshape(-1)
    items = np.empty((u.size, k), np.int32)
    scores = np.empty((u.size, k), np.float64)
    check(fn(handle, _lib.EALS_HOST, u.size, _ptr(u), k, int(bool(exclude_seen)), _ptr(items), _ptr(scores)))
    return items, scores


def _first_block(users, items, us, factors):
    """The first filtered item block's shape, device time and tensor rate (factors padded to 64 in fp16)."""
    kp = -(-factors // 64) * 64
    return {"users": int(users), "items": int(items), "ms": us / 1e3,
            "tflops": 2.0 * users * items * kp / (us * 1e-6) / 1e12}


def _recommend_stats(lib, h, factors):
    out = np.zeros(7, np.int64)
    check(lib.eals_recommend_stats(h, _ptr(out)))
    st = {"engine": "tcgen05" if out[0] == 1 else "fp64", "seed_items": int(out[1]), "pairs_rescored": int(out[2]),
          "users_left_after_first_block": int(out[3])}
    if out[6] > 0:
        st["first_block"] = _first_block(out[4], out[5], out[6], factors)
    return st


def _is_cuda(a) -> bool:
    return a is not None and not isinstance(a, np.ndarray) and getattr(a, "is_cuda", False)


def _same_space(arrays, device):
    """The arrays of one fold_in / recommend_vectors call in ONE memory space: torch tensors on ``device`` when any of
    them is a CUDA tensor, numpy arrays otherwise (None stays None).  ``arrays``: (array, numpy dtype) pairs.  An empty
    array becomes a one-element one, so that the library never sees a null pointer for a present argument."""
    on_dev = any(_is_cuda(a) for a, _ in arrays)
    out = []
    for a, dt in arrays:
        if a is None:
            out.append(None)
            continue
        if on_dev:
            import torch
            t = torch.as_tensor(a, device=device).to(torch.from_numpy(np.empty(0, dt)).dtype).contiguous()
            out.append(t if t.numel() else torch.zeros(1, dtype=t.dtype, device=device))
        else:
            h = a.cpu().numpy() if hasattr(a, "cpu") else a
            h = np.ascontiguousarray(h, dt)
            out.append(h if h.size else np.zeros(1, dt))
    if on_dev:
        import torch
        torch.cuda.current_stream(torch.device(device)).synchronize()
    return (_lib.EALS_DEVICE if on_dev else _lib.EALS_HOST), out


def _rows(a) -> int:
    return int(a.shape[0])


def _fold_in_call(fn, handle, factors, device, histories, init, n_iter):
    """One eals_fold_in / eals_group_fold_in call; returns float64 [n, factors] on the host."""
    n = _rows(histories.row_ptr) - 1
    if init is not None and tuple(init.shape) != (n, factors):
        raise ValueError(f"init must be [{n}, {factors}], got {tuple(init.shape)}")
    space, (rp, ci, rv, ini) = _same_space([(histories.row_ptr, np.int64), (histories.col_idx, np.int32),
                                            (histories.row_val, np.float64), (init, np.float64)], device)
    if space == _lib.EALS_DEVICE:
        import torch
        out = torch.empty((max(n, 1), factors), dtype=torch.float64, device=device)
    else:
        out = np.empty((max(n, 1), factors), np.float64)
    check(fn(handle, space, n, _ptr(rp), _ptr(ci), _ptr(rv), _ptr(ini), int(n_iter), _ptr(out)))
    out = out[:n]
    return out if isinstance(out, np.ndarray) else out.cpu().numpy()


def _recommend_vectors_call(fn, handle, factors, device, Q, k, exclude):
    """One eals_recommend_vectors / eals_group_recommend_vectors call; returns (items, scores) on the host."""
    k = int(k)
    if not hasattr(Q, "shape"):
        Q = np.asarray(Q, np.float64)
    n = _rows(Q)
    if len(Q.shape) != 2 or Q.shape[1] != factors:
        raise ValueError(f"Q must be [n, {factors}], got {tuple(Q.shape)}")
    if exclude is not None and _rows(exclude.row_ptr) - 1 != n:
        raise ValueError(f"exclude must have one row per query ({n}), got {_rows(exclude.row_ptr) - 1}")
    ex = (None, None) if exclude is None else (exclude.row_ptr, exclude.col_idx)
    space, (q, ep, ei) = _same_space([(Q, np.float64), (ex[0], np.int64), (ex[1], np.int32)], device)
    shape = (max(n, 1), max(k, 1))
    if space == _lib.EALS_DEVICE:
        import torch
        items = torch.empty(shape, dtype=torch.int32, device=device)
        scores = torch.empty(shape, dtype=torch.float64, device=device)
    else:
        items, scores = np.empty(shape, np.int32), np.empty(shape, np.float64)
    check(fn(handle, space, n, _ptr(q), _ptr(ep), _ptr(ei), k, _ptr(items), _ptr(scores)))
    items, scores = items[:n], scores[:n]
    return (items, scores) if isinstance(items, np.ndarray) else (items.cpu().numpy(), scores.cpu().numpy())


def _similar_call(fn, handle, which, device, ids, k):
    """One eals_similar / eals_group_similar call over the catalogue ``which`` (_lib.BUF_V items, _lib.BUF_U users);
    ``ids``: a sequence, a numpy array or a torch tensor (a CUDA tensor is read on the device).  Returns (ids, scores)
    on the host."""
    k = int(k)
    if not hasattr(ids, "shape"):
        ids = np.asarray(ids, np.int32)
    ids = ids.reshape(-1)
    n = _rows(ids)
    space, (q,) = _same_space([(ids, np.int32)], device)
    shape = (max(n, 1), max(k, 1))
    if space == _lib.EALS_DEVICE:
        import torch
        out_i = torch.empty(shape, dtype=torch.int32, device=device)
        out_s = torch.empty(shape, dtype=torch.float64, device=device)
    else:
        out_i, out_s = np.empty(shape, np.int32), np.empty(shape, np.float64)
    check(fn(handle, which, space, n, _ptr(q), k, _ptr(out_i), _ptr(out_s)))
    out_i, out_s = out_i[:n], out_s[:n]
    return (out_i, out_s) if isinstance(out_i, np.ndarray) else (out_i.cpu().numpy(), out_s.cpu().numpy())


RANKING_METRICS = ("hit_rate", "precision", "recall", "ndcg", "map", "mrr")


def _ranking_metrics_call(fn, handle, device, test, n_users, k, exclude_seen, rows, per_user, ranks):
    """One eals_ranking_metrics / eals_group_ranking_metrics call over ``rows`` = (first, end) user rows of ``test``
    (the rows the call reads).  Returns (sums or means [6], users with test items, per-user [end - first, 6] or None,
    ranks of the rows' test entries or None), the arrays on the host."""
    if _rows(test.row_ptr) - 1 != n_users:
        raise _lib.EalsError(_lib.ERR_ARG, f"the test matrix must have one row per user ({n_users}), got "
                                           f"{_rows(test.row_ptr) - 1}")
    space, (rp, ci) = _same_space([(test.row_ptr, np.int64), (test.col_idx, np.int32)], device)
    first, end = rows
    n_rows, n_ent = end - first, int(rp[end]) - int(rp[first])
    if space == _lib.EALS_DEVICE:
        import torch
        pu = torch.zeros((max(n_rows, 1), 6), dtype=torch.float64, device=device) if per_user else None
        rk = torch.full((max(n_ent, 1),), -1, dtype=torch.int32, device=device) if ranks else None
    else:
        pu = np.zeros((max(n_rows, 1), 6)) if per_user else None
        rk = np.full(max(n_ent, 1), -1, np.int32) if ranks else None
    sums, users = np.zeros(6), C.c_int64()
    check(fn(handle, space, _ptr(rp), _ptr(ci), int(k), int(bool(exclude_seen)), _ptr(sums), C.byref(users), _ptr(pu), _ptr(rk)))
    host = lambda a: None if a is None else (a if isinstance(a, np.ndarray) else a.cpu().numpy())
    pu, rk = host(pu), host(rk)
    return sums, int(users.value), None if pu is None else pu[:n_rows], None if rk is None else rk[:n_ent]


def _ranking_result(means, users, per_user, ranks):
    out = dict(zip(RANKING_METRICS, (float(x) for x in means)))
    out["users"] = int(users)
    if per_user is not None:
        out["per_user"] = per_user
    if ranks is not None:
        out["ranks"] = ranks
    return out


class _DevArray:
    """Expose a raw device pointer to torch through __cuda_array_interface__."""

    def __init__(self, ptr: int, shape, typestr="<f8"):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr,
                                         "data": (int(ptr), False), "version": 2}


class MF_fastALS:
    def __init__(self, trainMatrix: SparseMat, testRatings, topK=10, threadNum=1, factors=64,
                 maxIter=20, w0=10.0, alpha=0.75, reg=0.01, init_mean=0.0, init_stdev=0.01,
                 showProgress=False, showLoss=True, userCount=None, itemCount=None, *,
                 device=None, distributed=None, init=True, debug_sync=False, out=None):
        self.lib = _lib.load()
        self.trainMatrix = trainMatrix
        self.userCount = int(userCount if userCount is not None else trainMatrix.M)
        self.itemCount = int(itemCount if itemCount is not None else trainMatrix.N)
        if self.userCount != trainMatrix.M or self.itemCount != trainMatrix.N:
            raise ValueError("userCount/itemCount do not match the train matrix")
        self.topK, self.factors, self.maxIter = int(topK), int(factors), int(maxIter)
        self.w0, self.alpha, self.reg = float(w0), float(alpha), float(reg)
        self.init_mean, self.init_stdev = float(init_mean), float(init_stdev)
        self.showprogress, self.showloss = bool(showProgress), bool(showLoss)
        del threadNum                                   # dead in the reference too (MF_fastALS.cpp:30)
        self.out = out or sys.stdout
        self.testItems = None if testRatings is None else self._test_items(testRatings)

        # distributed context: one process per GPU
        self.rank, self.world, self.group = 0, 1, None
        if distributed is None:
            try:
                import torch.distributed as dist
                distributed = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
            except ImportError:
                distributed = False
        if distributed:
            import torch.distributed as dist
            self.rank, self.world = dist.get_rank(), dist.get_world_size()
        if device is None:
            import torch
            device = torch.cuda.current_device() if torch.cuda.is_available() else 0
        self.device = int(device)

        sm = trainMatrix
        if self.world > 1:
            rp = sm.row_ptr if isinstance(sm.row_ptr, np.ndarray) else sm.row_ptr.cpu().numpy()
            cp = sm.col_ptr if isinstance(sm.col_ptr, np.ndarray) else sm.col_ptr.cpu().numpy()
            part = partition_by_nnz if os.environ.get("EALS_PARTITION") == "nnz" else partition_by_cost
            self.user_bounds = part(rp, self.world)
            self.item_bounds = part(cp, self.world)
        else:
            self.user_bounds, self.item_bounds = [0, sm.M], [0, sm.N]

        p = EalsParams()
        self.lib.eals_default_params(C.byref(p))
        p.n_users, p.n_items, p.factors, p.topk = sm.M, sm.N, self.factors, self.topK
        p.w0, p.alpha, p.reg = self.w0, self.alpha, self.reg
        p.init_mean, p.init_stdev = self.init_mean, self.init_stdev
        p.device = self.device
        p.input_space = _lib.EALS_DEVICE if sm.on_device else _lib.EALS_HOST
        p.user_begin, p.user_end = self.user_bounds[self.rank], self.user_bounds[self.rank + 1]
        p.item_begin, p.item_end = self.item_bounds[self.rank], self.item_bounds[self.rank + 1]
        p.flags = _lib.FLAG_SYNC_EACH_CALL if debug_sync else 0
        if 1 < self.world <= 8:                           # lets the prediction caches span the ranks
            p.n_ranks, p.rank = self.world, self.rank
            for r in range(self.world + 1):
                p.user_bounds[r], p.item_bounds[r] = self.user_bounds[r], self.item_bounds[r]
        if self.world > 1 and (p.user_end == p.user_begin or p.item_end == p.item_begin):
            raise ValueError("more ranks than rows: a rank would own an empty range")
        self._params = p
        h = C.c_void_p()
        check(self.lib.eals_create(C.byref(p), _ptr(sm.row_ptr), _ptr(sm.col_idx), _ptr(sm.row_val),
                                   _ptr(sm.col_ptr), _ptr(sm.row_idx), _ptr(sm.col_val), C.byref(h)))
        self.h = h
        self.ld = self.lib.eals_leading_dim(self.h)
        # order the library's kernels with torch's (NCCL calls, CUDA events): share torch's current stream
        import torch
        with torch.cuda.device(self.device):
            check(self.lib.eals_set_stream(self.h, C.c_void_p(torch.cuda.current_stream().cuda_stream), 0))
        self.peer_store = self.peer_pred_cache = False
        if self.world > 1 and os.environ.get("EALS_PEER_STORE", "1") != "0":
            self._attach_peers()
        if init:
            check(self.lib.eals_init_factors(self.h))     # MF_fastALS.cpp:85-90
            self._replicas_written()

    # ---- helpers ---------------------------------------------------------------------------------
    def _attach_peers(self, factors=True):
        """Exchange CUDA IPC handles and map the other ranks' buffers: the U and V replicas (the sweep
        kernels then store finished rows into every replica themselves — the all-gather of SURVEY.md §8e
        fused into the sweep) and the prediction caches.  Needs all ranks on one box with peer access.
        ``factors=False`` (after setTrain): only the prediction caches, the replicas never move."""
        import torch
        import torch.distributed as dist
        if self.world - 1 > 7:
            return
        dev = f"cuda:{self.device}"
        shared = [_lib.BUF_U, _lib.BUF_V] if factors else []
        # The prediction caches are shared across ranks too: a sweep stages its final predictions locally in
        # destination order and peer-to-peer copies move each destination's segment into that rank's receive area.
        pc = os.environ.get("EALS_PEER_PRED_CACHE", "1") == "1" and self._pred_cache_everywhere()
        if pc:
            shared += [_lib.BUF_PC_USER, _lib.BUF_PC_ITEM]
        self.peer_pred_cache = pc
        if not shared:
            return
        # one all-gather for all handles
        mine = np.zeros((len(shared), 64), np.uint8)
        for k, which in enumerate(shared):
            check(self.lib.eals_ipc_handle(self.h, which, _ptr(mine[k])))
        t = torch.from_numpy(mine).to(dev)
        allh = [torch.empty_like(t) for _ in range(self.world)]
        dist.all_gather(allh, t, group=self.group)
        allh = [a.cpu().numpy() for a in allh]
        for k, which in enumerate(shared):
            others = np.ascontiguousarray(np.concatenate([allh[r][k] for r in range(self.world) if r != self.rank]), np.uint8)
            check(self.lib.eals_ipc_attach(self.h, which, self.world - 1, _ptr(others)))
        self.peer_store = True

    def _replicas_written(self):
        """Every whole-replica overwrite (factor init, setUV, checkpoint load) ends here when the sweep
        kernels of OTHER ranks store into this rank's replica: no rank may start a sweep — and peer-store
        finished rows into a replica — before every rank has finished writing its own copy, or a slower
        rank's upload lands on top of rows a faster rank already updated (silently stale factors; the
        1-in-5 deviating 8-GPU run of round 1, DESIGN.md §6)."""
        if self.world > 1:
            import torch.distributed as dist
            self.sync()
            dist.barrier(group=self.group)

    def _device_matrix(self, sm: SparseMat) -> SparseMat:
        """Several ranks, matrix in host memory: every rank needs the FULL index arrays on its GPU (its
        row and column slices, and both orientations for the position maps of the prediction caches).
        Instead of every rank pushing the whole matrix through its own PCIe link, rank r uploads the r-th
        1/world chunk and an NCCL all-gather over NVLink completes the arrays everywhere: the
        host-to-device bytes of a rank shrink by world (measured before, c4: setTrain 0.5 s at 2 ranks,
        2.1 s at 8).  The device buffers are kept for the next setTrain."""
        import torch
        dev = f"cuda:{self.device}"
        W, r = self.world, self.rank
        nnz = int(sm.row_ptr[-1])
        kinds = [("ci", sm.col_idx), ("ri", sm.row_idx)]
        if sm.row_val is not None:
            kinds += [("rv", sm.row_val), ("cv", sm.col_val)]
        bufs = self.__dict__.setdefault("_full_bufs", {})
        out = {}
        for name, host in kinds:
            out[name], bufs[name] = gather_full_array(host, nnz, r, W, dev, bufs.get(name), self.group)
        rp = torch.from_numpy(np.ascontiguousarray(sm.row_ptr, np.int64)).to(dev)
        cp = torch.from_numpy(np.ascontiguousarray(sm.col_ptr, np.int64)).to(dev)
        per = max(1, (nnz + W - 1) // W)
        self._h2d_bytes_last = sum(min(per, max(0, nnz - r * per)) * host.dtype.itemsize for _, host in kinds) \
            + 8 * (sm.M + 1 + sm.N + 1)
        return SparseMat(sm.M, sm.N, rp, out["ci"], cp, out["ri"], out.get("rv"), out.get("cv"))

    def _pred_cache_everywhere(self) -> bool:
        """True when every rank built its prediction caches (they are skipped e.g. for >= 2^32 nonzeros)."""
        import torch
        import torch.distributed as dist
        ptr, nbytes = C.c_void_p(), C.c_int64()
        check(self.lib.eals_device_buffer(self.h, _lib.BUF_PC_USER, C.byref(ptr), C.byref(nbytes)))
        ok = torch.tensor([1 if (ptr.value and nbytes.value > 0) else 0], device=f"cuda:{self.device}")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)
        return bool(ok.item())

    def _test_items(self, testRatings):
        a = np.asarray(testRatings)
        if a.ndim == 2:                                  # rows of (userId, itemId, ...) like Rating.h
            items = np.empty(self.userCount, np.int32)
            items[a[:, 0].astype(np.int64)] = a[:, 1].astype(np.int32)
            return items
        return np.ascontiguousarray(a, np.int32)

    def close(self):
        if getattr(self, "h", None):
            self.lib.eals_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def device_tensor(self, which):
        """torch view (no copy) of one of the model's device buffers, padded leading dimension."""
        import torch
        ptr, nbytes = C.c_void_p(), C.c_int64()
        check(self.lib.eals_device_buffer(self.h, which, C.byref(ptr), C.byref(nbytes)))
        if which in (_lib.BUF_WI, _lib.BUF_LOSS_TERMS):
            shape = (nbytes.value // 8,)
        else:
            shape = (nbytes.value // 8 // self.ld, self.ld)
        return torch.as_tensor(_DevArray(ptr.value, shape), device=f"cuda:{self.device}")

    def sync(self):
        check(self.lib.eals_sync(self.h))

    def factor_hash(self):
        """(hash(U), hash(V)) of this rank's replicas, computed on the device."""
        out = np.zeros(2, np.uint64)
        check(self.lib.eals_factor_hash(self.h, _ptr(out)))
        return int(out[0]), int(out[1])

    def replicas_consistent(self) -> bool:
        """True when the U and V replicas of ALL ranks are bit-identical (trivially true on one rank)."""
        if self.world == 1:
            return True
        import torch
        import torch.distributed as dist
        hu, hv = self.factor_hash()
        # two int64 words per hash halves (all_reduce MIN/MAX on signed ints: compare 32-bit pieces)
        parts = [hu & 0xffffffff, hu >> 32, hv & 0xffffffff, hv >> 32]
        lo = torch.tensor(parts, dtype=torch.int64, device=f"cuda:{self.device}")
        hi = lo.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=self.group)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=self.group)
        return bool(torch.equal(lo, hi))

    def _check_replicas(self, what):
        if self.world > 1 and os.environ.get("EALS_CHECK_REPLICAS") == "1":
            self._half_epochs = getattr(self, "_half_epochs", 0) + 1
            if not self.replicas_consistent():
                raise RuntimeError(f"rank {self.rank}: replicas diverged after half-epoch {self._half_epochs} ({what})")

    # ---- public members of the reference (MF_fastALS.h:31-46) as host copies ------------------------
    def _get_factors(self, want_u, want_v):
        U = np.empty((self.userCount, self.factors)) if want_u else None
        V = np.empty((self.itemCount, self.factors)) if want_v else None
        check(self.lib.eals_get_factors(self.h, _lib.EALS_HOST, _ptr(U), _ptr(V)))
        return U, V

    @property
    def U(self):
        return self._get_factors(True, False)[0]

    @property
    def V(self):
        return self._get_factors(False, True)[1]

    def _get_S(self, su, sv):
        SU = np.empty((self.factors, self.factors)) if su else None
        SV = np.empty((self.factors, self.factors)) if sv else None
        check(self.lib.eals_get_S(self.h, _lib.EALS_HOST, _ptr(SU), _ptr(SV)))
        return SU, SV

    @property
    def SU(self):
        return self._get_S(True, False)[0]

    @property
    def SV(self):
        return self._get_S(False, True)[1]

    @property
    def Wi(self):
        w = np.empty(self.itemCount)
        check(self.lib.eals_get_item_weights(self.h, _lib.EALS_HOST, _ptr(w)))
        return w

    @Wi.setter
    def Wi(self, w):
        w = np.ascontiguousarray(w, np.float64)
        check(self.lib.eals_set_item_weights(self.h, _lib.EALS_HOST, _ptr(w)))

    # ---- setters (MF_fastALS.cpp:94-110) -------------------------------------------------------------
    def setUV(self, U, V):
        if isinstance(U, np.ndarray) or U is None and isinstance(V, np.ndarray):
            U = None if U is None else np.ascontiguousarray(U, np.float64)
            V = None if V is None else np.ascontiguousarray(V, np.float64)
            space = _lib.EALS_HOST
        else:
            space = _lib.EALS_DEVICE
        if self.world > 1:       # no peer may still be storing rows of an unfinished sweep into this replica
            import torch.distributed as dist
            self.sync()
            dist.barrier(group=self.group)
        check(self.lib.eals_set_factors(self.h, space, _ptr(U), _ptr(V)))
        self._replicas_written()

    # ---- factor checkpoint (SURVEY.md §8 f4) ---------------------------------------------------------
    def save(self, path):
        """U, V and Wi to a binary file (format: include/eals_b200.h, eals_save_factors).  Every rank holds
        complete replicas, so with several ranks only rank 0 writes."""
        if self.rank == 0:
            check(self.lib.eals_save_factors(self.h, os.fsencode(path)))
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier(group=self.group)

    def load(self, path):
        """Replace U, V, Wi by a checkpoint written by ``save`` (same shape and K) and rebuild the S caches;
        buildModel / update_user / update_item then resume from that state."""
        if self.world > 1:
            import torch.distributed as dist
            self.sync()
            dist.barrier(group=self.group)
        check(self.lib.eals_load_factors(self.h, os.fsencode(path)))
        self._replicas_written()

    def refresh_S(self):
        """initS (MF_fastALS.cpp:583-595): rebuild both S caches from the current factors."""
        check(self.lib.eals_refresh_S(self.h))

    def setTrain(self, trainMatrix: SparseMat):
        import time as _t
        verbose = os.environ.get("EALS_VERBOSE") == "1"
        tg = _t.perf_counter()
        sm = trainMatrix
        if self.world > 1 and not sm.on_device and os.environ.get("EALS_GATHER_UPLOAD", "1") == "1":
            sm = self._device_matrix(sm)
            if verbose:
                self.sync()
                print(f"[eals] rank {self.rank} setTrain: chunk upload + all-gather {1e3 * (_t.perf_counter() - tg):.1f} ms", file=sys.stderr)
        space = _lib.EALS_DEVICE if sm.on_device else _lib.EALS_HOST
        t0 = _t.perf_counter()
        gen = self.lib.eals_ipc_generation(self.h)
        check(self.lib.eals_set_train(self.h, space, _ptr(sm.row_ptr), _ptr(sm.col_idx), _ptr(sm.row_val),
                                      _ptr(sm.col_ptr), _ptr(sm.row_idx), _ptr(sm.col_val)))
        self.trainMatrix = trainMatrix
        t1 = _t.perf_counter()
        if self.peer_store and self.peer_pred_cache:
            # the caches only move when one had to grow: then every rank exchanges handles again
            import torch
            import torch.distributed as dist
            moved = torch.tensor([int(self.lib.eals_ipc_generation(self.h) != gen)], device=f"cuda:{self.device}")
            dist.all_reduce(moved, op=dist.ReduceOp.MAX, group=self.group)
            if int(moved.item()):
                self._attach_peers(factors=False)
                dist.barrier(group=self.group)
                check(self.lib.eals_ipc_gc(self.h))
        if verbose:
            print(f"[eals] rank {self.rank} setTrain: library {1e3 * (t1 - t0):.1f} ms, attach {1e3 * (_t.perf_counter() - t1):.1f} ms",
                  file=sys.stderr)

    # ---- half-epochs ---------------------------------------------------------------------------------
    def update_user(self):
        """User sweep + SU refresh (MF_fastALS.cpp:127-132)."""
        check(self.lib.eals_sweep_users(self.h))
        if self.world > 1 and not self.peer_store:
            exchange_rows(self.device_tensor(_lib.BUF_U), self.user_bounds, self.rank, self.group)
        check(self.lib.eals_gram_users(self.h))
        if self.world > 1:
            allreduce_sum(self.device_tensor(_lib.BUF_SU), self.group)
            self._check_replicas("update_user")

    def update_item(self):
        """Item sweep + SV refresh (MF_fastALS.cpp:146-152)."""
        check(self.lib.eals_sweep_items(self.h))
        if self.world > 1 and not self.peer_store:
            exchange_rows(self.device_tensor(_lib.BUF_V), self.item_bounds, self.rank, self.group)
        check(self.lib.eals_gram_items(self.h))
        if self.world > 1:
            allreduce_sum(self.device_tensor(_lib.BUF_SV), self.group)
            self._check_replicas("update_item")

    def run_epochs(self, n, graph=True):
        """n epochs; with ``graph`` (single rank) one captured epoch is replayed as a CUDA graph — the launch-bound
        small configurations gain most.  Same results as n x (update_user, update_item)."""
        if self.world > 1:
            for _ in range(int(n)):
                self.update_user(); self.update_item()
            return
        check(self.lib.eals_run_epochs(self.h, int(n), int(bool(graph))))

    def update_user_thread(self, u):
        check(self.lib.eals_update_user_row(self.h, int(u)))

    def update_item_thread(self, i):
        check(self.lib.eals_update_item_row(self.h, int(i)))

    def update_user_SU(self, oldVector, uget):
        o, n = np.ascontiguousarray(oldVector, np.float64), np.ascontiguousarray(uget, np.float64)
        check(self.lib.eals_patch_SU(self.h, _ptr(o), _ptr(n)))

    def update_item_SV(self, i, oldVector, vget):
        o, n = np.ascontiguousarray(oldVector, np.float64), np.ascontiguousarray(vget, np.float64)
        check(self.lib.eals_patch_SV(self.h, int(i), _ptr(o), _ptr(n)))

    def _factor_row(self, which, r):
        """One row of U or V as a host vector (U.matrix[u] / V.matrix[i] of the reference)."""
        out = np.empty(self.factors)
        check(self.lib.eals_get_factor_row(self.h, which, int(r), _ptr(out)))
        return out

    def updateModel(self, u, i, patch_S=True, maxIterOnline=10):
        """Online update (MF_fastALS.cpp:223-242): add the interaction (u, i) with rating 1 = ``w_new``,
        give a brand-new item the weight w0 / itemCount (and its term in SV), then run 10 alternating
        single-row updates of user u and item i.

        The reference's version appends past the capacity of its SparseVec arrays and leaves SU / SV
        stale between the single-row updates (SURVEY.md §9); here the matrix is rebuilt with the entry
        at its sorted position and, with ``patch_S`` (default), the S caches follow every row update
        (update_user_SU / update_item_SV, MF_fastALS.cpp:324-335, 409-422) as in the paper's incremental
        mode.  ``patch_S=False`` reproduces the reference's arithmetic (stale caches)."""
        if self.world > 1 and not (self.peer_store and patch_S):
            raise NotImplementedError("updateModel on several ranks needs the peer-store exchange and patch_S=True")
        u, i = int(u), int(i)
        if not (0 <= u < self.userCount and 0 <= i < self.itemCount):
            raise IndexError("updateModel: (u, i) outside the matrix")
        sm = self.trainMatrix
        host = lambda a: None if a is None else (a if isinstance(a, np.ndarray) else a.cpu().numpy())
        sm = SparseMat(sm.M, sm.N, host(sm.row_ptr), host(sm.col_idx), host(sm.col_ptr), host(sm.row_idx),
                       host(sm.row_val), host(sm.col_val))
        grown = insert_interaction(sm, u, i)              # trainMatrix.setValue(u, i, 1); W.setValue(u, i, w_new)
        if grown is not None:
            self.setTrain(grown)                            # every rank: same matrix, same (unchanged) ranges
        Wi = self.Wi
        if Wi[i] == 0.0:                                    # a new item: weight and its term in the SV cache
            Wi[i] = self.w0 / self.itemCount
            self.Wi = Wi                                    # uploads and rebuilds SV with the new weight
        # Several ranks: the OWNER of the row runs the single-row kernel, which stores the new row into every
        # replica over NVLink; after a barrier every rank reads the row from its own replica and patches its S
        # caches.  The "old" row of a patch must be read BEFORE the owner's kernel can store into this replica: it is
        # read once up front (barrier), and afterwards the row a rank read after step n is the old row of step n+1 —
        # the owner's next store to it comes only after a barrier this rank joins after that read.  (Reading it at
        # the top of every step raced with a faster owner: a zero patch on the slow rank, S caches apart.)
        own_u = self.user_bounds[self.rank] <= u < self.user_bounds[self.rank + 1]
        own_i = self.item_bounds[self.rank] <= i < self.item_bounds[self.rank + 1]
        old_u = self._factor_row(_lib.BUF_U, u) if patch_S else None
        old_v = self._factor_row(_lib.BUF_V, i) if patch_S else None
        self._rank_barrier()
        for _ in range(int(maxIterOnline)):
            if own_u:
                self.update_user_thread(u)
            self._rank_barrier()
            if patch_S:
                new = self._factor_row(_lib.BUF_U, u)
                self.update_user_SU(old_u, new)
                old_u = new
            if own_i:
                self.update_item_thread(i)
            self._rank_barrier()
            if patch_S:
                new = self._factor_row(_lib.BUF_V, i)
                self.update_item_SV(i, old_v, new)
                old_v = new

    def barrier(self):
        """Several processes: call on EVERY rank between raw host reads of a replica (``U``, ``V``, ``predict``,
        ``_factor_row``) and the next sweep.  Those reads are local and not ordered against the other ranks: a rank
        that is ahead starts its next sweep and stores finished rows into this replica while a slower rank is still
        copying it out.  ``loss``, ``evaluate``, ``replicas_consistent``, ``setUV``, ``load`` and ``updateModel``
        end in a collective and need nothing extra.  No-op on one rank."""
        self._rank_barrier()

    def _rank_barrier(self):
        """Several processes: this rank's queued work is complete (its peer stores included) and every rank is here."""
        if self.world > 1:
            import torch.distributed as dist
            self.sync()
            dist.barrier(group=self.group)

    def runOneIteration(self):
        """One correct epoch (the reference's version leaves the S caches stale: :163-173)."""
        self.update_user()
        self.update_item()

    # ---- loss / predict --------------------------------------------------------------------------------
    def loss(self) -> float:
        terms = np.zeros(4)
        check(self.lib.eals_loss_terms(self.h, _ptr(terms)))
        if self.world > 1:
            import torch
            t = torch.from_numpy(terms[:3].copy()).to(f"cuda:{self.device}")
            allreduce_sum(t, self.group)
            terms[:3] = t.cpu().numpy()
        return float(self.reg * (terms[1] + terms[2]) + terms[0] + terms[3])

    def predict(self, u, i) -> float:
        s = C.c_double()
        check(self.lib.eals_predict(self.h, int(u), int(i), C.byref(s)))
        return s.value

    def showLoss(self, it, t, loss_pre):
        t0 = time.perf_counter()
        cur = self.loss()
        sym = "-" if loss_pre >= cur else "+"
        if self.rank == 0:
            print(f"Iter={it} {t:g} {sym} loss:{cur:g} {time.perf_counter() - t0:g}", file=self.out)
        return cur

    def buildModel(self):
        """maxIter x (user half-epoch, item half-epoch, optional loss) — MF_fastALS.cpp:112-161,
        with the reference's three stdout lines per iteration."""
        loss_pre = float("inf")
        self.losses = []
        for it in range(self.maxIter):
            t0 = time.perf_counter()
            self.update_user()
            self.sync()
            t_user = time.perf_counter() - t0
            if self.rank == 0:
                print(f"Time of user_update: {t_user:g}", file=self.out)
            t0 = time.perf_counter()
            self.update_item()
            self.sync()
            t_item = time.perf_counter() - t0
            if self.rank == 0:
                print(f"Time of item_update: {t_item:g}", file=self.out)
            if self.showloss:
                loss_pre = self.showLoss(it, t_user + t_item, loss_pre)
                self.losses.append(loss_pre)

    # ---- evaluation --------------------------------------------------------------------------------------
    def evaluate_for_user(self, u, gtItem, topK=None, exact=False):
        out = np.zeros(3)
        check(self.lib.eals_evaluate_user(self.h, int(u), int(gtItem), int(topK or self.topK),
                                          _lib.EVAL_EXACT if exact else _lib.EVAL_REFERENCE, _ptr(out)))
        return [float(x) for x in out]

    def evaluate(self, testRatings=None, topK=None, exact=False, per_user=False):
        """evaluate_model (main.cpp:37-65): mean HR, NDCG and reciprocal rank over ALL users.
        ``exact=False`` reproduces the reference's int-truncating ranking bug for bug."""
        items = self.testItems if testRatings is None else self._test_items(testRatings)
        topK = int(topK or self.topK)
        n_own = self.user_bounds[self.rank + 1] - self.user_bounds[self.rank]
        sums = np.zeros(3)
        hr = ndcg = prec = cnt = None
        if per_user:
            hr, ndcg, prec = np.zeros(n_own), np.zeros(n_own), np.zeros(n_own)
            cnt = np.zeros(n_own, np.int32)
        check(self.lib.eals_evaluate(self.h, _ptr(items), topK,
                                     _lib.EVAL_EXACT if exact else _lib.EVAL_REFERENCE, _ptr(sums),
                                     _ptr(hr), _ptr(ndcg), _ptr(prec), _ptr(cnt)))
        if self.world > 1:
            import torch
            t = torch.from_numpy(sums.copy()).to(f"cuda:{self.device}")
            allreduce_sum(t, self.group)
            sums = t.cpu().numpy()
        res = sums / self.userCount
        if per_user:
            return res, hr, ndcg, prec, cnt
        return res

    def init_factors(self):
        """U.init / V.init / initS again (MF_fastALS.cpp:85-90); returns the host seconds of the stream generation."""
        check(self.lib.eals_init_factors(self.h))
        self._replicas_written()
        v = C.c_double()
        check(self.lib.eals_init_seconds(self.h, C.byref(v)))
        return v.value

    def eval_stats(self):
        """Engine of the last evaluate() or ranking_metrics(): 'tcgen05' (fp16 tensor-core filter + exact fp64 re-score
        of the close calls) or 'fp64' (exact engine), the number of candidates (users, or test entries) and of
        re-scored pairs, and the first filtered item block's shape, time and tensor rate."""
        out = np.zeros(6, np.int64)
        check(self.lib.eals_eval_stats(self.h, _ptr(out)))
        st = {"engine": "tcgen05" if out[0] == 1 else "fp64", "candidates": int(out[1]), "pairs_rescored": int(out[2])}
        if out[5] > 0:
            st["first_block"] = _first_block(out[3], out[4], out[5], self.factors)
        return st

    # ---- top-k retrieval -------------------------------------------------------------------------------------
    def recommend(self, users, k, exclude_seen=True):
        """The k items of highest score for each user: ``(items int32[n, k], scores float64[n, k])`` in the order
        of ``users``, score = ``predict(u, i)`` bit for bit, ties by item id ascending.  ``exclude_seen`` leaves out
        the user's items in the current train matrix; slots that cannot be filled hold item -1, score -inf.
        ``users`` may be a torch CUDA tensor (no host round trip of the inputs).  With several ranks the call is
        collective: every rank answers the users it owns and an all-gather gives every rank the whole result."""
        if self.world == 1:
            items, scores = _recommend_call(self.lib.eals_recommend, self.h, users, k, exclude_seen)
            return (items.cpu().numpy(), scores.cpu().numpy()) if not isinstance(items, np.ndarray) else (items, scores)
        import torch
        import torch.distributed as dist
        dev = f"cuda:{self.device}"
        u = (users if hasattr(users, "to") else torch.from_numpy(np.ascontiguousarray(users, np.int32).reshape(-1)))
        u = u.to(device=dev, dtype=torch.int32).reshape(-1)
        n, k = u.numel(), int(k)
        bad = u[(u < 0) | (u >= self.userCount)][:1].contiguous()
        if bad.numel():                   # the library's own argument error (EALS_ERR_ARG)
            out = torch.empty((1, max(k, 1)), dtype=torch.int32, device=dev)
            check(self.lib.eals_recommend(self.h, _lib.EALS_DEVICE, 1, _ptr(bad), k, int(bool(exclude_seen)), _ptr(out), None))
        bounds = torch.tensor(self.user_bounds, dtype=torch.int32, device=dev)
        owner = torch.bucketize(u, bounds[1:-1], right=True)            # rank owning each position
        counts = torch.bincount(owner, minlength=self.world).tolist()
        mine = torch.nonzero(owner == self.rank).reshape(-1)
        width = max(1, max(counts))
        items = torch.full((width, k), -1, dtype=torch.int32, device=dev)
        scores = torch.full((width, k), float("-inf"), dtype=torch.float64, device=dev)
        # An error on one rank (arguments, out of memory, ...) must not leave the others waiting in the all-gather:
        # every rank reports success or failure first, and all of them raise together.
        err = None
        try:
            if mine.numel():
                it, sc = _recommend_call(self.lib.eals_recommend, self.h, u[mine].contiguous(), k, exclude_seen)
                items[:mine.numel()] = it
                scores[:mine.numel()] = sc
            else:
                check(self.lib.eals_recommend(self.h, _lib.EALS_DEVICE, 0, None, k, int(bool(exclude_seen)), None, None))
        except Exception as e:
            err = e
        failed = torch.tensor([0 if err is None else self.rank + 1], dtype=torch.int32, device=dev)
        dist.all_reduce(failed, op=dist.ReduceOp.MAX, group=self.group)
        if err is not None:
            raise err
        if int(failed.item()):
            raise RuntimeError(f"recommend failed on rank {int(failed.item()) - 1}")
        all_items = torch.empty((self.world * width, k), dtype=torch.int32, device=dev)
        all_scores = torch.empty((self.world * width, k), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(all_items, items, group=self.group)
        dist.all_gather_into_tensor(all_scores, scores, group=self.group)
        out_i = torch.empty((n, k), dtype=torch.int32, device=dev)
        out_s = torch.empty((n, k), dtype=torch.float64, device=dev)
        for q in range(self.world):
            pos = torch.nonzero(owner == q).reshape(-1)
            out_i[pos] = all_items[q * width:q * width + counts[q]]
            out_s[pos] = all_scores[q * width:q * width + counts[q]]
        return out_i.cpu().numpy(), out_s.cpu().numpy()

    def fold_in(self, histories: SparseMat, init=None, n_iter=10):
        """User vectors for interaction histories, the model left as it is: ``n_iter`` passes (default 10, the
        reference's ``maxIterOnline``) of ``update_user_thread`` over each row of ``histories`` (a SparseMat whose
        rows are histories over this model's items; ratings are the confidence weights, None = 1), starting from
        ``init`` ([n, factors], None = zeros), against the current V, SV, Wi and reg.  Returns float64 [n, factors].
        Covers new users, users whose history changed since training and "what if" queries; together with
        ``recommend_vectors(Q, k, exclude=histories)`` it recommends for a history.  Inputs may be torch CUDA
        tensors.  With several ranks the call is collective: every rank folds in a slice of the histories and an
        all-gather gives every rank the whole result."""
        if self.world == 1:
            return _fold_in_call(self.lib.eals_fold_in, self.h, self.factors, f"cuda:{self.device}", histories, init, n_iter)
        host = lambda a: None if a is None else (a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a))
        rp, ci, rv, ini = host(histories.row_ptr), host(histories.col_idx), host(histories.row_val), host(init)

        def run(lo, hi):
            part = SparseMat(hi - lo, histories.N, rp[lo:hi + 1], ci, None, None, rv)
            return (_fold_in_call(self.lib.eals_fold_in, self.h, self.factors, f"cuda:{self.device}", part,
                                  None if ini is None else ini[lo:hi], n_iter),)
        return self._collective_slices(len(rp) - 1, run, [((self.factors,), np.float64, 0.0)])[0]

    def recommend_vectors(self, Q, k, exclude: SparseMat = None):
        """``recommend`` for arbitrary query vectors: the k items of highest score ``seq_dot(Q[s], V[i])`` for each
        row of ``Q`` ([n, factors]; ``Q[s] == U[u]`` gives exactly ``recommend([u])``), the items of row s of
        ``exclude`` (a SparseMat with one row per query, or None) left out.  Returns ``(items int32[n, k], scores
        float64[n, k])``.  Inputs may be torch CUDA tensors.  With several ranks the call is collective, like
        ``recommend``."""
        if self.world == 1:
            return _recommend_vectors_call(self.lib.eals_recommend_vectors, self.h, self.factors, f"cuda:{self.device}",
                                           Q, k, exclude)
        host = lambda a: None if a is None else (a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a))
        q = host(Q)
        ep, ei = (None, None) if exclude is None else (host(exclude.row_ptr), host(exclude.col_idx))
        k = int(k)

        def run(lo, hi):
            part = None if ep is None else SparseMat(hi - lo, exclude.N, ep[lo:hi + 1], ei, None, None)
            return _recommend_vectors_call(self.lib.eals_recommend_vectors, self.h, self.factors, f"cuda:{self.device}",
                                           q[lo:hi], k, part)
        return tuple(self._collective_slices(len(q), run, [((max(k, 1),), np.int32, -1),
                                                           ((max(k, 1),), np.float64, float("-inf"))]))

    def similar_items(self, items, k):
        """The k items most similar to each of ``items`` by cosine similarity: ``(ids int32[n, k], scores float64[n, k])``.
        With ``v^ = v / sqrt(seq_dot(v, v))`` per row (a zero row stays zero) the score is ``seq_dot(v^_q, v^_r)`` bit for
        bit; the order is score descending, then item id ascending; only the query item itself is left out (other
        items with the same vector tie); slots that cannot be filled hold -1 and -inf.  1 <= k <= 1024.  ``items`` may
        be a torch CUDA tensor.  The model is not touched.  With several ranks the call is collective, like
        ``recommend_vectors``."""
        return self._similar(_lib.BUF_V, items, k)

    def similar_users(self, users, k):
        """``similar_items`` over the user factors: the k users most similar to each of ``users``."""
        return self._similar(_lib.BUF_U, users, k)

    def _similar(self, which, ids, k):
        dev = f"cuda:{self.device}"
        if self.world == 1:
            return _similar_call(self.lib.eals_similar, self.h, which, dev, ids, k)
        q = (ids.cpu().numpy() if hasattr(ids, "cpu") else np.asarray(ids)).reshape(-1)
        k = int(k)
        run = lambda lo, hi: _similar_call(self.lib.eals_similar, self.h, which, dev, q[lo:hi], k)
        return tuple(self._collective_slices(len(q), run, [((max(k, 1),), np.int32, -1),
                                                           ((max(k, 1),), np.float64, float("-inf"))]))

    def ranking_metrics(self, test: SparseMat, k, exclude_seen=True, per_user=False, ranks=False):
        """Ranking metrics at k on a held-out test matrix ``test`` (a SparseMat with one row per user over this model's
        items; only its CSR is read).  For a test entry (u, g) the rank is g's 0-based position in
        ``recommend([u], k, exclude_seen)[0]``, or -1 (with ``exclude_seen`` a test item in u's train row is always
        -1 and still counts in u's test items).  Returns a dict of the means over the users with test items of
        ``hit_rate``, ``precision`` (hits / k), ``recall`` (hits / n_u), ``ndcg``, ``map`` and ``mrr``, plus ``users``
        (their number); ``per_user=True`` adds ``per_user`` (float64 [userCount, 6] in that order, 0 for users without
        test items), ``ranks=True`` adds ``ranks`` (int32, one per test entry in CSR order).  The model is not touched.
        Inputs may be torch CUDA tensors.  With several ranks the call is collective: every rank ranks the rows it
        owns, every rank reports success or failure, then the sums are added in rank order and the arrays gathered."""
        dev = f"cuda:{self.device}"
        if self.world == 1:
            sums, users, pu, rk = _ranking_metrics_call(self.lib.eals_ranking_metrics, self.h, dev, test, self.userCount, k,
                                                        exclude_seen, (0, self.userCount), per_user, ranks)
            return _ranking_result(sums / users if users else sums * 0.0, users, pu, rk)
        import torch
        import torch.distributed as dist
        ub, ue = self.user_bounds[self.rank], self.user_bounds[self.rank + 1]
        err, sums, users, pu, rk = None, np.zeros(6), 0, None, None
        try:
            sums, users, pu, rk = _ranking_metrics_call(self.lib.eals_ranking_metrics, self.h, dev, test, self.userCount, k,
                                                        exclude_seen, (ub, ue), per_user, ranks)
        except Exception as e:
            err = e
        failed = torch.tensor([0 if err is None else self.rank + 1], dtype=torch.int32, device=dev)
        dist.all_reduce(failed, op=dist.ReduceOp.MAX, group=self.group)
        if err is not None:
            raise err
        if int(failed.item()):
            raise RuntimeError(f"ranking_metrics failed on rank {int(failed.item()) - 1}")
        part = torch.tensor([*sums.tolist(), float(users)], dtype=torch.float64, device=dev)
        every = torch.empty(self.world * 7, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(every, part, group=self.group)
        every = every.cpu().numpy().reshape(self.world, 7)
        tot, n = np.zeros(6), 0
        for q in range(self.world):          # rank order: the same sums on every rank
            tot += every[q, :6]
            n += int(every[q, 6])
        rp = test.row_ptr.cpu().numpy() if hasattr(test.row_ptr, "cpu") else np.asarray(test.row_ptr)
        if per_user:
            pu = self._gather_parts(pu, [self.user_bounds[q + 1] - self.user_bounds[q] for q in range(self.world)])
        if ranks:
            b = self.user_bounds
            rk = self._gather_parts(rk, [int(rp[b[q + 1]]) - int(rp[b[q]]) for q in range(self.world)])
        return _ranking_result(tot / n if n else tot, n, pu, rk)

    def _gather_parts(self, a, counts):
        """Every rank's host array ``a`` (counts[rank] leading rows) concatenated in rank order, on every rank."""
        import torch
        import torch.distributed as dist
        dev = f"cuda:{self.device}"
        width = max(1, max(counts))
        buf = torch.zeros((width, *a.shape[1:]), dtype=torch.from_numpy(a[:0]).dtype, device=dev)
        buf[:len(a)] = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        full = torch.empty((self.world * width, *a.shape[1:]), dtype=buf.dtype, device=dev)
        dist.all_gather_into_tensor(full, buf, group=self.group)
        return torch.cat([full[q * width:q * width + counts[q]] for q in range(self.world)]).cpu().numpy()

    def _collective_slices(self, n, run, outs):
        """Several processes: rank r answers the queries [n*r/world, n*(r+1)/world) with run(lo, hi), one host array
        per entry (trailing shape, dtype, pad) of ``outs``.  Every rank reports success or failure before an NCCL
        all-gather gives every rank the whole result, so an error on one rank raises on all of them instead of
        leaving the others in the all-gather, and no rank starts its next sweep (which stores into the other ranks'
        V replicas) while another still reads its own."""
        import torch
        import torch.distributed as dist
        dev = f"cuda:{self.device}"
        bounds = [n * q // self.world for q in range(self.world + 1)]
        width = max(1, max(bounds[q + 1] - bounds[q] for q in range(self.world)))
        tdt = lambda dt: torch.from_numpy(np.empty(0, dt)).dtype
        bufs = [torch.full((width, *shape), pad, dtype=tdt(dt), device=dev) for shape, dt, pad in outs]
        lo, hi = bounds[self.rank], bounds[self.rank + 1]
        err = None
        try:
            for b, a in zip(bufs, run(lo, hi)):
                b[:hi - lo] = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        except Exception as e:
            err = e
        failed = torch.tensor([0 if err is None else self.rank + 1], dtype=torch.int32, device=dev)
        dist.all_reduce(failed, op=dist.ReduceOp.MAX, group=self.group)
        if err is not None:
            raise err
        if int(failed.item()):
            raise RuntimeError(f"call failed on rank {int(failed.item()) - 1}")
        res = []
        for b in bufs:
            full = torch.empty((self.world * width, *b.shape[1:]), dtype=b.dtype, device=dev)
            dist.all_gather_into_tensor(full, b, group=self.group)
            res.append(torch.cat([full[q * width:q * width + bounds[q + 1] - bounds[q]] for q in range(self.world)]).cpu().numpy())
        return res

    def recommend_stats(self):
        """How the last recommend ran on this rank: engine ('tcgen05' or 'fp64'), exact seed size, pairs re-scored,
        users left after the first item block and that block's shape, time and tensor rate."""
        return _recommend_stats(self.lib, self.h, self.factors)

    # ---- instrumentation -----------------------------------------------------------------------------------
    def timings(self):
        ms = np.zeros(6)
        check(self.lib.eals_timings(self.h, _ptr(ms)))
        return dict(zip(("user_sweep", "user_gram", "item_sweep", "item_gram", "loss", "evaluate"), ms.tolist()))

    PHASES = ("user_sweep", "user_gram", "item_sweep", "item_gram", "loss", "evaluate")

    def timings_total(self, reset=False):
        """Accumulated device ms and call counts per phase since the last reset."""
        ms, calls = np.zeros(6), np.zeros(6, np.int64)
        check(self.lib.eals_timings_total(self.h, _ptr(ms), _ptr(calls), int(reset)))
        return dict(zip(self.PHASES, ms.tolist())), dict(zip(self.PHASES, calls.tolist()))

    def timings_detail(self):
        """Accumulated device ms of the sweep sub-phases (heavy / one-CTA / warp rows per side)."""
        ms, calls = np.zeros(6), np.zeros(6, np.int64)
        check(self.lib.eals_timings_detail(self.h, _ptr(ms), _ptr(calls)))
        names = ("user_heavy", "user_mid", "user_warp", "item_heavy", "item_mid", "item_warp")
        return dict(zip(names, ms.tolist()))

    def kernel_launches(self) -> int:
        return int(self.lib.eals_kernel_launches(self.h))

    def owned_nnz(self) -> int:
        return int(self.lib.eals_nnz(self.h))


# --------------------------------------------------------------------------------------------------
# The same class over eals_group: N ranks in ONE process (include/eals_b200.h, "eals_group").
# --------------------------------------------------------------------------------------------------
class GroupMF_fastALS:
    """``MF_fastALS`` with the multi-GPU split behind the C ABI: one process, one host thread, rank r on
    ``devices[r]``.  ``devices=[0, 0, 0, 0]`` runs four *virtual ranks* on one GPU — the whole sharded path
    (cost-model partition, peer stores of finished rows, routed prediction caches, fixed-order all-reduce of
    the partial Grams, setTrain re-attachment) without needing four GPUs; this is what the 1-GPU CI runs.
    Same method names and meanings as ``MF_fastALS`` (MF_fastALS.h:52-72)."""

    def __init__(self, trainMatrix: SparseMat, testRatings, topK=10, threadNum=1, factors=64, maxIter=20,
                 w0=10.0, alpha=0.75, reg=0.01, init_mean=0.0, init_stdev=0.01, showProgress=False,
                 showLoss=True, userCount=None, itemCount=None, *, devices=(0,), init=True, out=None):
        self.lib = _lib.load()
        sm = self.trainMatrix = trainMatrix
        self.userCount, self.itemCount = int(userCount or sm.M), int(itemCount or sm.N)
        self.topK, self.factors, self.maxIter = int(topK), int(factors), int(maxIter)
        self.w0, self.alpha, self.reg = float(w0), float(alpha), float(reg)
        self.showloss = bool(showLoss)
        del threadNum, showProgress
        self.out = out or sys.stdout
        self.devices = [int(d) for d in devices]
        self.world = len(self.devices)
        self.testItems = None if testRatings is None else np.ascontiguousarray(testRatings, np.int32)
        p = EalsParams()
        self.lib.eals_default_params(C.byref(p))
        p.n_users, p.n_items, p.factors, p.topk = sm.M, sm.N, self.factors, self.topK
        p.w0, p.alpha, p.reg = self.w0, self.alpha, self.reg
        p.init_mean, p.init_stdev = float(init_mean), float(init_stdev)
        p.input_space = _lib.EALS_DEVICE if sm.on_device else _lib.EALS_HOST
        dev = np.ascontiguousarray(self.devices, np.int32)
        g = C.c_void_p()
        check(self.lib.eals_group_create(C.byref(p), self.world, _ptr(dev), _ptr(sm.row_ptr), _ptr(sm.col_idx),
                                         _ptr(sm.row_val), _ptr(sm.col_ptr), _ptr(sm.row_idx), _ptr(sm.col_val), C.byref(g)))
        self.g = g
        ub, ib = np.zeros(self.world + 1, np.int32), np.zeros(self.world + 1, np.int32)
        check(self.lib.eals_group_bounds(self.g, _ptr(ub), _ptr(ib)))
        self.user_bounds, self.item_bounds = ub.tolist(), ib.tolist()
        if init:
            check(self.lib.eals_group_init_factors(self.g))

    def close(self):
        if getattr(self, "g", None):
            self.lib.eals_group_destroy(self.g)
            self.g = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def rank_model(self, r):
        h = C.c_void_p()
        check(self.lib.eals_group_model(self.g, int(r), C.byref(h)))
        return h

    def rank_factors(self, r):
        """(U, V) replicas of rank r as host arrays."""
        U, V = np.empty((self.userCount, self.factors)), np.empty((self.itemCount, self.factors))
        check(self.lib.eals_get_factors(self.rank_model(r), _lib.EALS_HOST, _ptr(U), _ptr(V)))
        return U, V

    def rank_S(self, r):
        SU, SV = np.empty((self.factors, self.factors)), np.empty((self.factors, self.factors))
        check(self.lib.eals_get_S(self.rank_model(r), _lib.EALS_HOST, _ptr(SU), _ptr(SV)))
        return SU, SV

    U = property(lambda s: s.rank_factors(0)[0])
    V = property(lambda s: s.rank_factors(0)[1])
    SU = property(lambda s: s.rank_S(0)[0])
    SV = property(lambda s: s.rank_S(0)[1])

    @property
    def Wi(self):
        w = np.empty(self.itemCount)
        check(self.lib.eals_group_get_item_weights(self.g, _lib.EALS_HOST, _ptr(w)))
        return w

    @Wi.setter
    def Wi(self, w):
        w = np.ascontiguousarray(w, np.float64)
        check(self.lib.eals_group_set_item_weights(self.g, _lib.EALS_HOST, _ptr(w)))

    def sync(self):
        check(self.lib.eals_group_sync(self.g))

    def setUV(self, U, V):
        U = None if U is None else np.ascontiguousarray(U, np.float64)
        V = None if V is None else np.ascontiguousarray(V, np.float64)
        check(self.lib.eals_group_set_factors(self.g, _lib.EALS_HOST, _ptr(U), _ptr(V)))

    def setTrain(self, sm: SparseMat):
        space = _lib.EALS_DEVICE if sm.on_device else _lib.EALS_HOST
        check(self.lib.eals_group_set_train(self.g, space, _ptr(sm.row_ptr), _ptr(sm.col_idx), _ptr(sm.row_val),
                                            _ptr(sm.col_ptr), _ptr(sm.row_idx), _ptr(sm.col_val)))
        self.trainMatrix = sm

    def update_user(self):
        check(self.lib.eals_group_update_user(self.g))

    def update_item(self):
        check(self.lib.eals_group_update_item(self.g))

    def runOneIteration(self):
        self.update_user()
        self.update_item()

    def update_user_thread(self, u):
        check(self.lib.eals_group_update_user_row(self.g, int(u)))

    def update_item_thread(self, i):
        check(self.lib.eals_group_update_item_row(self.g, int(i)))

    def update_user_SU(self, oldVector, uget):
        o, n = np.ascontiguousarray(oldVector, np.float64), np.ascontiguousarray(uget, np.float64)
        check(self.lib.eals_group_patch_SU(self.g, _ptr(o), _ptr(n)))

    def update_item_SV(self, i, oldVector, vget):
        o, n = np.ascontiguousarray(oldVector, np.float64), np.ascontiguousarray(vget, np.float64)
        check(self.lib.eals_group_patch_SV(self.g, int(i), _ptr(o), _ptr(n)))

    def _factor_row(self, which, r):
        out = np.empty(self.factors)
        check(self.lib.eals_group_get_factor_row(self.g, which, int(r), _ptr(out)))
        return out

    def updateModel(self, u, i, patch_S=True, maxIterOnline=10):
        """Online update on a sharded model (MF_fastALS.cpp:223-242): the owner of user u / item i runs the
        single-row kernel, which stores the new row into every replica; the S patches go to every rank."""
        u, i = int(u), int(i)
        grown = insert_interaction(self.trainMatrix, u, i)
        if grown is not None:
            self.setTrain(grown)
        Wi = self.Wi
        if Wi[i] == 0.0:
            Wi[i] = self.w0 / self.itemCount
            self.Wi = Wi
        for _ in range(int(maxIterOnline)):
            old = self._factor_row(_lib.BUF_U, u) if patch_S else None
            self.update_user_thread(u)
            if patch_S:
                self.update_user_SU(old, self._factor_row(_lib.BUF_U, u))
            old = self._factor_row(_lib.BUF_V, i) if patch_S else None
            self.update_item_thread(i)
            if patch_S:
                self.update_item_SV(i, old, self._factor_row(_lib.BUF_V, i))

    def loss(self) -> float:
        v = C.c_double()
        check(self.lib.eals_group_loss(self.g, C.byref(v)))
        return v.value

    def predict(self, u, i) -> float:
        s = C.c_double()
        check(self.lib.eals_group_predict(self.g, int(u), int(i), C.byref(s)))
        return s.value

    def evaluate(self, testRatings=None, topK=None, exact=False, per_user=False):
        items = self.testItems if testRatings is None else np.ascontiguousarray(testRatings, np.int32)
        topK = int(topK or self.topK)
        means = np.zeros(3)
        hr = ndcg = prec = cnt = None
        if per_user:
            hr, ndcg, prec = np.zeros(self.userCount), np.zeros(self.userCount), np.zeros(self.userCount)
            cnt = np.zeros(self.userCount, np.int32)
        check(self.lib.eals_group_evaluate(self.g, _ptr(items), topK, _lib.EVAL_EXACT if exact else _lib.EVAL_REFERENCE,
                                           _ptr(means), _ptr(hr), _ptr(ndcg), _ptr(prec), _ptr(cnt)))
        return (means, hr, ndcg, prec, cnt) if per_user else means

    def recommend(self, users, k, exclude_seen=True):
        """``MF_fastALS.recommend`` over all ranks: each user is answered by the rank that owns it."""
        items, scores = _recommend_call(self.lib.eals_group_recommend, self.g, users, k, exclude_seen)
        return (items.cpu().numpy(), scores.cpu().numpy()) if not isinstance(items, np.ndarray) else (items, scores)

    def fold_in(self, histories: SparseMat, init=None, n_iter=10):
        """``MF_fastALS.fold_in`` over all ranks: balanced contiguous slices of the histories, one per rank."""
        return _fold_in_call(self.lib.eals_group_fold_in, self.g, self.factors, f"cuda:{self.devices[0]}", histories,
                             init, n_iter)

    def recommend_vectors(self, Q, k, exclude: SparseMat = None):
        """``MF_fastALS.recommend_vectors`` over all ranks: balanced contiguous slices of the queries, one per rank."""
        return _recommend_vectors_call(self.lib.eals_group_recommend_vectors, self.g, self.factors, f"cuda:{self.devices[0]}",
                                       Q, k, exclude)

    def similar_items(self, items, k):
        """``MF_fastALS.similar_items`` over all ranks: balanced contiguous slices of the queries, one per rank."""
        return _similar_call(self.lib.eals_group_similar, self.g, _lib.BUF_V, f"cuda:{self.devices[0]}", items, k)

    def similar_users(self, users, k):
        """``MF_fastALS.similar_users`` over all ranks: balanced contiguous slices of the queries, one per rank."""
        return _similar_call(self.lib.eals_group_similar, self.g, _lib.BUF_U, f"cuda:{self.devices[0]}", users, k)

    def ranking_metrics(self, test: SparseMat, k, exclude_seen=True, per_user=False, ranks=False):
        """``MF_fastALS.ranking_metrics`` over all ranks: each rank ranks the test rows it owns, sums in rank order."""
        means, users, pu, rk = _ranking_metrics_call(self.lib.eals_group_ranking_metrics, self.g, f"cuda:{self.devices[0]}", test,
                                                     self.userCount, k, exclude_seen, (0, self.userCount), per_user, ranks)
        return _ranking_result(means, users, pu, rk)

    def replicas_consistent(self) -> bool:
        ok = C.c_int32()
        check(self.lib.eals_group_replicas_consistent(self.g, C.byref(ok)))
        return bool(ok.value)

    def save(self, path):
        check(self.lib.eals_group_save_factors(self.g, os.fsencode(path)))

    def load(self, path):
        check(self.lib.eals_group_load_factors(self.g, os.fsencode(path)))

    def buildModel(self):
        loss_pre = float("inf")
        self.losses = []
        for it in range(self.maxIter):
            t0 = time.perf_counter()
            self.update_user(); self.sync()
            t_user = time.perf_counter() - t0
            print(f"Time of user_update: {t_user:g}", file=self.out)
            t0 = time.perf_counter()
            self.update_item(); self.sync()
            t_item = time.perf_counter() - t0
            print(f"Time of item_update: {t_item:g}", file=self.out)
            if self.showloss:
                t0 = time.perf_counter()
                cur = self.loss()
                print(f"Iter={it} {t_user + t_item:g} {'-' if loss_pre >= cur else '+'} loss:{cur:g} {time.perf_counter() - t0:g}", file=self.out)
                loss_pre = cur
                self.losses.append(cur)

    def kernel_launches(self) -> int:
        return int(self.lib.eals_group_kernel_launches(self.g))
