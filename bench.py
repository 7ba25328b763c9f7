#!/usr/bin/env python
"""bench.py — eALS epoch throughput on B200 (BASELINE.json metric: nnz*K updates/s, epoch time).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c4|c3|c2|c1|c4s|small]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's CPU path on the host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed epoch's outputs as DIR/<name>.npy

A step = one eALS epoch (user half-epoch + item half-epoch, each incl. the S-cache Gram and, with
N > 1, the exchange of the updated factor rows and the all-reduce of the partial Grams) — what the
reference prints as the 2nd field of its `Iter=` line (MF_fastALS.cpp:125-158).  loss()/evaluate()
are outside the timed region, as in the reference.

value  = 2*nnz*K / epoch seconds, inputs resident in HBM, device-timed (CUDA events, max over ranks)
e2e    = same metric through the public API with HOST (pinned) train-matrix buffers: every step
         uploads the CSR+CSC arrays (setTrain), runs the epoch and reads the loss back.
Workload: the north-star target configuration (BASELINE.json configs[3], "c4": 10M x 2M, 500M
interactions, K=128) — it fits one B200 (about 25 GB), so it is also the N=1 workload; N > 1 shards
the SAME matrix (strong scaling).  Synthetic power-law data (no dataset ships with the reference).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "eals_nnzK_updates_per_s"
UNIT = "nnz*K updates/s"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


def cd_bytes_per_epoch(M, N, K, nnz_user_side, nnz_item_side, rows_u, rows_i):
    """Algorithmic bytes of the two CD sweeps (SURVEY.md §8d, DESIGN.md §4), all-ones ratings:
    every nonzero gathers the other side's K-vector once per sweep (K*8 B) and its index (4 B);
    every updated row is read and written once (2*K*8 B); offsets 8 B per row; Wi 8 B per item
    read on the user side (per nonzero it is an L2-resident gather, counted once per item) and once
    per row on the item side."""
    s = 8
    return ((nnz_user_side + nnz_item_side) * (K * s + 4)
            + 2 * (rows_u + rows_i) * K * s
            + (rows_u + rows_i + 2) * 8
            + 2 * N * s)


def workload_string(name, spec, nnz):
    """The ONE description of a workload both arms print (config.workload)."""
    return (f"{name}: {spec['M']} users x {spec['N']} items, {nnz} interactions, K={spec['K']}, "
            f"power-law (Zipf {spec['zipf']}) synthetic, all ratings 1, w0=10 alpha=0.75 reg=0.01")


def fp64_pipe_floor_ms(nnz_both_sweeps, K, sms=148, sm_mhz=1965.0):
    """Second ceiling of the CD sweeps (DESIGN.md §3.1): the blocked formulation issues 5 DMMA.884 per 4
    nonzeros and 16-factor block; a DMMA occupies an SM sub-partition's fp64 pipe for 16.1 cycles (measured,
    profiles/r01_fp64_rate_b200.txt); 4 sub-partitions per SM."""
    dmma = nnz_both_sweeps * ((K + 15) // 16) * 1.25
    return dmma * 16.1 / (4 * sms * sm_mhz * 1e6) * 1e3


# --------------------------------------------------------------------------------------------------
# clocks: NVML sampler thread (nvidia-smi's numbers without forking)
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index, period=0.1):
        self.samples, self.reasons, self.stop_flag = [], set(), False
        self.max_mhz = None
        self.period = period
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:            # pragma: no cover
            self.nv = None
            self.err = repr(e)
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def __enter__(self):
        if self.nv:
            self.t.start()
        return self

    def __exit__(self, *a):
        self.stop_flag = True
        if self.nv:
            self.t.join(timeout=2)

    def summary(self):
        if not self.nv or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------------
# workload
# --------------------------------------------------------------------------------------------------
def build_workload(name, device):
    """Synthetic matrix of the named shape, generated on the GPU (torch = plumbing: RNG/sort)."""
    import torch
    from eals_cpp_b200 import datasets
    from eals_cpp_b200.model import SparseMat
    spec = dict(datasets.WORKLOADS[name])
    t0 = time.perf_counter()
    with torch.cuda.device(device):
        row_ptr, col_idx, test_items = datasets.powerlaw_csr_device(device=f"cuda:{device}", **spec)
        sm = SparseMat.from_csr_device(spec["M"], spec["N"], row_ptr, col_idx)
        torch.cuda.synchronize()
    log(f"[bench] workload {name}: M={spec['M']} N={spec['N']} nnz={sm.nnz} K={spec['K']} "
        f"generated in {time.perf_counter() - t0:.1f}s")
    return spec, sm, test_items


def random_factors(M, N, K, device, seed=1234):
    """N(0, 0.01) factors on the device — the reference's init distribution (main.cpp:141-142); the
    libstdc++-exact sequential stream is used by the parity tests, not at 1.5e9 values."""
    import torch
    g = torch.Generator(device=f"cuda:{device}")
    g.manual_seed(seed)
    U = torch.randn(M, K, generator=g, device=f"cuda:{device}", dtype=torch.float64) * 0.01
    V = torch.randn(N, K, generator=g, device=f"cuda:{device}", dtype=torch.float64) * 0.01
    return U, V


DUMP_BYTES = 64_000_000


def dump_outputs(fals, out_dir, seed=2024):
    """Write what a caller of the timed path holds after its last epoch, as float64 .npy files: the S caches
    SU and SV whole, and U and V whole when everything fits in DUMP_BYTES.  Otherwise U_rows / V_rows hold a
    sample of rows: the same sorted, seeded row ids in every run with the same arguments (the inputs are seeded
    too), so the files of two builds can be compared one for one.  Reads through the library's host copies,
    which leave the prediction caches valid: the rest of the run computes what it would without the dump."""
    from eals_cpp_b200 import _lib
    os.makedirs(out_dir, exist_ok=True)
    M, N, K = fals.userCount, fals.itemCount, fals.factors
    out = {"SU": fals.SU, "SV": fals.SV}
    rows_each = (DUMP_BYTES - 2 * K * K * 8 - 4 * 4096) // (2 * K * 8)     # 4096: room for the .npy headers
    rng = np.random.default_rng(seed)
    for name, which, n in (("U", _lib.BUF_U, M), ("V", _lib.BUF_V, N)):
        if n <= rows_each:
            out[name] = fals.U if which == _lib.BUF_U else fals.V
        else:
            rows = np.sort(rng.choice(n, size=rows_each, replace=False))
            out[name + "_rows"] = np.stack([fals._factor_row(which, r) for r in rows])
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, np.float64))
    log(f"[bench] outputs of the last timed step in {out_dir}: " +
        ", ".join(f"{k} {tuple(v.shape)}" for k, v in out.items()))


# --------------------------------------------------------------------------------------------------
# CPU side (test infrastructure used as the reported baseline / the reference arm)
# --------------------------------------------------------------------------------------------------
def cpu_port_sample(sm, K, reg, w0, alpha, target_nnz, threads, seed=7):
    """Time the oracle port (oracle/eals_oracle.c: the reference's update_user_thread /
    update_item_thread arithmetic on flat arrays) on a bounded sample of this workload: the first
    users and the first items whose rows hold ~target_nnz nonzeros each, with the factor rows they
    gather compacted into dense host arrays.  Rows are independent inside a half-epoch, so `threads`
    host threads each take a contiguous sub-range (ctypes releases the GIL)."""
    import torch
    from oracle.bindings import Port
    port = Port()
    rng = np.random.default_rng(seed)

    def side(ptr_t, idx_t, n_other):
        ptr = ptr_t.cpu().numpy() if hasattr(ptr_t, "cpu") else np.asarray(ptr_t)
        rows = int(np.searchsorted(ptr, target_nnz, side="left"))
        rows = max(1, min(rows, len(ptr) - 1))
        nnz = int(ptr[rows])
        idx = idx_t[:nnz]
        if hasattr(idx, "cpu"):
            uniq, inv = torch.unique(idx.long(), return_inverse=True)
            uniq, inv = uniq.cpu().numpy(), inv.cpu().numpy().astype(np.int32)
        else:
            uniq, inv = np.unique(np.asarray(idx), return_inverse=True)
            inv = inv.astype(np.int32)
        return np.ascontiguousarray(ptr[:rows + 1]), np.ascontiguousarray(inv), uniq, rows, nnz

    def fill(n):      # N(0, 0.01) block tiled: timing does not depend on the values
        base = rng.normal(0, 0.01, (min(n, 4096), K))
        return np.ascontiguousarray(np.tile(base, ((n + len(base) - 1) // len(base), 1))[:n])

    out = {}
    # user side: sampled users gather item vectors
    rp, ci, items, Mu, nnz_u = side(sm.row_ptr, sm.col_idx, sm.N)
    # item side: sampled items gather user vectors
    cp, ri, users, Ni, nnz_i = side(sm.col_ptr, sm.row_idx, sm.M)

    def run(fn, ptr, idx, X, Y, SX, SY, Wi, nrows):
        bounds = np.linspace(0, nrows, threads + 1).astype(int)
        # balance by nnz rather than rows
        tot = ptr[nrows]
        bounds = [int(np.searchsorted(ptr, tot * t / threads)) for t in range(threads)] + [nrows]
        ths = [threading.Thread(target=fn, args=(ptr, idx, None, X, Y, SX, SY, Wi, reg, bounds[t], bounds[t + 1], False))
               for t in range(threads) if bounds[t + 1] > bounds[t]]
        t0 = time.perf_counter()
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        return time.perf_counter() - t0

    # user sweep: X = U[Mu], Y = V compact
    U = fill(Mu)
    Vc = fill(len(items))
    Wi = np.full(len(items), w0 / max(sm.N, 1))
    SV = Vc.T @ (Vc * Wi[:, None]) * (sm.N / max(len(items), 1))
    SU = np.eye(K)
    t_user = run(lambda p, i, v, X, Y, SX, SY, W, r, b, e, ps: port.update_user_sweep(p, i, v, X, Y, SX, SY, W, r, b, e, ps),
                 rp, ci, U, Vc, SU, SV, Wi, Mu)
    # item sweep: X = V[Ni], Y = U compact
    V = fill(Ni)
    Uc = fill(len(users))
    Wi2 = np.full(Ni, w0 / max(sm.N, 1))
    SU2 = Uc.T @ Uc * (sm.M / max(len(users), 1))
    t_item = run(lambda p, i, v, X, Y, SX, SY, W, r, b, e, ps: port.update_item_sweep(p, i, v, Y, X, SY, SX, W, r, b, e, ps),
                 cp, ri, V, Uc, np.eye(K), SU2, Wi2, Ni)
    nnz = sm.nnz
    epoch_s = nnz / (nnz_u / t_user) + nnz / (nnz_i / t_item)     # extrapolated whole-epoch CPU time
    out.update(value=2.0 * nnz * K / epoch_s, unit=UNIT, cores=threads, kind="port",
               sample=(f"oracle port (eals_oracle.c, gcc -O2) on the first {Mu} users ({nnz_u} nnz, {t_user:.2f}s) and "
                       f"first {Ni} items ({nnz_i} nnz, {t_item:.2f}s) of this workload, gathered factor rows "
                       f"compacted on the host, {threads} threads over disjoint row ranges, S patch excluded; "
                       f"extrapolated epoch {epoch_s:.1f}s"),
               epoch_s_extrapolated=epoch_s, sample_seconds=t_user + t_item)
    return out


def _submatrix_by_rows(ptr, idx, n_rows, take):
    """CSR of every `take`-th row of (ptr, idx) (torch tensors on any device or numpy), with the column ids
    relabelled to 0..n_distinct-1 in ascending order (rows stay ascending).  Returns host arrays."""
    import torch
    ptr = torch.as_tensor(ptr)
    idx = torch.as_tensor(idx)
    rows = torch.arange(0, n_rows, take, device=ptr.device)
    lens = ptr[rows + 1] - ptr[rows]
    new_ptr = torch.zeros(len(rows) + 1, dtype=torch.int64, device=ptr.device)
    new_ptr[1:] = torch.cumsum(lens, 0)
    total = int(new_ptr[-1])
    src = torch.repeat_interleave(ptr[rows] - new_ptr[:-1], lens) + torch.arange(total, device=ptr.device)
    cols = idx[src].long()
    uniq, inv = torch.unique(cols, return_inverse=True)
    return new_ptr.cpu().numpy(), inv.to(torch.int32).cpu().numpy(), int(len(rows)), int(len(uniq))


def _transpose_csr(n_rows, n_cols, ptr, idx):
    rows = np.repeat(np.arange(n_rows, dtype=np.int32), np.diff(ptr))
    order = np.argsort(idx, kind="stable")
    tptr = np.zeros(n_cols + 1, np.int64)
    np.cumsum(np.bincount(idx, minlength=n_cols), out=tptr[1:])
    return tptr, np.ascontiguousarray(rows[order])


def cpu_reference_sampled(sm, M, N, K, target_nnz, steps, warmup):
    """The REAL MF_fastALS object (oracle/_ref: the reference's own translation units, -O3, one thread — the
    reference has no working threading) on a row-sampled sub-matrix of a workload it cannot hold whole
    (SURVEY.md §8d).  User half-epoch: every s-th user with ALL its nonzeros (a user row's work is exactly what
    it is in the full matrix), the items it touches relabelled densely.  Item half-epoch: every t-th item with
    all its nonzeros, users relabelled.  Each is timed through the reference's own sweep + S-patch calls
    (MF_fastALS.cpp:127-132, 146-152) and scaled by the sampling factor."""
    from oracle.bindings import Reference
    nnz = sm.nnz
    take_u = max(1, int(round(nnz / target_nnz)))
    take_i = max(1, int(round(nnz / target_nnz)))
    rp, ci, Mu, Nu = _submatrix_by_rows(sm.row_ptr, sm.col_idx, M, take_u)
    cp, ri, Ni, Mi = _submatrix_by_rows(sm.col_ptr, sm.row_idx, N, take_i)
    # the item sample arrives as "items x users"; the reference's constructor wants users x items
    rp_i, ci_i = _transpose_csr(Ni, Mi, cp, ri)
    t0 = time.perf_counter()
    ref_u = Reference(Mu, Nu, rp, ci, factors=K, fast=True)
    ref_i = Reference(Mi, Ni, rp_i, ci_i, factors=K, fast=True)
    build_s = time.perf_counter() - t0
    tu, ti = [], []
    for it in range(warmup + steps):
        t0 = time.perf_counter(); ref_u.update_user(); t1 = time.perf_counter()
        ref_i.update_item(); t2 = time.perf_counter()
        if it >= warmup:
            tu.append(t1 - t0); ti.append(t2 - t1)
    nnz_u, nnz_i = int(rp[-1]), int(cp[-1])
    epoch_s = float(np.mean(tu)) * (nnz / max(nnz_u, 1)) * 1.0 + float(np.mean(ti)) * (nnz / max(nnz_i, 1)) * 1.0
    # scale by rows, not nonzeros, for the user side (uniform row sample): identical up to sampling noise
    epoch_rows = float(np.mean(tu)) * (M / Mu) + float(np.mean(ti)) * (N / Ni)
    sample = (f"oracle/_ref (the reference's own TUs, g++ -O3, 1 thread) on a row sample: every {take_u}th user "
              f"({Mu} users, {nnz_u} nnz, {Nu} distinct items relabelled; user sweep + SU patch {np.mean(tu):.3f}s) and every "
              f"{take_i}th item ({Ni} items, {nnz_i} nnz, {Mi} distinct users relabelled; item sweep + SV patch {np.mean(ti):.3f}s), "
              f"scaled by the row-sampling factors to the whole matrix: extrapolated epoch {epoch_rows:.1f}s "
              f"(by nonzeros: {epoch_s:.1f}s); objects built in {build_s:.1f}s; mean of {steps} steps")
    return epoch_rows, sample


def cpu_reference_full(sm_host, K, steps, warmup):
    """The real MF_fastALS object (oracle/_ref, -O3 build), whole epochs, 1 thread."""
    from oracle.bindings import Reference
    ref = Reference(sm_host.M, sm_host.N, sm_host.row_ptr, sm_host.col_idx, factors=K, fast=True)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        ref.update_user()
        ref.update_item()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    return float(np.mean(times))


def cpu_port_full(sm_host, K, steps, warmup):
    """The same whole epochs through the oracle port (PortModel: the reference's arithmetic and S patches), 1 thread."""
    from oracle.bindings import PortModel
    port = PortModel(sm_host.M, sm_host.N, sm_host.row_ptr, sm_host.col_idx, factors=K)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        port.update_user()
        port.update_item()
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    return float(np.mean(times))


# --------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("EALS_BENCH_WORKLOAD", "c4"))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the c1/c2/c3 epochs and the C5 evaluation after the main run")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--cpu-nnz", type=int, default=0, help="nonzeros per side in the CPU sample (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed epoch computed (U, V rows and the S caches) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        log("[bench] note: fewer than 3 warm-up steps requested")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return 0
        return reference_arm(args)

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    import __graft_entry__ as g
    if rank == 0:
        g.build()
    if world > 1:
        dist.barrier()

    from eals_cpp_b200.model import MF_fastALS, SparseMat
    spec, sm, test_items = build_workload(args.workload, local_rank)
    M, N, K, nnz = spec["M"], spec["N"], spec["K"], sm.nnz
    fals = MF_fastALS(sm, None, topK=spec["topK"], factors=K, showLoss=False, init=False, device=local_rank)
    U0, V0 = random_factors(M, N, K, local_rank)
    fals.setUV(U0, V0)
    del U0, V0
    torch.cuda.empty_cache()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def epoch():
        fals.update_user()
        fals.update_item()

    for _ in range(args.warmup):
        epoch()
    barrier()
    fals.timings_total(reset=True)
    launches0 = fals.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        barrier()
        e0.record()
        for _ in range(args.steps):
            epoch()
        e1.record()
        barrier()
    ms_total = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:     # before anything else trains the factors further
        dump_outputs(fals, args.dump_outputs)
    if world > 1:
        t = torch.tensor([ms_total], device=f"cuda:{local_rank}", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / args.steps
    launches = fals.kernel_launches() - launches0
    detail_ms = fals.timings_detail()
    phase_ms, phase_calls = fals.timings_total(reset=True)
    value = 2.0 * nnz * K / (ms_step * 1e-3)
    per_rank = None
    if world > 1:       # every rank's own phase timers: load balance of the partition (DESIGN.md §6)
        mine = torch.tensor([phase_ms[k] / args.steps for k in ("user_sweep", "user_gram", "item_sweep", "item_gram")],
                            device=f"cuda:{local_rank}", dtype=torch.float64)
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = {k: [round(float(a[i]), 3) for a in allr] for i, k in enumerate(("user_sweep", "user_gram", "item_sweep", "item_gram"))}

    # roofline of the dominant kernel family: the CD sweeps (this rank's owned rows)
    peaks, peak_src = measured_peaks()
    ub, ue = fals.user_bounds[rank], fals.user_bounds[rank + 1]
    ib, ie = fals.item_bounds[rank], fals.item_bounds[rank + 1]
    nnz_u = int(sm.row_ptr[ue] - sm.row_ptr[ub])
    nnz_i = int(sm.col_ptr[ie] - sm.col_ptr[ib])
    alg_bytes = cd_bytes_per_epoch(M, N, K, nnz_u, nnz_i, ue - ub, ie - ib)
    sweep_ms = (phase_ms["user_sweep"] + phase_ms["item_sweep"]) / args.steps
    achieved = alg_bytes / (sweep_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if world == 1 and os.path.exists(tpath):      # the ncu capture is a 1-GPU whole-epoch figure; per-rank traffic was not captured
        try:
            with open(tpath) as f:
                traffic = json.load(f).get(args.workload, {}).get("cd_sweep_dram_bytes_per_epoch")
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": "cd_sweep (user + item CD sweep kernels of one epoch)",
                "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                "traffic": traffic, "algorithmic_bytes": alg_bytes, "kernel_ms": sweep_ms, "peak_source": peak_src}
    floor = fp64_pipe_floor_ms(nnz_u + nnz_i, K, sms=torch.cuda.get_device_properties(local_rank).multi_processor_count)
    roofline["fp64_pipe"] = {"bound": "fp64 pipe (DMMA.884: 5 per 4 nonzeros and 16-factor block, 16.1 SMSP cycles each, measured)",
                             "floor_ms": floor, "frac": floor / sweep_ms,
                             "hbm_floor_ms": alg_bytes / (peaks["hbm_gbs"] * 1e9) * 1e3}

    loss = fals.loss()
    replicas_ok = fals.replicas_consistent()    # every rank's U and V replicas bit-identical (hash on device)

    # ---- e2e: through the public API with HOST buffers -------------------------------------------------
    e2e = None
    if not args.no_e2e:
        def pinned(t):
            h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            h.copy_(t)
            return h
        keep = [pinned(x) for x in (sm.row_ptr, sm.col_idx, sm.col_ptr, sm.row_idx)]
        sm_host = SparseMat(M, N, *[k.numpy() for k in keep])
        own_u = int(sm.row_ptr[ue] - sm.row_ptr[ub]); own_i = int(sm.col_ptr[ie] - sm.col_ptr[ib])
        h2d = (own_u + own_i) * 4 + (ue - ub + 1 + ie - ib + 1) * 8      # what the library uploads per step
        times, parts = [], []
        for it in range(1 + args.e2e_steps):
            barrier()
            t0 = time.perf_counter()
            fals.setTrain(sm_host)          # H2D of the CSR + CSC arrays, bucketing, position maps
            h2d = getattr(fals, "_h2d_bytes_last", h2d)   # several ranks: 1/world chunk each + all-gather
            torch.cuda.synchronize(); t1 = time.perf_counter()
            epoch()
            torch.cuda.synchronize(); t2 = time.perf_counter()
            _ = fals.loss()                 # D2H of the step's result
            barrier()
            t3 = time.perf_counter()
            if it > 0:
                times.append(t3 - t0)
                parts.append((t1 - t0, t2 - t1, t3 - t2))
        t_e2e = float(np.mean(times))
        e2e_parts = dict(zip(("set_train_s", "epoch_s", "loss_s"), np.mean(np.asarray(parts), axis=0).tolist()))
        if world > 1:
            t = torch.tensor([t_e2e, float(h2d)], device=f"cuda:{local_rank}", dtype=torch.float64)
            tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            t_e2e, h2d = float(tmax[0].item()), int(t[1].item())
        e2e = {"value": 2.0 * nnz * K / t_e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": 32 * world, "s_per_step": t_e2e, "steps": args.e2e_steps,
               "what": "setTrain(host pinned CSR+CSC) + update_user + update_item + loss() per step",
               "breakdown": e2e_parts}
        del keep, sm_host

    # ---- CPU baseline (rank 0, N = 1 only) ------------------------------------------------------------------
    cpu = None
    if not args.no_cpu and world == 1:
        try:
            from oracle import bindings
            if bindings.reference_available(fast=True):     # the reference's own code, 1 thread, bounded row sample
                ep, sample = cpu_reference_sampled(sm, M, N, K, args.cpu_nnz or int(4.0e7 / K), 2, 0)
                cpu = {"value": 2.0 * nnz * K / ep, "unit": UNIT, "cores": 1, "kind": "reference", "sample": sample,
                       "epoch_s_extrapolated": ep}
            else:
                threads = os.cpu_count() or 1
                cpu = cpu_port_sample(sm, K, 0.01, 10.0, 0.75, max(min(nnz // 2, 4_000_000), 1000), threads)
        except Exception as e:      # the baseline must never take the GPU number down with it
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": f"failed: {e!r}"}

    # ---- the other BASELINE.json configurations, driver-visible: c1 / c2 / c3 epochs, C5 evaluation ---------------
    configs = None
    if not args.no_configs:
        configs = {}
        if args.workload in ("c4", "c4s") and test_items is not None:
            # configs[4]: full-catalogue leave-one-out evaluate, top-100, on the model the timed epochs trained
            gt = test_items.cpu().numpy().astype(np.int32) if hasattr(test_items, "cpu") else np.asarray(test_items, np.int32)
            ev = []
            for _ in range(2):
                barrier(); t0 = time.perf_counter()
                res = fals.evaluate(gt, spec["topK"])
                barrier(); ev.append(time.perf_counter() - t0)
            st = fals.eval_stats()
            flop = 2.0 * M * N * K
            configs["c5_evaluate"] = {
                "what": f"leave-one-out evaluate(), top-{spec['topK']}, all {M} users x {N} items, reference-compatible ranking, on the "
                        f"factors after {args.warmup + args.steps + (args.e2e_steps + 1 if not args.no_e2e else 0)} epochs",
                "seconds": ev[-1], "first_call_seconds": ev[0], "hr_ndcg_rr": [float(x) for x in res],
                "engine": st["engine"], "candidate_users_this_rank": st["candidates"], "pairs_rescored_fp64_this_rank": st["pairs_rescored"],
                "candidate_fraction_this_rank": st["candidates"] / max(1, fals.user_bounds[rank + 1] - fals.user_bounds[rank]),
                "dense_equivalent_tflops": flop / ev[-1] / 1e12,
                "roofline": None if "first_block" not in st else {
                    "bound": "tensor", "kernel": "eval_filter_kernel (tcgen05.mma fp16 -> fp32 in TMEM), first item block of this rank: "
                                                 f"{st['first_block']['users']} users x {st['first_block']['items']} items",
                    "achieved": st["first_block"]["tflops"], "unit": "TFLOP/s", "peak": peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]),
                    "frac": st["first_block"]["tflops"] / peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]),
                    "kernel_ms": st["first_block"]["ms"], "peak_source": peak_src + " — sustained bf16 figure: the kernel runs inside a long step"},
                "note": "tcgen05 fp16 filter with a rigorous error bound decides the clear cases (users leave the working set once "
                        "more than topK items certainly beat the held-out one); every close call is re-scored in fp64; "
                        "dense_equivalent_tflops counts 2*M*N*K although decided users skip the rest of the catalogue"}
        for name in ("c3", "c1", "c2"):
            if args.workload == name or (world > 1 and name != "c3"):
                continue
            try:
                sp2, sm2, _ = build_workload(name, local_rank)
                f2 = MF_fastALS(sm2, None, topK=sp2["topK"], factors=sp2["K"], showLoss=False, init=False, device=local_rank)
                U2, V2 = random_factors(sp2["M"], sp2["N"], sp2["K"], local_rank)
                f2.setUV(U2, V2)
                del U2, V2
                for _ in range(3):
                    f2.update_user(); f2.update_item()
                barrier()
                f2.timings_total(reset=True)
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
                n_ep = 10
                for _ in range(n_ep):
                    f2.update_user(); f2.update_item()
                a1.record()
                barrier()
                ms2 = a0.elapsed_time(a1) / n_ep
                if world > 1:
                    t = torch.tensor([ms2], device=f"cuda:{local_rank}", dtype=torch.float64)
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                    ms2 = float(t.item())
                ph, _ = f2.timings_total(reset=True)
                ms_graph = None
                if world == 1:      # the same epochs replayed as ONE captured CUDA graph (launch-bound small configs gain most)
                    f2.run_epochs(3, graph=True)
                    torch.cuda.synchronize()
                    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    g0.record()
                    f2.run_epochs(n_ep, graph=True)
                    g1.record()
                    torch.cuda.synchronize()
                    ms_graph = g0.elapsed_time(g1) / n_ep
                ub2, ue2 = f2.user_bounds[rank], f2.user_bounds[rank + 1]
                ib2, ie2 = f2.item_bounds[rank], f2.item_bounds[rank + 1]
                nu2 = int(sm2.row_ptr[ue2] - sm2.row_ptr[ub2]); ni2 = int(sm2.col_ptr[ie2] - sm2.col_ptr[ib2])
                by2 = cd_bytes_per_epoch(sp2["M"], sp2["N"], sp2["K"], nu2, ni2, ue2 - ub2, ie2 - ib2)
                sw2 = (ph["user_sweep"] + ph["item_sweep"]) / n_ep
                configs[name] = {"workload": workload_string(name, sp2, sm2.nnz), "epoch_ms": ms2, "epoch_ms_cuda_graph": ms_graph,
                                 "value_cuda_graph": None if ms_graph is None else 2.0 * sm2.nnz * sp2["K"] / (ms_graph * 1e-3),
                                 "value": 2.0 * sm2.nnz * sp2["K"] / (ms2 * 1e-3), "unit": UNIT, "sweep_ms": sw2,
                                 "hbm_frac": by2 / (sw2 * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                 "working_set_fits_l2": (sp2["M"] + sp2["N"]) * sp2["K"] * 8 + sm2.nnz * 8 < 126e6, "loss_after": f2.loss(), "epochs_timed": n_ep}
                f2.close()
                del f2, sm2
                torch.cuda.empty_cache()
            except Exception as e:       # a side measurement must never take the headline down with it
                configs[name] = {"error": repr(e)}

    if configs is not None and world == 1 and args.workload in ("c4", "c4s"):
        # the reference's own factor initialisation at this scale (DenseMat.cpp:54-62: one sequential libstdc++ stream;
        # ours is the same stream generated in parallel by LCG skip-ahead, bit-identical) — LAST, it overwrites the factors
        try:
            t0 = time.perf_counter()
            stream_s = fals.init_factors()
            configs["c4_init_factors"] = {"seconds": time.perf_counter() - t0, "host_stream_seconds": stream_s,
                                          "values": max(M, N) * K, "host_threads": min(32, os.cpu_count() or 1),
                                          "what": "eals_init_factors: libstdc++ minstd_rand0 + polar normal stream, bit-identical to the reference, + upload + initS"}
        except Exception as e:
            configs["c4_init_factors"] = {"error": repr(e)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_string(args.workload, spec, nnz),
                       "step": "one eALS epoch = update_user + update_item incl. S-cache Gram and (N>1) exchange",
                       "parallelism": f"users/items sharded over {world} GPU(s), U/V replicated",
                       "l2": "inputs (>= 12 GB of factors + 4 GB of indices) far exceed the 126 MB L2; no flush needed"
                             if args.workload in ("c4", "c4s", "c3") else "working set fits L2: latency/launch-bound",
                       "baseline_note": "BASELINE.md's only published figure (8.16e7 /s) is the reference on real yelp.rating, K=64, 1 CPU thread — a different config"},
            "clocks": clk.summary(), "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": cpu,
            "phase_ms_per_step": {k: v / args.steps for k, v in phase_ms.items() if phase_calls[k]},
            "sweep_detail_ms_per_step": {k: v / args.steps for k, v in detail_ms.items()},
            "per_rank_phase_ms_per_step": per_rank,
            "loss_after": loss, "replicas_consistent": replicas_ok,
            "configs": configs,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def reference_arm(args):
    """The reference's own CPU implementation of the same path on the host cores: the real MF_fastALS object
    from oracle/_ref (the reference's translation units compiled where they lie, -O3), ONE thread — the
    reference has no working threading (SURVEY.md §0.3) — timed through its own sweep + S-patch calls.
    Workloads it can hold (c1 / c2 / small) run whole epochs; for the large ones every step is a bounded
    row sample of the same matrix (see cpu_reference_sampled) and `value` is the throughput measured on it.
    The oracle port on every host core is printed beside it as a labelled "modified reference" figure.
    Nothing of the product (libeals_b200.so) is loaded here."""
    from oracle import bindings
    bindings.build("port")
    bindings.build("ref")
    from eals_cpp_b200 import datasets
    from eals_cpp_b200.model import SparseMat
    name = args.workload
    spec = dict(datasets.WORKLOADS[name])
    M, N, K = spec["M"], spec["N"], spec["K"]
    small = spec["nnz"] <= 2_000_000
    threaded = None
    # without the reference's sources oracle/_ref is not built: its C restatement stands in, labelled "port"
    kind = "reference" if bindings.reference_available(fast=True) else "port"
    if small:
        data = datasets.powerlaw_csr(**spec)
        sm = SparseMat.from_csr(data.M, data.N, data.row_ptr, data.col_idx)
        nnz = sm.nnz
        if kind == "reference":
            epoch_s = cpu_reference_full(sm, K, args.steps, min(args.warmup, 1))
            sample = f"oracle/_ref (reference TUs, g++ -O3), whole epochs incl. S patches, 1 thread, mean of {args.steps}"
        else:
            epoch_s = cpu_port_full(sm, K, args.steps, min(args.warmup, 1))
            sample = f"oracle port (eals_oracle.c, gcc -O2), whole epochs incl. S patches, 1 thread, mean of {args.steps}"
        step_s = epoch_s
    else:
        import torch
        assert torch.cuda.is_available(), "the large synthetic workloads are generated on the GPU (torch: plumbing)"
        _, sm, _ = build_workload(name, 0)
        nnz = sm.nnz
        target = args.cpu_nnz or int(6.4e7 / K)
        t0 = time.perf_counter()
        if kind == "reference":
            epoch_s, sample = cpu_reference_sampled(sm, M, N, K, target, args.steps, min(args.warmup, 1))
        else:
            r = cpu_port_sample(sm, K, 0.01, 10.0, 0.75, target, 1)
            epoch_s, sample = r["epoch_s_extrapolated"], r["sample"]
        step_s = (time.perf_counter() - t0) / (args.steps + min(args.warmup, 1))
        try:
            r = cpu_port_sample(sm, K, 0.01, 10.0, 0.75, min(nnz // 2, 4_000_000), os.cpu_count() or 1)
            threaded = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port (modified reference: threaded, S patch excluded)",
                        "sample": r["sample"]}
        except Exception as e:      # pragma: no cover
            threaded = {"value": None, "sample": f"failed: {e!r}"}
    value = 2.0 * nnz * K / epoch_s
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_s * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_string(name, spec, nnz),
                   "step": "one eALS epoch = update_user + update_item incl. the S-cache patches" +
                           ("" if small else " — measured on a bounded row sample per step, value = throughput on the sample scaled to the whole matrix")},
        "epoch_ms_whole_matrix": epoch_s * 1e3,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": kind, "sample": sample},
        "cpu_baseline_threaded_port": threaded,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
