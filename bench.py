#!/usr/bin/env python
"""bench.py -- benchmark of the ScaML-GP hot path (BASELINE.json metric, configs 3 / 4 / 5).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--metric evals|posterior]
                  [--dump-outputs DIR]

Headline (`--metric evals`, the default): config 3 of BASELINE.json -- **4096 meta-tasks in total** x n=256 x d=6,
R=6 hyper-parameter rows per task (1 warm start + 5 prior samples, reference scamlgp/utils.py:173-203).  A "step" is
one pass of the fused LML+grad kernel over every (task, row) followed by the scalar LML / failure-count reduction.
With N GPUs the 4096 tasks are block-partitioned over the ranks exactly as `scamlgp_b200.sharded.task_partition`
does it behind `ShardedSources` (tasks factor independently: reference scamlgp/model.py:176-188), every rank runs
its block, and ONE all_reduce(sum) over [sum LML, #failed] is the only collective (north_star item 5) -- STRONG
scaling of a fixed-size problem.  `value` = evaluations of all ranks / max-over-ranks device time with inputs
resident in HBM; `e2e` = the same through the engine call with pinned HOST buffers (H2D of this rank's X, Y, theta and
D2H of lml, grad inside the timed region).  Weak scaling (every rank a full 4096-task batch, no collective) is
reported beside it under `weak_scaling`.

Further legs on the same line: `posterior` (second half of the metric, config 5: weighted mean + variance of the
4096 base GPs at 1 Mi candidates, tasks sharded, candidates replicated, one all_reduce over [2, B]), `config4`
(16384 tasks x n=512 x d=10, blocked DMMA Cholesky), `kernel_matrix` (stand-alone assembly,
HBM-bound), `conditioned` and `acq_grad` (target-GP conditioning and analytic candidate gradients).
`--metric posterior` prints the posterior leg as its own line (same contract) so that the driver can pair it with
`--impl reference --metric posterior`.

`--impl reference` times the reference's CPU path (the oracle restatement of its botorch/gpytorch arithmetic -- those
packages cannot be installed here, SURVEY 8c) on the box's host cores in the reference's own parallel style: one
single-threaded process per core over disjoint task slices (scamlgp/benchmarking/local_runner.py:107-108,174-181).

`--dump-outputs DIR` writes what the last timed step of the printed metric computed, gathered over all ranks, as
DIR/<name>.npy in float64: for `evals` lml [4096, 6], grad [4096, 6, 8], info [4096, 6] (0 = factorised) and
stats [2] (sum of LML, failed rows); for `posterior` mean and var [candidates] (8 MB each at 1 Mi candidates).  The
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

M_TASKS, R_ROWS, N_PTS, DIM = 4096, 6, 256, 6
WORKLOAD = ("config3: 4096 meta-tasks in total x n=256 x d=6, R=6 hyper-parameter rows/task, LML+grad; "
            "tasks block-partitioned over the GPUs (strong scaling)")
C4_TASKS, C4_R, C4_N, C4_D, C4_BLOCK = 16384, 2, 512, 10, 2048
C5_CANDIDATES = 1 << 20
POST_WORKLOAD = ("config5: weighted posterior mean+variance of 4096 fitted base GPs (n=256, d=6) at 1048576 "
                 "acquisition candidates (q=1); tasks block-partitioned over the GPUs, candidates replicated")
CSRC = os.path.join(ROOT, "scalable-meta-learning-with-gaussian-processes_b200", "csrc")


def config_of(metric: str) -> dict:
    """The `config` object of the JSON line: names the workload, identical in both arms (details of a run -- shard
    sizes, checks, samples -- go under `details` / `cpu_baseline.sample`)."""
    if metric == "posterior":
        return {"workload": POST_WORKLOAD, "tasks_total": M_TASKS, "n": N_PTS, "d": DIM, "candidates": C5_CANDIDATES}
    return {"workload": WORKLOAD, "tasks_total": M_TASKS, "rows_per_task": R_ROWS, "n": N_PTS, "d": DIM}


def algorithmic_flops(n: int, d: int) -> float:
    """SURVEY 8d: F_lml = n^3 + n^2 (5d/2 + 10) flop per evaluation."""
    return float(n) ** 3 + float(n) ** 2 * (2.5 * d + 10.0)


def point_flops(n: int, d: int) -> float:
    """SURVEY 8d: F_pt = n^2 + n (3d + 12) flop per (task, candidate) posterior point (mean + variance)."""
    return float(n) ** 2 + float(n) * (3.0 * d + 12.0)


# --------------------------------------------------------------------------------------- #
# CPU side (oracle) -- used for cpu_baseline and for --impl reference
# --------------------------------------------------------------------------------------- #
_CPU_JOB = {}


def _cpu_worker(args):
    lo, hi = args
    import torch

    from oracle import scaml_oracle as O

    torch.set_num_threads(1)
    X, Yt, th, spec = _CPU_JOB["X"], _CPU_JOB["Yt"], _CPU_JOB["th"], _CPU_JOB["spec"]
    R = th.shape[1]
    t0 = time.perf_counter()
    acc = 0.0
    for e in range(lo, hi):
        m, r = divmod(e, R)
        v, g = O.lml_and_grad_autograd(X[m], Yt[m], th[m, r], spec, mode="expansion")
        acc += float(v)
    return hi - lo, time.perf_counter() - t0, acc


def _cpu_post_worker(args):
    """Reference-style posterior of the source GPs: Python loop over tasks (scamlgp/model.py:128-134), each a
    kernel row block, an alpha dot and a triangular solve for the variance."""
    lo, hi = args
    import torch

    from oracle import scaml_oracle as O

    torch.set_num_threads(1)
    states, Xc = _CPU_JOB["states"], _CPU_JOB["Xc"]
    t0 = time.perf_counter()
    acc = 0.0
    for m in range(lo, hi):
        mu, var = O.posterior(states[m], Xc)
        acc += float(mu[0]) + float(var[0])
    return (hi - lo) * Xc.shape[0], time.perf_counter() - t0, acc


class CpuReference:
    """Reference-style CPU evaluation of LML+grad / posterior on a bounded sample of the workload."""

    def __init__(self, tasks: int, cores: int, candidates: int = 2048):
        import torch

        import datagen
        from oracle import scaml_oracle as O

        torch.set_num_threads(1)
        self.cores, self.tasks, self.candidates = cores, tasks, candidates
        X, Y = datagen.synthetic_tasks(tasks, N_PTS, DIM, seed=0)
        spec = O.HyperSpec.source()
        Yt = torch.stack([O.standardize(Y[m])[0] for m in range(tasks)])
        th = datagen.sample_theta_raw(tasks, R_ROWS, DIM, spec, seed=0)
        g = torch.Generator().manual_seed(5)
        _CPU_JOB.update(X=X, Yt=Yt, th=th, spec=spec,
                        states=[O.factorize(X[m], Y[m], th[m, 0], spec) for m in range(tasks)],
                        Xc=torch.rand(candidates, DIM, dtype=torch.float64, generator=g))
        import multiprocessing as mp

        self.pool = mp.get_context("fork").Pool(cores)
        self.evals = tasks * R_ROWS

    def step(self) -> float:
        """Evaluates the whole sample once across the pool; returns wall seconds."""
        per = (self.evals + self.cores - 1) // self.cores
        chunks = [(i, min(i + per, self.evals)) for i in range(0, self.evals, per)]
        t0 = time.perf_counter()
        self.pool.map(_cpu_worker, chunks)
        return time.perf_counter() - t0

    def posterior_step(self) -> float:
        per = (self.tasks + self.cores - 1) // self.cores
        chunks = [(i, min(i + per, self.tasks)) for i in range(0, self.tasks, per)]
        t0 = time.perf_counter()
        self.pool.map(_cpu_post_worker, chunks)
        return time.perf_counter() - t0

    def posterior_points_per_s(self, passes: int = 2) -> dict:
        """points/s of the per-task posterior (mean + variance) on the same sample of tasks."""
        self.posterior_step()  # warm-up
        dt = sum(self.posterior_step() for _ in range(passes))
        return {"value": self.tasks * self.candidates * passes / dt, "unit": "points/s", "cores": self.cores,
                "kind": "port", "sample": self.posterior_sample(passes)}

    def posterior_sample(self, passes: int) -> str:
        return (f"{self.tasks} of {M_TASKS} fitted tasks (n={N_PTS}, d={DIM}) x {self.candidates} of {C5_CANDIDATES} "
                f"candidates, oracle posterior mean+variance per task, {self.cores} single-threaded processes, "
                f"{passes} timed passes")

    def sequential_evals_per_s(self, evals: int = 192) -> dict:
        """BASELINE.md section 2, CPU mode 1: the reference's own loop (scamlgp/model.py:176) -- ONE process, tasks one
        after another, torch's default intra-op threads."""
        import torch

        from oracle import scaml_oracle as O

        X, Yt, th, spec = _CPU_JOB["X"], _CPU_JOB["Yt"], _CPU_JOB["th"], _CPU_JOB["spec"]
        threads = max(1, min(self.cores, os.cpu_count() or 1))
        torch.set_num_threads(threads)
        try:
            evals = min(evals, self.evals)
            for e in range(4):  # warm-up
                O.lml_and_grad_autograd(X[e // R_ROWS], Yt[e // R_ROWS], th[e // R_ROWS, e % R_ROWS], spec, mode="expansion")
            t0 = time.perf_counter()
            for e in range(evals):
                m, r = divmod(e, R_ROWS)
                O.lml_and_grad_autograd(X[m], Yt[m], th[m, r], spec, mode="expansion")
            dt = time.perf_counter() - t0
        finally:
            torch.set_num_threads(1)
        return {"value": evals / dt, "unit": "evals/s", "cores": threads, "kind": "port",
                "sample": f"{evals} evaluations one after another in one process, {threads} intra-op threads "
                          "(the reference's sequential task loop, model.py:176)"}

    def close(self):
        self.pool.close()
        self.pool.join()


def host_cores() -> int:
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def cpu_sample_tasks(cores: int) -> int:
    # ~6 evaluations/task; aim at roughly 2-3 s of wall per step with ~5 ms per evaluation
    return max(8, min(M_TASKS, cores * 128 // R_ROWS))


# --------------------------------------------------------------------------------------- #
# clocks
# --------------------------------------------------------------------------------------- #
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return

        def rd():
            for line in self.proc.stdout:
                self.rows.append(line.strip())

        self.thread = threading.Thread(target=rd, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for row in self.rows:
            f = [x.strip() for x in row.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------- #
def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    tasks = cpu_sample_tasks(cores)
    if args.metric == "posterior":
        ref = CpuReference(tasks, cores, candidates=2048)
        for _ in range(args.warmup):
            ref.posterior_step()
        times = [ref.posterior_step() for _ in range(args.steps)]
        ref.close()
        total = sum(times)
        value = tasks * ref.candidates * args.steps / total
        sample = ref.posterior_sample(args.steps)
        metric, unit, workload = "posterior points/s over all tasks", "points/s", POST_WORKLOAD
    else:
        ref = CpuReference(tasks, cores)
        for _ in range(args.warmup):
            ref.step()
        times = [ref.step() for _ in range(args.steps)]
        ref.close()
        total = sum(times)
        value = ref.evals * args.steps / total
        sample = (f"{tasks} of {M_TASKS} tasks x R={R_ROWS} rows per step, oracle LML + autograd gradient "
                  f"(gpytorch-style expansion distances), {cores} single-threaded processes")
        metric, unit, workload = "meta-task LML+grad evals/s (n=256,d=6)", "evals/s", WORKLOAD
    line = {
        "impl": "reference", "metric": metric, "value": value, "unit": unit,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_of(args.metric),
        "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def _sha16(paths) -> str:
    h = hashlib.sha256()
    for p in paths:
        with open(os.path.join(CSRC, p), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def ncu_traffic(kernel: str):
    """(DRAM bytes read + written per launch of `kernel`, stale?) from the committed ncu capture
    (profiles/ncu_traffic.json).  Every entry is stamped with a hash of the kernel's source files at capture time;
    when the sources have changed since, the number describes an older kernel and `traffic_stale` says so."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f)[kernel]
        total = float(t["dram_bytes_read"]) + float(t["dram_bytes_write"])
        stale = ("source_sha16" not in t) or (t["source_sha16"] != _sha16(t.get("sources", [])))
        return total, bool(stale), t.get("launch")
    except Exception:
        return None, True, None


def measure_fp64_peak(torch, lib_path: str, device) -> dict:
    """Live FP64 denominators: register-resident DFMA chains and DMMA chains."""
    import ctypes as C

    L = C.CDLL(lib_path)
    L.scaml_microbench_fp64.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_double), C.c_void_p]
    blocks = 148 * 8
    out = torch.empty(blocks * 256, dtype=torch.float64, device=device)
    res = {}
    stream = torch.cuda.current_stream(device).cuda_stream
    for mode, name, iters in ((0, "dfma", 4000), (1, "dmma_m8n8k4", 4000), (2, "dmma_m16n8k16", 2000)):
        flops = C.c_double(0.0)
        best = 0.0
        for rep in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = L.scaml_microbench_fp64(mode, blocks, iters, out.data_ptr(), C.byref(flops), stream)
            e1.record()
            torch.cuda.synchronize(device)
            if rc != 0:
                break
            ms = e0.elapsed_time(e1)
            if rep > 0:
                best = max(best, flops.value / (ms * 1e-3) / 1e12)
        res[name] = best
    # library DGEMM for reference (BASELINE.md: "quote roofline fractions of measured DGEMM / DFMA")
    try:
        n = 8192
        a = torch.randn(n, n, dtype=torch.float64, device=device)
        b = torch.randn(n, n, dtype=torch.float64, device=device)
        torch.matmul(a, b)
        best = 0.0
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            torch.cuda.synchronize(device)
            best = max(best, 2.0 * n ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        res["cublas_dgemm_8192"] = best
        del a, b
    except Exception:
        res["cublas_dgemm_8192"] = None
    return res


def measured_hbm_gbs():
    """Copy bandwidth of this pool's B200s (driver-written MEASURED_PEAKS.json), else the profiling guide's fallback."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (torch copy, read+write bytes)"
    except Exception:
        return 6550.0, "fallback of /opt/skills/guides/B200_PROFILING.md (no MEASURED_PEAKS.json)"


def dump_outputs(out_dir: str, arrays: dict) -> None:
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.detach().cpu().double().numpy())


def run_ours(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = host_cores()
    full = not args.quick

    # CPU baseline first (fork-based pool must be created before CUDA is initialised)
    cpu_baseline = cpu_posterior = cpu_sequential = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        tasks = cpu_sample_tasks(cores)
        ref = CpuReference(tasks, cores)
        ref.step()  # warm-up
        ts = [ref.step() for _ in range(3)]
        cpu_posterior = None if args.no_posterior else ref.posterior_points_per_s()
        cpu_sequential = ref.sequential_evals_per_s()
        ref.close()
        cpu_baseline = {
            "value": ref.evals * len(ts) / sum(ts), "unit": "evals/s", "cores": cores, "kind": "port",
            "sample": f"{tasks} of {M_TASKS} tasks x R={R_ROWS}, oracle LML+autograd grad (expansion distances), "
                      f"{cores} single-threaded processes, {len(ts)} timed passes",
        }

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a CUDA device; there is no CPU fallback. "
                         "Use --impl reference for the CPU baseline.")
    torch.cuda.set_device(local_rank)
    device = torch.device(f"cuda:{local_rank}")
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    import datagen  # synthetic inputs only; the product arm imports nothing from oracle/
    from scamlgp_b200 import HyperSpec
    from scamlgp_b200._capi import CUDA_LIB_PATH
    from scamlgp_b200.engine import Engine, SourceBatch
    from scamlgp_b200.sharded import task_partition

    eng = Engine(device)
    spec = HyperSpec.source()
    M, R, n, d = M_TASKS, R_ROWS, N_PTS, DIM
    lo, hi = task_partition(M, world)[rank]
    Ml = hi - lo
    X, Y = datagen.synthetic_tasks(M, n, d, seed=0)  # the SAME 4096 tasks whatever N is
    th = datagen.sample_theta_raw(M, R, d, spec, seed=0)
    hX, hY, hT = X[lo:hi].contiguous().pin_memory(), Y[lo:hi].contiguous().pin_memory(), th[lo:hi].contiguous().pin_memory()
    batch = SourceBatch.from_padded(hX.to(device), hY.to(device))
    thd = hT.to(device).contiguous()
    lml = torch.empty(Ml, R, dtype=torch.float64, device=device)
    grad = torch.empty(Ml, R, d + 2, dtype=torch.float64, device=device)
    info = torch.empty(Ml, R, dtype=torch.int32, device=device)
    stats = torch.zeros(2, dtype=torch.float64, device=device)  # [sum of LML, failed rows] over ALL tasks
    h_lml = torch.empty(Ml, R, dtype=torch.float64).pin_memory()
    h_grad = torch.empty(Ml, R, d + 2, dtype=torch.float64).pin_memory()
    h_stats = torch.empty(2, dtype=torch.float64).pin_memory()
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=device)  # 256 MB > 126 MB L2

    peaks = measure_fp64_peak(torch, CUDA_LIB_PATH, device) if rank == 0 else {}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    dumps = {}  # --dump-outputs: the last timed step's results, copied before later legs reuse the buffers

    def all_tasks(t):
        """This rank's block of tasks -> all M tasks on rank 0, None on the others (blocks may differ in size)."""
        if world == 1:
            return t.clone()
        parts = [None] * world if rank == 0 else None
        dist.gather_object(t.cpu(), parts, dst=0)
        return torch.cat(parts) if rank == 0 else None

    def reduce_stats(l, i):
        # the scalar LML / failure-count reduction of a sharded fit (SURVEY 8e): local sums, one all_reduce
        stats[0] = torch.nan_to_num(l, nan=0.0).sum()
        stats[1] = (i != 0).sum()
        if world > 1:
            dist.all_reduce(stats, op=dist.ReduceOp.SUM)

    def step_resident():
        l, g, i = eng.lml_grad_raw(batch, thd, spec, out=(lml, grad, info))
        reduce_stats(l, i)

    # e2e: host buffers in, host buffers out, every step.  The inputs are double-buffered on the device and the H2D copy
    # of step i + 1 is issued on a second stream while step i computes (the copy engines run beside the SMs), so a
    # step costs max(copy, compute) instead of their sum; each step still moves its full inputs and reads its results.
    copy_stream = torch.cuda.Stream(device)
    dbuf = [[torch.empty_like(hX, device=device), torch.empty_like(hY, device=device), torch.empty_like(hT, device=device),
             torch.cuda.Event(), torch.cuda.Event()] for _ in range(2)]  # X, Y, theta, `copied`, `consumed`
    e2e_state = {"i": 0, "primed": False}

    def e2e_prefetch(slot):
        bx, by, bt, copied, consumed = dbuf[slot]
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed)  # the step that last read this slot has finished with it
            bx.copy_(hX, non_blocking=True)
            by.copy_(hY, non_blocking=True)
            bt.copy_(hT, non_blocking=True)
            copied.record(copy_stream)

    def step_e2e():
        cur = torch.cuda.current_stream(device)
        i = e2e_state["i"]
        if not e2e_state["primed"]:
            for sl in range(2):
                dbuf[sl][4].record(cur)
            e2e_prefetch(i & 1)
            e2e_state["primed"] = True
        bx, by, bt, copied, consumed = dbuf[i & 1]
        e2e_prefetch((i + 1) & 1)  # next step's inputs: overlaps this step's kernel
        cur.wait_event(copied)
        b = SourceBatch.from_padded(bx, by)
        l, g, ii = eng.lml_grad_raw(b, bt, spec, out=(lml, grad, info))
        consumed.record(cur)
        reduce_stats(l, ii)
        h_lml.copy_(l, non_blocking=True)
        h_grad.copy_(g, non_blocking=True)
        h_stats.copy_(stats, non_blocking=True)
        cur.synchronize()
        e2e_state["i"] = i + 1

    def timed(fn, steps, warmup, do_flush=True):
        for _ in range(warmup):
            fn()
        barrier()
        launches0 = eng.launches
        evs = []
        for _ in range(steps):
            if do_flush:
                flush.zero_()  # evict L2 between timed iterations
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            evs.append((e0, e1))
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), eng.launches - launches0

    # ---- cross-rank identity: a block of another rank's tasks re-evaluated here must match it bit for bit ---- #
    def cross_rank_check():
        if world == 1:
            return None
        eng.lml_grad_raw(batch, thd, spec, out=(lml, grad, info))
        k = min(16, Ml)
        mine = torch.cat([lml[:k].reshape(-1), grad[:k].reshape(-1)]).contiguous()
        gathered = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)
        peer = (rank + 1) % world
        plo = task_partition(M, world)[peer][0]
        pb = SourceBatch.from_padded(X[plo:plo + k].to(device), Y[plo:plo + k].to(device))
        pl, pg, _ = eng.lml_grad_raw(pb, th[plo:plo + k].to(device).contiguous(), spec)
        same = bool(torch.equal(torch.cat([pl.reshape(-1), pg.reshape(-1)]), gathered[peer]))
        t = torch.tensor([int(same)], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return "bit-identical" if int(t.item()) == 1 else "MISMATCH"

    # ---- second half of BASELINE.json's metric: posterior points/s over all tasks (config 5) -------------- #
    def posterior_bench(full_size: bool):
        """Weighted ScaML-GP prior prediction (mean + variance reduced over the rank's block of the 4096 fitted
        base GPs inside the kernel, then ONE all_reduce(sum) over [2, B]) at B replicated candidates; one "point" =
        one (task, candidate) pair.  Config 5 asks for B = 1 Mi: each timed step covers all of them (warm-up on 3
        slices of 2 x 148 x 64 candidates)."""
        B_SLICE = 2 * 148 * 64
        B_STEP = C5_CANDIDATES if full_size else B_SLICE
        fs = eng.factorize(batch, thd[:, 0].contiguous(), spec)
        w = torch.full((Ml,), 1.0 / M, dtype=torch.float64, device=device)
        g = torch.Generator().manual_seed(100)  # the SAME candidates on every rank
        hXc = torch.rand(B_STEP, d, dtype=torch.float64, generator=g).pin_memory()
        Xc = hXc.to(device)
        part = torch.empty(2, B_STEP, dtype=torch.float64, device=device)
        h_out = torch.empty(2, B_STEP, dtype=torch.float64).pin_memory()

        def predict(xc, out):
            eng.predict_weighted(fs, w, xc, out=(out[0, :xc.shape[0]], out[1, :xc.shape[0]]))

        def step_res():
            predict(Xc, part)
            if world > 1:  # sum of weighted predictions over the task shards (north_star item 5)
                dist.all_reduce(part, op=dist.ReduceOp.SUM)

        def step_kernel_only():
            predict(Xc, part)

        def step_e2e():
            xc = hXc.to(device, non_blocking=True)
            predict(xc, part)
            if world > 1:
                dist.all_reduce(part, op=dist.ReduceOp.SUM)
            h_out.copy_(part, non_blocking=True)
            torch.cuda.current_stream(device).synchronize()

        for _ in range(3):  # warm-up slices
            predict(Xc[:B_SLICE], part)
        if args.metric == "posterior":  # the printed metric: --steps timed steps, resident and end to end
            psteps = esteps = args.steps
        else:  # a side leg of the evals line
            psteps = (1 if world == 1 else 2) if full_size else max(2, min(args.steps, 4))
            esteps = 1 if full_size else psteps
        ms_r, nl = timed(step_res, psteps, 0 if full_size else 1)
        if args.dump_outputs and args.metric == "posterior":  # `part` holds the prediction over all tasks
            dumps.update(mean=part[0].clone(), var=part[1].clone())
        ms_k = timed(step_kernel_only, 1, 0)[0] if world > 1 else ms_r / psteps  # per step, kernel alone
        ms_e, _ = timed(step_e2e, esteps, 0)  # leaves the all-reduced prediction in `part`
        finite = bool(torch.isfinite(part).all() and (part[1] > 0).all())
        # replicated-candidate check: the all-reduced prediction equals ONE GPU holding all 4096 tasks (first 512
        # candidates), to rounding of the cross-rank summation order
        check = None
        if world > 1:
            ball = SourceBatch.from_padded(X.to(device), Y.to(device))
            fall = eng.factorize(ball, th[:, 0].to(device).contiguous(), spec)
            wall = torch.full((M,), 1.0 / M, dtype=torch.float64, device=device)
            rm, rv = eng.predict_weighted(fall, wall, Xc[:512].contiguous())
            em = float((part[0, :512] - rm).abs().max() / rm.abs().max())
            ev = float((part[1, :512] - rv).abs().max() / rv.abs().max())
            t = torch.tensor([em, ev], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            check = {"candidates": 512, "mean_rel_err": float(t[0]), "var_rel_err": float(t[1]),
                     "ok": bool(t[0] < 1e-12 and t[1] < 1e-12)}
            del ball, fall
        ok_info = int((fs.info == 0).all())
        pts = float(M) * B_STEP  # (task, candidate) pairs of the WHOLE job per step
        Fp = point_flops(n, d)
        ach = float(Ml) * B_STEP * Fp / (ms_k * 1e-3) / 1e12  # this GPU's kernel
        traffic, stale, tl = ncu_traffic("scaml_predict_kernel<RBF>")
        out = {"metric": "posterior points/s over all tasks", "value": pts * psteps / (ms_r * 1e-3),
               "unit": "points/s", "ms_per_step": ms_r / psteps, "steps": psteps, "n_gpus": world, "scaling": "strong",
               "config": config_of("posterior") if full_size else
               {"workload": f"config5 slice: {M} fitted base GPs x {B_STEP} candidates per step (--quick)"},
               "details": {"candidates_per_step": B_STEP, "tasks_per_gpu": Ml,
                          "factor_info_zero": bool(ok_info), "finite": finite,
                          "l2": "per-step inputs (this rank's packed factors: %.2f GB) exceed the 126 MB L2" %
                                (fs.linv.numel() * 8 / 1e9),
                          "replicated_candidates_check": check},
               "e2e": {"value": pts * esteps / (ms_e * 1e-3), "unit": "points/s",
                       "h2d_bytes_per_step": int(hXc.numel()) * 8, "d2h_bytes_per_step": int(h_out.numel()) * 8,
                       "collective": "all_reduce(sum) [2,B] fp64 over ranks" if world > 1 else None},
               "gpu_launches": nl,
               "phase_ms": {"predict_kernel": ms_k,
                            "all_reduce_[2,B]": max(0.0, ms_r / psteps - ms_k) if world > 1 else 0.0},
               "roofline": {"bound": "tensor", "pipe": "FP64 tensor cores (DMMA)", "achieved": ach,
                            "unit": "TFLOP/s", "flops_per_point": Fp, "traffic": traffic, "traffic_stale": stale,
                            "traffic_launch": tl, "traffic_unit": "DRAM bytes per launch (ncu)",
                            "algorithmic_bytes": 8.0 * (Ml * (n * n / 2 + n * d + n) * 2 + B_STEP * (d + 2)),
                            "kernel": "scaml_predict_kernel<RBF>"}}
        return out, fs, Xc

    def conditioned_and_grad(fs, Xc):
        """Target-GP legs at n_t = 32 target points on this rank's tasks: fused conditioned prediction (prior mean /
        variance + cross-covariance, DESIGN 3.3b) and one value + analytic-gradient evaluation at 64 candidates."""
        B_SLICE = 2 * 148 * 64
        Xs = Xc[:B_SLICE].contiguous()
        w = torch.full((Ml,), 1.0 / M, dtype=torch.float64, device=device)
        n_t = 32
        g = torch.Generator().manual_seed(101)
        Xt = torch.rand(n_t, d, dtype=torch.float64, generator=g).to(device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        eng.cond_prepare(fs, Xt)
        e0.record()
        A = eng.cond_prepare(fs, Xt)
        e1.record()
        torch.cuda.synchronize(device)
        ms_prep = e0.elapsed_time(e1)
        ms_c, _ = timed(lambda: eng.predict_conditioned(fs, w, Xs, Xt, A), 2, 1)
        Bg = 64
        Yt = torch.sin(3.0 * Xt).sum(1)
        Yall = torch.cat([batch.Y_raw.reshape(-1), Yt])
        mu_a, s_a = float(Yall.mean()), float(Yall.std())
        smn, scv = eng.cond_caches(fs, Xt, A)
        tsp = HyperSpec.target()
        tht = datagen.initial_theta_raw(d, tsp).to(device)
        tstate = eng.target_factorize(smn, scv, Xt, ((Yt - mu_a) / s_a).contiguous(), w, tht, mu_a, s_a, tsp)
        del smn, scv
        Xg = Xc[:Bg].contiguous()

        def step_grad():
            U = eng.cond_prepare(fs, Xg)
            a_, b_, c_ = eng.values_from_u(fs, w, Xg, U, Xt, A)
            _, _, beta = eng.target_posterior_beta(tstate, a_, b_, c_, Xg)
            return eng.posterior_grad(fs, w, Xg, U, tstate, A, beta)

        ms_g, nl_g = timed(step_grad, 3, 2)
        gdm, gdv = step_grad()
        grad_finite = bool(torch.isfinite(gdm).all() and torch.isfinite(gdv).all()) and tstate.info == 0
        peak = peaks.get("dfma", 0.0) or None
        # algorithmic flop per (task, candidate): prior point + the k*^T A_m contraction (2 n n_t)
        Fc = point_flops(n, d) + 2.0 * n * n_t
        ach_c = float(Ml) * B_SLICE * Fc / (ms_c / 2 * 1e-3) / 1e12
        # value + gradient: K_m^-1 k* (2 n^2), mix (2 n n_t), contraction n (5 d + 45), values from U (2 n (n_t + 1) + n (3d + 12))
        Fg = 2.0 * n * n + 2.0 * n * n_t + n * (5.0 * d + 45.0) + 2.0 * n * (n_t + 1) + n * (3.0 * d + 12.0)
        ach_g = float(Ml) * Bg * Fg / (ms_g / 3 * 1e-3) / 1e12
        tr_c, st_c, tl_c = ncu_traffic("scaml_predict_kernel<RBF,64,CROSS>")
        tr_p, st_p, tl_p = ncu_traffic("scaml_cond_prepare_kernel<RBF>")
        cond = {"n_t": n_t, "value": float(Ml) * B_SLICE * 2 / (ms_c * 1e-3), "unit": "points/s (this GPU's tasks)",
                "ms_per_step": ms_c / 2, "prepare_ms": ms_prep, "candidates_per_step": B_SLICE,
                "what": "weighted prior mean/variance + cross-covariance with n_t target inputs (fused)",
                "roofline": {"bound": "tensor", "achieved": ach_c, "peak": peak, "unit": "TFLOP/s",
                             "frac": (ach_c / peak) if peak else None, "flops_per_point": Fc,
                             "kernel": "scaml_predict_kernel<RBF,64,CROSS>", "traffic": tr_c, "traffic_stale": st_c,
                             "traffic_launch": tl_c}}
        acq = {"n_t": n_t, "candidates": Bg, "ms_per_step": ms_g / 3, "gpu_launches": nl_g // 3,
               "value": float(Ml) * Bg * 3 / (ms_g * 1e-3), "unit": "(task, candidate) gradients/s (this GPU's tasks)",
               "finite": grad_finite,
               "what": "posterior value + analytic d mean/dx, d var/dx (conditioned on n_t target points): "
                       "cond_prepare at the candidates, values from U, beta, DMMA mix, gradient contraction",
               "roofline": {"bound": "tensor", "achieved": ach_g, "peak": peak, "unit": "TFLOP/s",
                            "frac": (ach_g / peak) if peak else None, "flops_per_point": Fg,
                            "kernel": "scaml_cond_prepare_kernel<RBF> (dominant) + grad kernels", "traffic": tr_p,
                            "traffic_stale": st_p, "traffic_launch": tl_p,
                            "traffic_note": "DRAM bytes of the dominant kernel only (cond_prepare, 64-column panel)"}}
        return cond, acq

    # ---- config 4: 16384 tasks x n = 512 x d = 10, blocked DMMA Cholesky (4-warp kernel, 3 CTAs/SM) ---- #
    def config4_bench():
        nblocks = C4_TASKS // C4_BLOCK
        if nblocks % world != 0:
            return {"skipped": f"{nblocks} task blocks do not divide over {world} ranks"}
        mine = list(range(rank * nblocks // world, (rank + 1) * nblocks // world))
        Xs, Ys, Ts = [], [], []
        for b in mine:  # block b of the global data set has its own seed: the SAME 16384 tasks whatever N is
            xb, yb = datagen.synthetic_tasks(C4_BLOCK, C4_N, C4_D, seed=1000 + b)
            Xs.append(xb)
            Ys.append(yb)
            Ts.append(datagen.sample_theta_raw(C4_BLOCK, C4_R, C4_D, spec, seed=1000 + b))
        b4 = SourceBatch.from_padded(torch.cat(Xs).to(device), torch.cat(Ys).to(device))
        t4 = torch.cat(Ts).to(device).contiguous()
        del Xs, Ys, Ts
        M4 = b4.M
        o4 = (torch.empty(M4, C4_R, dtype=torch.float64, device=device),
              torch.empty(M4, C4_R, C4_D + 2, dtype=torch.float64, device=device),
              torch.empty(M4, C4_R, dtype=torch.int32, device=device))

        def step4():
            l, g, i = eng.lml_grad_raw(b4, t4, spec, out=o4)
            reduce_stats(l, i)

        ms4, nl4 = timed(step4, 3, 3)
        ok4 = int((o4[2] == 0).all())
        F4 = algorithmic_flops(C4_N, C4_D)
        ach = float(M4) * C4_R * F4 / (ms4 / 3 * 1e-3) / 1e12
        peak = peaks.get("dfma", 0.0) or None
        traffic, stale, tl = ncu_traffic("scaml_fit_kernel<RBF> config4")
        out = {"metric": "meta-task LML+grad evals/s (n=512,d=10)", "value": float(C4_TASKS) * C4_R * 3 / (ms4 * 1e-3),
               "unit": "evals/s", "ms_per_step": ms4 / 3, "steps": 3, "n_gpus": world, "scaling": "strong",
               "config": {"workload": f"config4: {C4_TASKS} meta-tasks in total x n={C4_N} x d={C4_D}, R={C4_R} rows/task, "
                                      "blocked DMMA Cholesky (4-warp kernel), tasks block-partitioned over the GPUs",
                          "tasks_per_gpu": M4, "all_info_zero": bool(ok4)},
               "gpu_launches": nl4,
               "roofline": {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                            "frac": (ach / peak) if peak else None, "flops_per_eval": F4,
                            "kernel": "scaml_fit_kernel<RBF> (4-warp; 3 CTAs/SM)", "traffic": traffic, "traffic_stale": stale,
                            "traffic_launch": tl}}
        del b4, t4, o4
        return out

    # ---- north_star item 1: stand-alone batched kernel-matrix assembly (HBM-bound) --------------------------- #
    def kmat_bench():
        thc = torch.rand(Ml, d + 2, dtype=torch.float64, device=device) * 0.5 + 0.25
        K = torch.empty(Ml, n, n, dtype=torch.float64, device=device)
        ms, nl = timed(lambda: eng.kernel_matrix(batch.X, thc, 0, out=K), 5, 3)
        bytes_alg = float(Ml) * n * n * 8 + float(Ml) * n * d * 8
        hbm, src = measured_hbm_gbs()
        ach = bytes_alg / (ms / 5 * 1e-3) / 1e9
        traffic, stale, tl = ncu_traffic("scaml_kmat_kernel<RBF>")
        del K
        return {"metric": "kernel-matrix assembly GB/s", "value": ach, "unit": "GB/s (this GPU)", "ms_per_step": ms / 5,
                "config": {"workload": f"{Ml} tasks x {n}x{n} fp64 K stored, ARD-RBF, d={d}"}, "gpu_launches": nl,
                "roofline": {"bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
                             "peak_source": src, "algorithmic_bytes": bytes_alg, "traffic": traffic,
                             "traffic_stale": stale, "traffic_launch": tl, "kernel": "scaml_kmat_task_kernel<RBF>"}}

    # ------------------------------------------------------------------------------------------------------ #
    if args.metric == "posterior":
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        post, fs, Xc = posterior_bench(full)
        clocks = sampler.stop() if rank == 0 else None
        if rank == 0:
            pk = peaks.get("dfma", 0.0) or None
            post["roofline"]["peak"] = pk
            post["roofline"]["frac"] = (post["roofline"]["achieved"] / pk) if pk else None
            post["roofline"]["peak_source"] = "live register-resident DFMA microbench in this run"
            post.update({"warmup": 3, "higher_is_better": True, "vs_baseline": None, "dtype": "f64",
                         "data": "synthetic", "clocks": clocks})
            if cpu_posterior is not None:
                post["cpu_baseline"] = cpu_posterior
            if args.dump_outputs:
                dump_outputs(args.dump_outputs, dumps)
            print(json.dumps(post), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    xcheck = cross_rank_check()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_res, launches = timed(step_resident, args.steps, max(3, args.warmup))
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dumps.update(lml=all_tasks(lml), grad=all_tasks(grad), info=all_tasks(info), stats=stats.clone())
    e2e_steps = max(2, min(args.steps, 5))
    ms_e2e, _ = timed(step_e2e, e2e_steps, 2)
    ok = int((info == 0).all())
    # per-phase breakdown of the resident step: the kernel alone vs kernel + local sums + all_reduce
    ms_kernel, _ = timed(lambda: eng.lml_grad_raw(batch, thd, spec, out=(lml, grad, info)), max(3, min(args.steps, 10)), 1)
    ksteps = max(3, min(args.steps, 10))
    # weak scaling beside it: every rank evaluates a FULL 4096-task batch, no collective
    weak = None
    if world > 1 and not args.no_weak:
        bw = SourceBatch.from_padded(X.to(device), Y.to(device))
        tw = th.to(device).contiguous()
        ow = (torch.empty(M, R, dtype=torch.float64, device=device),
              torch.empty(M, R, d + 2, dtype=torch.float64, device=device),
              torch.empty(M, R, dtype=torch.int32, device=device))
        ms_w, _ = timed(lambda: eng.lml_grad_raw(bw, tw, spec, out=ow), 5, 3)
        weak = {"value": float(M) * R * world * 5 / (ms_w * 1e-3), "unit": "evals/s", "tasks_per_gpu": M,
                "ms_per_step": ms_w / 5, "scaling": "weak", "collective": None}
        del bw, tw, ow
    if world > 1:
        okt = torch.tensor([ok], device=device)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        ok = int(okt.item())

    posterior = conditioned = acq = None
    if not args.no_posterior:
        posterior, fs, Xc = posterior_bench(full)
        conditioned, acq = conditioned_and_grad(fs, Xc)
        del fs, Xc
    config4 = config4_bench() if full else None
    kmat = kmat_bench()

    if rank == 0:
        evals_per_step = M * R  # the whole job: all 4096 tasks, whatever N is
        value = evals_per_step * args.steps / (ms_res * 1e-3)
        e2e_value = evals_per_step * e2e_steps / (ms_e2e * 1e-3)
        F = algorithmic_flops(n, d)
        kernel_ms = ms_kernel / ksteps  # the dominant kernel alone (max over ranks)
        achieved = Ml * R * F / (kernel_ms * 1e-3) / 1e12  # this GPU's launch
        peak = peaks.get("dfma", 0.0) or None
        traffic, stale, tl = ncu_traffic("scaml_fit_kernel<RBF>")
        line = {
            "metric": "meta-task LML+grad evals/s (n=256,d=6)", "value": value, "unit": "evals/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_res / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_of("evals"),
            "details": {"tasks_per_gpu": Ml, "l2": "256 MB flush buffer written between timed iterations",
                       "parallelism": f"task-sharded x{world} (scamlgp_b200.sharded.task_partition); per step one "
                                      "all_reduce(sum) over [sum LML, #failed rows]" if world > 1 else
                                      "1 GPU; per step the local [sum LML, #failed rows] reduction",
                       "all_info_zero": bool(ok), "cross_rank_check": xcheck},
            "e2e": {"value": e2e_value, "unit": "evals/s",
                    "h2d_bytes_per_step": int(hX.numel() + hY.numel() + hT.numel()) * 8 * world,
                    "d2h_bytes_per_step": int(h_lml.numel() + h_grad.numel() + 2) * 8 * world, "steps": e2e_steps,
                    "overlap": "inputs double-buffered on the device; the H2D copy of step i+1 runs on a second stream "
                               "under the kernel of step i; every step copies its full inputs and reads its results back",
                    "note": "bytes summed over ranks (every rank copies its own block)"},
            "gpu_launches": launches,
            "phase_ms": {"lml_grad_kernel": kernel_ms, "scalar_reduce_and_all_reduce": max(0.0, ms_res / args.steps - kernel_ms),
                         "limiting": "lml_grad_kernel"},
            "roofline": {"bound": "tensor", "pipe": "FP64 tensor cores (mma.sync f64 -> DMMA; shares its pipe with DFMA)",
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": (achieved / peak) if peak else None,
                         "traffic": traffic, "traffic_stale": stale, "traffic_launch": tl,
                         "traffic_unit": "DRAM bytes per launch (ncu)",
                         "algorithmic_bytes": 8.0 * Ml * (n * d + n + R * (2 * (d + 2) + 1)),
                         "kernel": "scaml_fit_kernel<RBF>", "flops_per_eval": F, "evals_per_launch": Ml * R,
                         "peak_source": "live register-resident DFMA microbench in this run "
                                        "(MEASURED_PEAKS.json has no FP64 entry)",
                         "fp64_peaks_tflops": peaks},
            "clocks": clocks,
        }
        if weak is not None:
            line["weak_scaling"] = weak
        if posterior is not None:
            pk = peak
            posterior["roofline"]["peak"] = pk
            posterior["roofline"]["frac"] = (posterior["roofline"]["achieved"] / pk) if pk else None
            if cpu_posterior is not None:
                posterior["cpu_baseline"] = cpu_posterior
            posterior["conditioned"] = conditioned
            posterior["acq_grad"] = acq
            line["posterior"] = posterior
        if config4 is not None:
            line["config4"] = config4
        line["kernel_matrix"] = kmat
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
            line["cpu_baseline_sequential"] = cpu_sequential
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dumps)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps of the printed metric (default 20; for --impl ours --metric posterior 1, 2 on "
                         "several GPUs, 4 with --quick)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--metric", choices=["evals", "posterior"], default="evals",
                    help="which half of BASELINE.json's metric the printed line is about")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-posterior", action="store_true", help="skip the posterior / conditioned / gradient legs")
    ap.add_argument("--no-weak", action="store_true", help="skip the weak-scaling side measurement (N > 1)")
    ap.add_argument("--quick", action="store_true",
                    help="profiling runs: posterior leg on a 18944-candidate slice instead of 1 Mi, no config-4 leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps is None:
        if args.impl == "ours" and args.metric == "posterior":
            # one full-size step (4096 tasks x 1 Mi candidates) takes about 12 s on one B200 at a 1000 W power limit
            args.steps = 4 if args.quick else (1 if int(os.environ.get("WORLD_SIZE", "1")) == 1 else 2)
        else:
            args.steps = 20
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
