"""Cost of batch (q > 1) acquisition at 4096 meta-tasks x n = 256 x d = 6 with n_t = 32 target observations.

  1. one qUCB value + gradient evaluation at 32 blocks x q = 4 (ScaMLGP.posterior_blocks + its VJP),
  2. in the same run, the q = 1 UpperConfidenceBound.value_and_grad at 128 candidates (the same number of points),
  3. one ScaMLGPBO.generate_evaluation_specifications(4) against four generate_evaluation_specification() calls
     (each one conditioned on the points already pending).
Device events around every timed call, after warm-up; medians over the repetitions.  Prints one JSON line per
measurement and the GPU's name and power limit.

    python scripts/qbatch_bench.py [--tasks 4096] [--n 256] [--d 6] [--nt 32] [--reps 20]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def timed(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tasks", type=int, default=4096)
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--d", type=int, default=6)
    ap.add_argument("--nt", type=int, default=32)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--bo-reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("qbatch_bench.py measures the GPU: no CUDA device")
    import __graft_entry__ as g

    g.build()
    from datagen import synthetic_tasks
    from scamlgp_b200.optimizer import ScaMLGPBO
    from scamlgp_b200.space import ContinuousParameter, Evaluation, Objective, ParameterSpace
    from scamlgp_b200.utils import UpperConfidenceBound, qUpperConfidenceBound

    name, pl = gpu_info()
    M, n, d, nt = args.tasks, args.n, args.d, args.nt
    print(json.dumps({"gpu": name, "power_limit": pl, "tasks": M, "n": n, "d": d, "n_t": nt}), flush=True)
    X, Y = synthetic_tasks(M, n, d, seed=0)
    Xn, Yn = X.numpy(), Y.numpy()
    space = ParameterSpace()
    for k in range(d):
        space.add(ContinuousParameter(f"x{k}", (0.0, 1.0)))
    keys = [f"x{k}" for k in range(d)]
    t0 = time.time()
    md = {m: [Evaluation(configuration=dict(zip(keys, map(float, Xn[m, i]))), objectives={"loss": float(Yn[m, i])})
              for i in range(n)] for m in range(M)}
    opt = ScaMLGPBO(space, Objective("loss", greater_is_better=False), md, seed=0, max_pending_evaluations=8)
    rng = np.random.default_rng(1)
    evs = []
    for _ in range(nt):
        c = dict(zip(keys, map(float, rng.uniform(0, 1, d))))
        evs.append(Evaluation(configuration=c, objectives={"loss": float(np.sin(3 * np.array(list(c.values()))).sum())}))
    opt.report(evs)
    torch.cuda.synchronize()
    print(json.dumps({"setup_s": round(time.time() - t0, 2)}), flush=True)
    model = opt.model
    gen = torch.Generator().manual_seed(2)

    # 1 + 2: one value-and-gradient evaluation, q = 4 blocks vs q = 1 at the same number of points
    Xb = torch.rand(32, 4, d, dtype=torch.float64, generator=gen)
    X1 = Xb.reshape(128, d).clone()
    qucb, ucb = qUpperConfidenceBound(model), UpperConfidenceBound(model)
    res = {}
    for rnd in range(2):  # alternate the two, twice
        res.setdefault("qucb_q4_32blocks_value_and_grad_ms", []).append(timed(lambda: qucb.value_and_grad(Xb),
                                                                              args.reps))
        res.setdefault("ucb_q1_128cand_value_and_grad_ms", []).append(timed(lambda: ucb.value_and_grad(X1), args.reps))
    for k, v in res.items():
        print(json.dumps({"metric": k, "median_ms": [round(x[0], 3) for x in v], "min_ms": [round(x[1], 3) for x in v],
                          "max_ms": [round(x[2], 3) for x in v], "reps": args.reps}), flush=True)

    # 3: one joint batch of 4 vs four sequential proposals (kriging-believer fantasies of the pending points)
    def batch():
        opt.generate_evaluation_specifications(4)
        opt.pending_specifications.clear()

    def sequential():
        for _ in range(4):
            opt.generate_evaluation_specification()
        opt.pending_specifications.clear()

    bo = {}
    for rnd in range(args.bo_reps):
        for k, fn in (("generate_evaluation_specifications_q4_s", batch), ("four_sequential_proposals_s", sequential)):
            torch.cuda.synchronize()
            t = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            bo.setdefault(k, []).append(time.perf_counter() - t)
    for k, v in bo.items():
        print(json.dumps({"metric": k, "runs_s": [round(x, 3) for x in v], "median_s": round(float(np.median(v)), 3)}),
              flush=True)


if __name__ == "__main__":
    main()
