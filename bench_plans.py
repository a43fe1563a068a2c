#!/usr/bin/env python
"""bench_plans.py — time StochGPMPBatch.best_plans (collision check + choice of each problem's plan) at the benchmark shapes.

    python bench_plans.py [--runs 25] [--warmup 5] [--iters 3]

Panda C4 (bench.py's flagship workload: 4096 problems x 4 particles, T = 64, 5 spheres per problem, fp32): a few optimize()
iterations, then best_plans at n_interp = 0, 4, 8, 16.  Planar C2 (1024 problems x 4 particles, T = 64, per-problem occupancy
maps): best_plans at n_interp = 8.  Each time is the median of --runs calls between CUDA events after --warmup calls, and is
printed next to the time of one optimize() iteration of the same planner (same events, same count), the card's name and its
power limit.  One JSON line per shape.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _median_ms(fn, runs, warmup):
    import torch
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(runs):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    times.sort()
    return times[len(times) // 2]


def _power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=25)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--iters", type=int, default=3, help="optimize() iterations before the plans are chosen")
    args = ap.parse_args()
    if args.runs < 20:
        raise SystemExit("--runs must be >= 20")
    import torch
    import bench
    if not torch.cuda.is_available():
        raise SystemExit("bench_plans.py needs a CUDA device")
    dev = torch.device("cuda:0")
    card = dict(gpu=torch.cuda.get_device_name(0), power_limit_w=_power_limit_w())
    for name, B, n_interps in (("panda", 4096, (0, 4, 8, 16)), ("planar", 1024, (8,))):
        w = bench.workload(name, B)
        pl = bench.build_planner(w, B, dev)
        obs = {}
        if w["spheres"] is not None:
            obs["obstacle_spheres"] = torch.tensor(w["spheres"], device=dev, dtype=torch.float32)
        pl.optimize(opt_iters=args.iters, **obs)
        means = pl.particle_means.clone()
        t_iter = _median_ms(lambda: pl.optimize(opt_iters=1, **obs), args.runs, args.warmup)
        pl.particle_means = means
        rows = {}
        for m in n_interps:
            t = _median_ms(lambda: pl.best_plans(n_interp=m, **obs), args.runs, args.warmup)
            r = pl.best_plans(n_interp=m, **obs)
            rows[str(m)] = dict(ms=round(t, 4), collision_free=int(r.collision_free.sum().item()))
        print(json.dumps(dict(workload=w["name"], problems=B, particles=pl.num_particles, T=w["T"], best_plans_ms_by_n_interp=rows,
                              optimize_iteration_ms=round(t_iter, 4), runs=args.runs, warmup=args.warmup, **card)), flush=True)


if __name__ == "__main__":
    main()
