#!/usr/bin/env python
"""bench.py — StochGPMP hot-path benchmark (driver contract + tier keys: roofline, cpu_baseline, e2e).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|reference-cuda] [--workload panda|planar]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

metric   trajectory-samples/s per optimize() iteration (BASELINE.json), whole job over all ranks.
step     ONE optimize() iteration of the hot path over the whole problem batch (the reference's examples
         call optimize() with opt_iters=1 in a loop: examples/panda_environment.py:141-146).
workload BASELINE.json configs[3], "Panda 7-DoF batched: 4096 problems x 4 goals x 512 particles x traj_len 64, sharded by
         problem at 1/2/4/8 B200".  N=1: all 4096 problems on one B200.  N>1: the SAME 4096 problems, 4096/N per GPU
         (STRONG scaling, --scaling weak keeps 4096 per GPU), sharded by problem with no data-path collective; RNG streams
         are keyed by global problem ids, so every N computes the identical plan.
value    inputs resident in HBM, fused kernel only (CUDA events around each step, L2 flushed between steps).
e2e      same metric through the public API (StochGPMPBatch.optimize) from HOST buffers: per step the
         observation (obstacle spheres) is copied H2D from pinned memory and the plan (particle means) is
         read back D2H, both inside the timed region (host clock).  The batch is sharded into --e2e-shards
         StochGPMPBatch objects on their own streams so that a shard's D2H overlaps the next shard's kernel;
         the host waits for every shard at the end of every step.
dump     --dump-outputs DIR writes what the last timed step returned (see dump_outputs) as DIR/<name>.npy, so that two builds
         run with the same arguments can be compared output for output: the inputs are seeded and identical from run to run.
extra    N=1: `configs` (C1 planar as shipped fp64, C2 planar 1024 problems, C3 Panda single problem) and `soft_regime` (C4 at a
         temperature with ESS >> 1: the second RNG sweep of the update is no longer skipped).  N>1: `weak` (4096 problems per
         GPU) and `split` (BASELINE configs[4]: the samples of every particle divided over the N ranks, NCCL all_gather of the
         weighted statistics issued from C; checked against the un-split loop in fp64).
The reference arm (--impl reference) times the reference's CPU algorithm (oracle/reference_port.py, pinned to
the real reference by tests/test_reference_port.py; the reference itself is pure Python and does not travel
to the GPU box) on the host cores, on a bounded sample of the same workload.  --impl reference-cuda runs the same
dense torch formulation with its tensors on cuda:0 (stock cuBLAS / cuSOLVER path: "what device='cuda' buys").
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "trajectory_samples_per_s_per_iteration"
UNIT = "traj-samples/s"
DUMP_BYTES = 60 * 10 ** 6           # --dump-outputs stays under 64 MB: a larger batch is sampled by problem


# ------------------------------------------------------------------------------------------------ workload
def workload(name, B):
    """Shapes, sigmas and synthetic inputs (SURVEY §8d: C4 Panda batched / C2 planar batched)."""
    import numpy as np
    from stoch_gpmp_b200 import scenarios as sc
    if name == "panda":
        start, goals, spheres = sc.panda_batch(B, G=4, O=5, seed0=0)
        return dict(name="panda_7dof_batched", n_dof=7, T=64, dt=0.05, G=4, K=1, S=512, temperature=1.0, step_size=0.1,
                    start=start, goals=goals, spheres=spheres, sig=sc.PANDA_SIGMAS, cost=sc.PANDA_COST, n_links=11, O=5)
    if name == "planar":
        start, goals = sc.planar_batch(B, G=4, seed0=0)
        return dict(name="planar_2dof_batched", n_dof=2, T=64, dt=0.02, G=4, K=1, S=256, temperature=1.0, step_size=0.5,
                    start=start, goals=goals, spheres=None, sig=sc.PLANAR_SIGMAS, cost=sc.PLANAR_COST, n_links=0, O=0)
    if name == "planar_shipped":        # C1: examples/planar_environment.py as shipped (one problem, fp64, seed 0)
        start = np.array([[-9., -9., 0., 0.]])
        goals = np.array([sc.PLANAR_GOALS], dtype=np.float64)
        return dict(name="planar_2dof_shipped_fp64", n_dof=2, T=64, dt=0.02, G=3, K=5, S=128, temperature=1.0, step_size=0.5,
                    start=start, goals=goals, spheres=None, sig=sc.PLANAR_SIGMAS, cost=sc.PLANAR_COST, n_links=0, O=0, f64=True)
    raise SystemExit("unknown workload %r" % name)


def algorithmic_flops_per_traj(w):
    """ALGORITHMIC FP32 flops per trajectory-sample-iteration (FMA = 2), SURVEY §8(d) constants:
    banded sampling 16 T n; GP factor 10 (T-1) n; start+goal 6 d; IS dot 2 M; softmax/update 2 M + 10;
    Panda: FK (specialised z-axis chain) (7*36 + 3*18)(T-1); sphere RBF 10 L O (T-1);
    planar: map index arithmetic 10 (T-1).  MUFU ops (sin/cos, exp, Box-Muller) are counted separately."""
    T, n = w["T"], w["n_dof"]
    d, M = 2 * n, 2 * n * T
    f = 16 * T * n + 10 * (T - 1) * n + 6 * d + 2 * M + 2 * M + 10
    mufu = 0
    if w["spheres"] is not None:
        f += (7 * 36 + 3 * 18) * (T - 1) + 10 * w["n_links"] * w["O"] * (T - 1)
        mufu += 14 * (T - 1) + w["n_links"] * w["O"] * (T - 1)
    else:
        f += 10 * (T - 1)
    mufu += 2 * M          # Box-Muller: ~2 MUFU-class ops per normal (log, sqrt, sin, cos shared by a pair)
    return f, mufu


def build_planner(w, B, dev, problem_offset=0, seed=0, temperature=None):
    import torch
    from stoch_gpmp_b200.costs.cost_functions import CostCollision, CostComposite, CostGP, CostGoalPrior
    from stoch_gpmp_b200.costs.fields import LinkDistanceField
    from stoch_gpmp_b200.planner import StochGPMPBatch
    from stoch_gpmp_b200.robots import PandaFK
    ta = {"device": dev, "dtype": torch.float64 if w.get("f64") else torch.float32}
    n, T, K, S = w["n_dof"], w["T"], w["K"], w["S"]
    s = torch.tensor(w["start"], **ta)
    g = torch.tensor(w["goals"], **ta)
    cl = [CostGP(n, T, s, w["dt"], dict(sigma_start=w["cost"]["sigma_start"], sigma_gp=w["cost"]["sigma_gp"]), ta),
          CostGoalPrior(n, T, multi_goal_states=g, num_particles_per_goal=K, num_samples=S,
                        sigma_goal_prior=w["cost"]["sigma_goal_prior"], tensor_args=ta)]
    FK = None
    if w["spheres"] is not None:
        FK = PandaFK()
        cl.append(CostCollision(n, T, field=LinkDistanceField(tensor_args=ta), sigma_coll=w["cost"]["sigma_coll"]))
    else:
        import random
        import numpy as np
        from stoch_gpmp_b200.envs.map_generator import generate_obstacle_map
        maps = []
        for b in range(min(16, B)):     # 16 distinct 200x200 maps cycled over the problems (C1: the seed-0 map of the example)
            random.seed(1000 + b if B > 1 else 0)
            np.random.seed(1000 + b if B > 1 else 0)
            maps.append(generate_obstacle_map(map_dim=[20, 20], cell_size=0.1, random_gen=True, num_obst=15,
                                              rand_limits=[[-7.5, 7.5], [-7.5, 7.5]], rand_rect_shape=[2, 2], tensor_args=ta)[0])
        cl.append(CostCollision(n, T, field=[maps[b % len(maps)] for b in range(B)] if B > 1 else maps[0], sigma_coll=w["cost"]["sigma_coll"]))
    cost = CostComposite(n, T, cl, FK=FK, tensor_args=ta)
    return StochGPMPBatch(num_particles_per_goal=K, num_samples=S, traj_len=T, opt_iters=1, dt=w["dt"], n_dof=n,
                          step_size=w["step_size"], temperature=w["temperature"] if temperature is None else temperature,
                          start_state=s, multi_goal_states=g,
                          initial_particle_means="const_vel", cost=cost, seed=seed, tensor_args=ta,
                          problem_offset=problem_offset, **w["sig"])


# -------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.proc.wait()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in self.rows if len(r) >= 9 for k in range(4) if r[5 + k].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------ reference arm
def cpu_reference_time(w, n_problems, iters, warmup, device="cpu"):
    """Seconds per iteration of ONE problem for the reference's algorithm (oracle/reference_port.py) on `device`."""
    import numpy as np
    import torch
    from oracle import fk as OFK
    from oracle.reference_port import time_port
    spec = dict(n_dof=w["n_dof"], T=w["T"], dt=w["dt"], G=w["G"], K=w["K"], S=w["S"], temperature=w["temperature"],
                step_size=w["step_size"], start=np.asarray(w["start"][0]), goals=np.asarray(w["goals"][0]),
                cost_sigma_start=w["cost"]["sigma_start"], cost_sigma_gp=w["cost"]["sigma_gp"],
                sigma_goal_prior=w["cost"]["sigma_goal_prior"], sigma_coll=w["cost"]["sigma_coll"], **w["sig"])
    fk = None
    dtype = torch.float32
    if w["spheres"] is not None:
        spec["spheres"] = np.asarray(w["spheres"][0])
        fk = OFK.fk_all_links_torch()
    else:
        spec["sigma_coll"] = None        # planar CPU sample: GP + goal factors (the reference needs fp64 here)
        dtype = torch.float64
    return time_port(spec, dtype, n_problems, iters, warmup, fk=fk, device=device)


def run_reference(args, rank, world):
    if rank != 0:
        return
    cuda = args.impl == "reference-cuda"
    w = workload(args.workload, 1)
    t0 = time.time()
    sec, cores = cpu_reference_time(w, 1, args.steps, args.warmup, device="cuda:0" if cuda else "cpu")
    ntraj = w["G"] * w["K"] * w["S"]
    val = ntraj / sec
    sample = "%d timed optimize() iterations (+%d warm-up) of 1 problem of the workload (G=%d,K=%d,S=%d,T=%d,n=%d), %s" % (
        args.steps, args.warmup, w["G"], w["K"], w["S"], w["T"], w["n_dof"], "fp32" if w["spheres"] is not None else "fp64")
    where = ("its tensors on cuda:0 — stock torch CUDA ops (cuBLAS bmm / cuSOLVER potrf+trsm), informational: what device='cuda' buys the "
             "reference's formulation; none of this repo's kernels run" if cuda else "torch CPU, all host threads")
    line = {"impl": args.impl, "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32" if w["spheres"] is not None else "f64", "data": "synthetic",
            "config": {"workload": w["name"], "problems_per_step": 1, "goals": w["G"], "particles_per_goal": w["K"] * w["S"],
                       "traj_len": w["T"], "n_dof": w["n_dof"], "note": "reference algorithm (oracle/reference_port.py; the "
                       "pure-Python reference does not travel to the GPU box), " + where},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.time() - t0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
NOMINAL_FP32_TFLOPS = 74.4     # 148 SM x 128 lanes x 2 x 1.965 GHz (SURVEY §6)
NOMINAL_MUFU_TOPS = 4.65       # 148 SM x 16 x 1.965 GHz


def probe_peaks(dev):
    """Measured FP32-FMA and MUFU pipe peaks (the denominators MEASURED_PEAKS.json lacks)."""
    import torch
    from stoch_gpmp_b200 import _lib
    lib = _lib.load()
    scratch = torch.zeros(16, device=dev)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = {}
    blocks = torch.cuda.get_device_properties(dev).multi_processor_count * 8
    for mode, name, per_thread_iter in ((0, "fp32_tflops", 128 * 2), (1, "mufu_tops", 64)):
        iters = 2000
        _lib.check(lib.sgpmp_probe(mode, blocks, 200, ctypes.c_void_p(scratch.data_ptr()), st), "probe")
        best = 0.0
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.check(lib.sgpmp_probe(mode, blocks, iters, ctypes.c_void_p(scratch.data_ptr()), st), "probe")
            e1.record()
            torch.cuda.synchronize()
            best = max(best, blocks * 256 * iters * per_thread_iter / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        out[name] = best
    return out


def fused_kernel_name(w, n_particles):
    if w["spheres"] is not None and n_particles * 2 > 2 * 148:
        return "sgpmp::iterate_split_kernel<7,1,4,4> (state warps + link warps)"
    if w["spheres"] is None and not w.get("f64") and w["n_dof"] in (2, 3, 4, 6) and n_particles > 148:
        return "sgpmp::iterate_split_kernel<%d,0,4,0> (state warps only)" % w["n_dof"]
    return "sgpmp::iterate_kernel<%s,2,%d,%d,%d,1>" % ("double" if w.get("f64") else "float", w["n_dof"],
                                                      128 if (w["spheres"] is None and n_particles >= 10 * 148) else 256,
                                                      1 if w["spheres"] is not None else 0)


def roofline_block(w, ntraj_per_launch, launch_ms, peaks, B, kernel=None):
    """FP32-pipe roofline of the fused iteration kernel from the ALGORITHMIC counts of SURVEY §8(d) (DESIGN.md §4.1)."""
    measured = {}
    try:
        measured = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    traffic, ncu_facts, src = None, None, None
    for rnd in ("r2", "r1"):
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", rnd, "traffic.json"))).get(w["name"])
            if tj and tj["problems"] == B:
                traffic = tj["dram_read_bytes"] + tj["dram_write_bytes"]
                ncu_facts = {k: tj[k] for k in ("thread_instructions_per_traj_sample", "issue_active_pct", "pipe_fma_pct", "pipe_alu_pct", "pipe_xu_pct") if k in tj}
                src = "profiles/%s/traffic.json (ncu --set full capture of this command)" % rnd
                break
        except Exception:
            pass
    flops, mufu = algorithmic_flops_per_traj(w)
    ach_tf = ntraj_per_launch * flops / (launch_ms * 1e-3) / 1e12
    ach_mufu = ntraj_per_launch * mufu / (launch_ms * 1e-3) / 1e12
    return {"bound": "fp32", "kernel": kernel or fused_kernel_name(w, B * w["G"] * w["K"]), "achieved": ach_tf,
            "peak": peaks["fp32_tflops"], "unit": "TFLOP/s", "frac": ach_tf / peaks["fp32_tflops"],
            "frac_of_nominal": ach_tf / NOMINAL_FP32_TFLOPS, "nominal_peak": NOMINAL_FP32_TFLOPS,
            "traffic": traffic, "traffic_source": src, "ncu": ncu_facts,
            "peak_source": "FP32 FMA probe kernel timed in this run (MEASURED_PEAKS.json has no FP32-pipe entry; nominal 74.4)",
            "algorithmic_flops_per_traj_sample": flops, "launch_ms": launch_ms,
            "mufu": {"achieved_tops": ach_mufu, "peak_tops": peaks["mufu_tops"], "frac": ach_mufu / peaks["mufu_tops"],
                     "frac_of_nominal": ach_mufu / NOMINAL_MUFU_TOPS, "algorithmic_mufu_per_traj_sample": mufu},
            "binding": ("mufu" if mufu / peaks["mufu_tops"] > flops / peaks["fp32_tflops"] else "fp32"),
            "binding_note": "lower-bound time = max(flops/FP32 peak, MUFU ops/MUFU peak) from the ALGORITHMIC counts of SURVEY 8(d) "
                            "(+2 MUFU per Box-Muller normal); the implementation trades MUFU for FMA-pipe polynomials and "
                            "structural savings, so the executed pipe utilisations are the ncu figures",
            "hbm_note": "fused kernel: HBM traffic is O(B*NP*M) per step; materialised 3-kernel dataflow would move %.1f GB/step"
                        % (3 * 2 * w["n_dof"] * w["T"] * (8 if w.get("f64") else 4) * ntraj_per_launch / 1e9),
            "measured_hbm_gbs": measured.get("hbm_gbs")}


def time_steps(pl, obs, steps, warmup, flush=None):
    """ms per optimize() iteration: CUDA events around each step (L2 flushed outside the event pair), mean over steps."""
    import torch
    for _ in range(warmup):
        pl.optimize(return_samples=False, **obs)
    torch.cuda.synchronize()
    evs = []
    for _ in range(steps):
        if flush is not None:
            flush.fill_(1.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        pl.optimize(return_samples=False, **obs)
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in evs) / steps


def dump_outputs(out, path):
    """Write what an optimize() call of a StochGPMPBatch returned, with return_samples=False, as <path>/<name>.npy in the
    planner's dtype: means_pos / means_vel [B,NP,T,n] (the means the step started from), costs [B,NP,S], grad [B,NP,T,2n].
    When all B problems exceed DUMP_BYTES, a fixed sample of problems is written (numpy default_rng(0), sorted), the same one
    for every run with the same batch size."""
    import numpy as np
    import torch
    arrays = {"means_pos": out[0], "means_vel": out[1], "costs": out[4], "grad": out[5]}
    B = out[0].shape[0]
    per_problem = sum(a[0].numel() * a.element_size() for a in arrays.values())
    keep = min(B, DUMP_BYTES // per_problem)
    idx = np.sort(np.random.default_rng(0).choice(B, keep, replace=False)) if keep < B else np.arange(B)
    idx = torch.as_tensor(idx, device=out[0].device)
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a.index_select(0, idx).cpu().numpy())


def extra_configs(dev, peaks, flush):
    """C1 / C2 / C3 of BASELINE.json (SURVEY §8d) on one GPU, each with its own roofline line."""
    import torch
    out = {}
    # C2: planar 1024 problems x 4 goals x 256 samples, fp32
    w = workload("planar", 1024)
    pl = build_planner(w, 1024, dev)
    ms = time_steps(pl, {}, 20, 3, flush)
    nt = 1024 * w["G"] * w["K"] * w["S"]
    r = roofline_block(w, nt, ms, peaks, 1024)
    out["planar_1024"] = {"workload": "C2: planar 2-DoF batched, 1024 problems x 4 goals x 256 samples x T 64, fp32", "ms_per_step": ms,
                          "value": nt / (ms * 1e-3), "unit": UNIT,
                          "roofline": dict({k: r[k] for k in ("bound", "kernel", "achieved", "peak", "unit", "frac", "frac_of_nominal", "algorithmic_flops_per_traj_sample", "mufu", "binding", "traffic", "traffic_source", "ncu")},
                                           note="issue-bound, not pipe-bound: ~110 instructions per (sample, step), 59 of them the Philox / Box-Muller draw of "
                                                "the four normals (integer work that the algorithmic FLOP / MUFU counts do not contain); the utilisation to "
                                                "read is ncu.issue_active_pct")}
    del pl
    # C3: one Panda problem, 4 goals x 512 samples (per-iteration latency + the 400-iteration plan)
    w = workload("panda", 1)
    pl = build_planner(w, 1, dev)
    obs = {"obstacle_spheres": torch.tensor(w["spheres"], dtype=torch.float32, device=dev)}
    pl.optimize(opt_iters=3, return_samples=False, **obs)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    pl.optimize(opt_iters=400, return_samples=False, **obs)
    e1.record()
    torch.cuda.synchronize()
    plan_ms = e0.elapsed_time(e1)
    nt = w["G"] * w["K"] * w["S"]
    out["panda_single"] = {"workload": "C3: Panda 7-DoF single problem, 4 goals x 512 samples x T 64, fp32", "ms_per_step": plan_ms / 400,
                           "value": nt / (plan_ms / 400 * 1e-3), "unit": UNIT, "ms_per_plan_400_iterations": plan_ms,
                           "roofline": {"bound": "latency", "frac": None,
                                        "note": "2,048 trajectory samples cannot fill 148 SMs: the low-latency three-kernel form (csrc/sgpmp_lowlat.cu) "
                                                "is bound by T = 64 dependent steps per sample, not by a pipe; the number to read is ms per plan"}}
    del pl
    # C1: planar as shipped (fp64, G=3, K=5, S=128, one problem): 500-iteration plan
    w = workload("planar_shipped", 1)
    pl = build_planner(w, 1, dev)
    pl.optimize(opt_iters=3, return_samples=False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    pl.optimize(opt_iters=500, return_samples=False)
    e1.record()
    torch.cuda.synchronize()
    plan_ms = e0.elapsed_time(e1)
    nt = w["G"] * w["K"] * w["S"]
    out["planar_shipped_fp64"] = {"workload": "C1: examples/planar_environment.py as shipped (fp64, 3 goals x 5 particles x 128 samples, seed 0)",
                                  "ms_per_step": plan_ms / 500, "value": nt / (plan_ms / 500 * 1e-3), "unit": UNIT,
                                  "ms_per_plan_500_iterations": plan_ms,
                                  "roofline": {"bound": "latency", "frac": None, "note": "1,920 fp64 trajectory samples: latency-bound like C3"}}
    return out


def soft_regime(w, wl, B, dev, flush, lo):
    """C4 shapes in a regime where the softmax is NOT one-hot: the update's second RNG sweep (pass 2) then visits every sample.
    With the shipped sigmas the weights are one-hot at ANY temperature (the importance term x^T Sigma^-1 mu does not scale with it and
    its spread over samples is sqrt(mu^T Sigma^-1 mu) >> 1), so this is a constructed case: the soft sigma set of the golden case
    panda_soft_f64 (oracle/make_golden.py: sampling sigmas 4 / 4 / 0.5, cost sigmas 0.5 / 0.5 / 0.3 / 20), start and goals scaled
    towards the origin (x 0.05, as in the soft goldens), and the smallest temperature of a decade ladder whose median effective
    sample size reaches S/16.  The arithmetic per step does not depend on the values."""
    import numpy as np
    import torch
    ws = dict(wl, start=0.05 * np.asarray(wl["start"]), goals=0.05 * np.asarray(wl["goals"]),
              sig=dict(sigma_start_init=0.5, sigma_goal_init=0.5, sigma_gp_init=0.8, sigma_start_sample=4.0, sigma_goal_sample=4.0,
                           sigma_gp_sample=0.5),
              cost=dict(sigma_start=0.5, sigma_gp=0.5, sigma_coll=0.3, sigma_goal_prior=20.), step_size=0.5)
    obs = {"obstacle_spheres": torch.tensor(wl["spheres"], dtype=torch.float32, device=dev)} if w["spheres"] is not None else {}
    tau, ess_med, pls, means0 = None, None, None, None
    for cand in (200., 2e3, 2e4, 2e5, 2e6):
        pls = build_planner(ws, B, dev, problem_offset=lo, seed=0, temperature=cand)
        means0 = pls._means.clone()
        pls.optimize(return_samples=False, **obs)
        wts = pls._weights_raw.double()
        tau, ess_med = cand, float((1.0 / (wts * wts).sum(-1)).median())
        if ess_med >= w["S"] / 16:
            break
    # every timed step starts from the SAME means (the loop sharpens the distribution within a few iterations, which would
    # turn the measurement back into the one-hot regime): the restore is outside the event pair
    evs = []
    for k in range(3 + 10):
        pls._means.copy_(means0)
        flush.fill_(1.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        pls.optimize(return_samples=False, **obs)
        e1.record()
        if k >= 3:
            evs.append((e0, e1))
    torch.cuda.synchronize()
    ms = sum(a.elapsed_time(b) for a, b in evs) / len(evs)
    wts = pls._weights_raw.double()
    ess_med = float((1.0 / (wts * wts).sum(-1)).median())
    return {"temperature": tau, "ess_median": ess_med, "S": w["S"], "ms_per_step": ms,
            "value": B * w["G"] * w["K"] * w["S"] / (ms * 1e-3), "unit": UNIT,
            "sigmas": "panda_soft_f64 set (sampling 4 / 4 / 0.5, cost 0.5 / 0.5, coll 0.3, goal prior 20), step 0.5, start/goals x 0.05",
            "note": "C4 shapes; with the shipped sigmas the softmax is one-hot and pass 2 regenerates one sample per particle; here it "
                    "regenerates every sample with a non-zero weight (a second Philox/Box-Muller sweep, no sample is ever stored)"}


def split_leg(args, rank, world, dev):
    """BASELINE configs[4]: every particle's samples divided over the `world` ranks (NCCL all_gather of the weighted statistics
    issued from C, csrc/sgpmp_nccl.cu).  Timed on 64 Panda problems (fp32) next to the un-split fused loop on ONE rank's GPU, and
    checked against it in fp64 (2 problems)."""
    import torch
    import torch.distributed as dist
    Bs = 64
    w = workload("panda", Bs)
    pl = build_planner(w, Bs, dev)
    obs = {"obstacle_spheres": torch.tensor(w["spheres"], dtype=torch.float32, device=dev)}
    iters = 20
    pl.optimize_split(opt_iters=3, **obs)
    torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    pl.optimize_split(opt_iters=iters, **obs)
    e1.record()
    torch.cuda.synchronize()
    ms_split = e0.elapsed_time(e1) / iters
    one = build_planner(w, Bs, dev)
    one.optimize(opt_iters=3, return_samples=False, **obs)
    torch.cuda.synchronize()
    e0.record()
    one.optimize(opt_iters=iters, return_samples=False, **obs)
    e1.record()
    torch.cuda.synchronize()
    ms_one = e0.elapsed_time(e1) / iters
    # fp64 equality on 2 problems, 3 iterations
    w2 = dict(workload("panda", 2), f64=True)
    a = build_planner(w2, 2, dev)
    b = build_planner(w2, 2, dev)
    obs2 = {"obstacle_spheres": torch.tensor(w2["spheres"], dtype=torch.float64, device=dev)}
    a.optimize_split(opt_iters=3, **obs2)
    b.optimize(opt_iters=3, return_samples=False, **obs2)
    diff = float((a.particle_means - b.particle_means).abs().max() / b.particle_means.abs().max())
    t = torch.tensor([ms_split, ms_one, diff], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_split, ms_one, diff = [float(x) for x in t.tolist()]
    M = w["T"] * 2 * w["n_dof"]
    return {"ranks": world, "problems": Bs, "goals": w["G"], "samples_per_particle": w["S"], "samples_per_rank": w["S"] // world,
            "ms_per_iteration": ms_split, "single_rank_ms_per_iteration": ms_one, "ratio_to_single_rank": ms_split / ms_one,
            "allgather_bytes_per_rank_per_iteration": Bs * w["G"] * w["K"] * (M + 2) * 4,
            "launches_per_iteration": 3, "max_rel_diff_vs_unsplit_fp64": diff, "fp64_check_passed": bool(diff < 1e-9),
            "note": "per iteration: one fused stats launch over this rank's samples, one ncclAllGather on the compute stream, one "
                    "merge + update launch; all iterations enqueued by one C call (sgpmp_iterate_split_particles)"}


def run_ours(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist
    from stoch_gpmp_b200 import _lib
    from stoch_gpmp_b200.parallel import shard_range

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    strong = args.scaling == "strong"
    total = args.problems if strong else args.problems * world
    lo, hi = shard_range(total, rank, world)
    B = hi - lo
    w = workload(args.workload, total)
    wl = dict(w, start=w["start"][lo:hi], goals=w["goals"][lo:hi],
              spheres=None if w["spheres"] is None else w["spheres"][lo:hi])
    pl = build_planner(wl, B, dev, problem_offset=lo, seed=0)
    obs = {}
    if w["spheres"] is not None:
        obs = {"obstacle_spheres": torch.tensor(wl["spheres"], dtype=torch.float32).pin_memory().to(dev)}
    ntraj_total = total * w["G"] * w["K"] * w["S"]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    # ---------------- warm-up
    for _ in range(max(args.warmup, 3)):
        pl.optimize(return_samples=False, **obs)
    barrier()

    # ---------------- timed: device-resident inputs ("value")
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    launches0 = _lib.launch_count()
    evs = []
    barrier()
    wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.fill_(1.0)                                  # L2 flush (126 MB L2 < 256 MiB), outside the event pair
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = pl.optimize(return_samples=False, **obs)
        e1.record()
        evs.append((e0, e1))
    barrier()
    wall = time.perf_counter() - wall0
    launches = _lib.launch_count() - launches0
    clk = clocks.stop() if rank == 0 else None
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    if args.dump_outputs:
        dump_outputs(out, args.dump_outputs)       # before the end-to-end leg, which may run `pl` again

    # ---------------- timed: end to end from host buffers ("e2e")
    # Public API only: the batch is sharded into E2E_SHARDS StochGPMPBatch objects (problem_offset keeps every RNG stream where it
    # was, results are bit-identical to the single batch: tests/test_gpu_planner.py::test_fused_problem_sharding_invariance), one
    # CUDA stream each.  Per step every shard copies its inputs H2D, runs optimize() and copies its plan D2H on its own stream, so
    # the D2H of shard k rides under the kernel of shard k+1; the host waits for ALL shards before the next step starts
    # ("the user has the plan on the host every step").
    n_sh = max(1, min(args.e2e_shards, B))
    while B % n_sh:
        n_sh -= 1
    Bs = B // n_sh
    from stoch_gpmp_b200.parallel import StreamShards
    planners, host_in = [], []
    for k in range(n_sh):
        a = k * Bs
        wk = dict(w, start=wl["start"][a:a + Bs], goals=wl["goals"][a:a + Bs], spheres=None if wl["spheres"] is None else wl["spheres"][a:a + Bs])
        planners.append(build_planner(wk, Bs, dev, problem_offset=lo + a, seed=0) if n_sh > 1 else pl)
        if wl["spheres"] is not None:
            host_in.append(torch.tensor(wk["spheres"], dtype=torch.float32).pin_memory())
        else:      # planar: the per-step host input is the start/goal set of every problem
            host_in.append(torch.tensor(np.concatenate([wk["start"].reshape(Bs, -1), wk["goals"].reshape(Bs, -1)], 1), dtype=torch.float32).pin_memory())
    shards = StreamShards(planners, obs_key="obstacle_spheres" if wl["spheres"] is not None else None, host_inputs=host_in)
    h2d = sum(h.numel() for h in host_in) * 4
    d2h = sum(m.numel() for m in shards.host_means) * 4

    def e2e_step():
        shards.step()
        shards.wait()                                       # the user has the whole plan on the host every step

    torch.cuda.synchronize()
    for _ in range(3):
        e2e_step()
    barrier()
    launches_e2e0 = _lib.launch_count()
    e2e_wall0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    e2e_wall = time.perf_counter() - e2e_wall0               # host clock: every step ends with a host-side wait on all streams
    launches_e2e = _lib.launch_count() - launches_e2e0
    barrier()
    e2e_ms = e2e_wall * 1e3
    del shards, planners

    # ---------------- N > 1: weak-scaling companion (4096 problems per GPU) and the split-particle leg
    weak = split = None
    if world > 1 and strong and not args.no_extras:
        ww = workload(args.workload, args.problems * world)
        a = rank * args.problems
        wwl = dict(ww, start=ww["start"][a:a + args.problems], goals=ww["goals"][a:a + args.problems],
                   spheres=None if ww["spheres"] is None else ww["spheres"][a:a + args.problems])
        plw = build_planner(wwl, args.problems, dev, problem_offset=a, seed=0)
        obsw = {"obstacle_spheres": torch.tensor(wwl["spheres"], dtype=torch.float32, device=dev)} if ww["spheres"] is not None else {}
        barrier()
        ms_w = time_steps(plw, obsw, 5, 3, flush)
        del plw
        tw = torch.tensor([ms_w], dtype=torch.float64, device=dev)
        dist.all_reduce(tw, op=dist.ReduceOp.MAX)
        ms_w = float(tw[0])
        weak = {"problems_per_gpu": args.problems, "problems_total": args.problems * world, "ms_per_step": ms_w,
                "value": args.problems * world * w["G"] * w["K"] * w["S"] / (ms_w * 1e-3), "unit": UNIT}
        if w["spheres"] is not None and w["S"] % world == 0:
            split = split_leg(args, rank, world, dev)

    # ---------------- max over ranks
    t = torch.tensor([dev_ms, e2e_ms, wall * 1e3, e2e_wall * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, wall_ms, e2e_wall_ms = [float(x) for x in t.tolist()]
    if rank != 0:
        return
    ms_per_step = dev_ms / args.steps
    value = ntraj_total / (ms_per_step * 1e-3)
    e2e_value = ntraj_total * args.steps / (max(e2e_ms, e2e_wall_ms) * 1e-3)

    # ---------------- roofline of the dominant kernel (the fused iteration kernel: one launch per step)
    peaks = probe_peaks(dev)
    roof = roofline_block(w, B * w["G"] * w["K"] * w["S"], ms_per_step, peaks, B)

    # ---------------- CPU baseline (bounded sample, rank 0, N=1 only)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        sec, cores = cpu_reference_time(w, 2, 2, 1)
        cpu = {"value": w["G"] * w["K"] * w["S"] / sec, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "2 problems x (1 warm-up + 2 timed) optimize() iterations of the workload's per-problem shape, "
                         "run sequentially (the reference has no problem-batch axis); value = NP*S / mean s per iteration",
               "s_per_iteration_per_problem": sec}

    # ---------------- "ms per plan" of ONE problem (the metric's second half): all iterations in one fused launch
    plan_iters = 400 if w["spheres"] is not None else 500
    w1 = dict(w, start=w["start"][:1], goals=w["goals"][:1], spheres=None if w["spheres"] is None else w["spheres"][:1])
    p1 = build_planner(w1, 1, dev, problem_offset=0, seed=0)
    obs1 = {"obstacle_spheres": torch.tensor(w1["spheres"], dtype=torch.float32, device=dev)} if w["spheres"] is not None else {}
    p1.optimize(opt_iters=3, return_samples=False, **obs1)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    p1.optimize(opt_iters=plan_iters, return_samples=False, **obs1)
    e1.record()
    torch.cuda.synchronize()
    plan_ms_single = e0.elapsed_time(e1)

    # ---------------- N = 1: the other BASELINE configs and the soft-softmax regime
    configs = soft = None
    if world == 1 and not args.no_extras:
        del pl
        configs = extra_configs(dev, peaks, flush)
        soft = soft_regime(w, wl, B, dev, flush, lo)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": w["name"], "problems_per_gpu": B, "problems_total": total, "goals": w["G"],
                       "particles_per_goal": w["K"] * w["S"], "K": w["K"], "S": w["S"], "traj_len": w["T"], "n_dof": w["n_dof"],
                       "traj_samples_per_step": ntraj_total, "opt_iters_per_step": 1,
                       "parallelism": "problem-sharded x%d (%s: %d problems in total), no collective" % (world, "strong" if strong else "weak", total),
                       "l2": "256 MiB write between timed steps (outside the CUDA-event pair)", "prior": "fp64 factor, fp32 run-time",
                       "rng": "in-kernel Philox4x32-7, one call per (time step, DoF pair)"},
            "clocks": clk, "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world,
                                   "ms_per_step": max(e2e_ms, e2e_wall_ms) / args.steps, "shards_per_gpu": n_sh,
                                   "launches_per_step": launches_e2e / args.steps,
                                   "note": "StochGPMPBatch per shard on its own stream: H2D inputs, optimize(), D2H plan; host waits for all shards every step"},
            "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu, "wall_ms_per_step_incl_flush": wall_ms / args.steps,
            "ms_per_plan": {"iterations": plan_iters, "single_problem_ms": plan_ms_single,
                            "amortised_over_batch_ms": ms_per_step * plan_iters / B,
                            "note": "single problem = one StochGPMP (B=1), all iterations enqueued by one optimize() call (low-latency three-kernel form, csrc/sgpmp_lowlat.cu)"}}
    if configs is not None:
        line["configs"] = configs
        line["soft_regime"] = soft
    if weak is not None:
        line["weak"] = weak
    if split is not None:
        line["split"] = split
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cuda"])
    ap.add_argument("--workload", default="panda", choices=["panda", "planar"])
    ap.add_argument("--problems", type=int, default=4096, help="problems in total (strong scaling) or per GPU (weak scaling)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs / soft_regime / weak / split blocks")
    ap.add_argument("--e2e-shards", type=int, default=8, help="StochGPMPBatch shards (CUDA streams) per GPU in the end-to-end measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or world > 1):
        ap.error("--dump-outputs needs --impl ours in a single process")
    if args.impl in ("reference", "reference-cuda"):
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (which may be read-only)
    main()
