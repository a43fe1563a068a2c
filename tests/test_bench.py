"""bench.py --dump-outputs and --steps: the dump holds what the timed path returned, under 64 MB, the same from run to run;
--steps sets the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ["costs.npy", "grad.npy", "means_pos.npy", "means_vel.npy"]


def _outputs(B, NP, T, n, S, dtype):
    """An optimize() return tuple whose costs carry the problem index, so that a dumped row names its problem."""
    g = torch.Generator().manual_seed(0)
    mp = torch.randn(B, NP, T, 2 * n, generator=g, dtype=dtype)
    costs = torch.arange(B, dtype=dtype)[:, None, None].expand(B, NP, S).contiguous()
    return (mp[..., :n], mp[..., n:], None, None, costs, torch.randn(B, NP, T, 2 * n, generator=g, dtype=dtype))


def test_dump_outputs_samples_the_flagship_batch_under_64mb(tmp_path):
    out = _outputs(4096, 4, 64, 7, 512, torch.float32)       # the flagship batch: 151 MB of outputs
    for d in ("a", "b"):
        bench.dump_outputs(out, str(tmp_path / d))
    assert sorted(os.listdir(tmp_path / "a")) == NAMES
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in NAMES) <= 64 * 10 ** 6
    for f in NAMES:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float32 and np.array_equal(a, b)
    idx = np.load(tmp_path / "a" / "costs.npy")[:, 0, 0].astype(np.int64)
    assert len(idx) > 1000 and np.all(np.diff(idx) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "means_pos.npy"), out[0].numpy()[idx])
    assert np.array_equal(np.load(tmp_path / "a" / "means_vel.npy"), out[1].numpy()[idx])
    assert np.array_equal(np.load(tmp_path / "a" / "grad.npy"), out[5].numpy()[idx])


def test_dump_outputs_writes_a_small_batch_whole(tmp_path):
    out = _outputs(3, 15, 64, 2, 128, torch.float64)
    bench.dump_outputs(out, str(tmp_path))
    assert sorted(os.listdir(tmp_path)) == NAMES
    for f, a in zip(NAMES, (out[4], out[5], out[0], out[1])):
        got = np.load(tmp_path / f)
        assert got.dtype == np.float64 and np.array_equal(got, a.numpy())


def _bench(steps, dump=None):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
           "--problems", "16", "--no-cpu-baseline", "--no-extras"] + (["--dump-outputs", dump] if dump else [])
    r = subprocess.run(cmd, check=True, capture_output=True, text=True, timeout=600)
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_bench_dump_is_reproducible_and_steps_are_timed(cuda, tmp_path):
    a = _bench(2, str(tmp_path / "a"))
    b = _bench(2, str(tmp_path / "b"))
    c = _bench(3)
    for f in NAMES:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    # the dump is the return of the last timed step: the same seeded planner, called warm-up + timed times, returns it
    w = bench.workload("panda", 16)
    pl = bench.build_planner(w, 16, cuda)
    obs = {"obstacle_spheres": torch.tensor(w["spheres"], dtype=torch.float32, device=cuda)}
    for _ in range(a["warmup"] + a["steps"]):
        r = pl.optimize(return_samples=False, **obs)
    want = {"means_pos.npy": (r[0], (16, 4, 64, 7)), "means_vel.npy": (r[1], (16, 4, 64, 7)), "costs.npy": (r[4], (16, 4, 512)),
            "grad.npy": (r[5], (16, 4, 64, 14))}
    for f, (t, shape) in want.items():
        got = np.load(tmp_path / "a" / f)
        assert got.shape == shape and np.array_equal(got, t.cpu().numpy()), f
    assert (a["steps"], c["steps"]) == (2, 3)
    assert a["gpu_launches"] > 0 and a["gpu_launches"] * 3 == c["gpu_launches"] * 2       # launches of the timed loop ~ --steps
