"""bench.py --dump-outputs: refused for a primary workload without control() outputs (CPU); -m gpu: the dump holds
what the last timed step returned (replayed on the CPU oracle), the same in every run of the same arguments, and
--steps sets the number of timed steps."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from helpers import assert_abs_rel_close, make_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=900)


def test_dump_needs_a_control_workload(tmp_path):
    for extra in (["--workload", "c3"], ["--impl", "reference"]):
        r = bench("--dump-outputs", str(tmp_path / "dump"), *extra)
        assert r.returncode == 2 and "--dump-outputs" in r.stderr, r.stderr[-2000:]
    assert not (tmp_path / "dump").exists()


def replay_last_step(line, instances):
    """u0, metric, ut of the given instances after the last timed step of a single-GPU c2 run: the step ran batch
    (controller) (K - 1) mod n_rot, which bench_solve had stepped in its warm-up rounds and in every earlier timed step
    that fell on it, always from the same seeded states x"""
    import bench as b

    wl, seed = b.WORKLOADS["c2"], 0xE16C0D1C + 2
    B, K, W = line["config"]["instances_total"], line["steps"], line["warmup"]
    n_rot = int(re.search(r"rotate over (\d+) independent batches", line["config"]["l2"]).group(1))
    j = (K - 1) % n_rot
    calls = sum(i % n_rot == j for i in range(max(W, n_rot))) + sum(i % n_rot == j for i in range(K))
    x, ut, _ = b.synth_inputs(wl, B, seed)
    if j:
        ut = b.synth_inputs(dict(wl, mem=0), B, seed=0xE16C0D1C + 1000 * (j + 1))[1]
    out = {"u0": [], "metric": [], "ut": []}
    for i in instances:
        o = make_oracle(wl["model"], nb=wl["nb"], horizon=wl["horizon"])
        o.set_ut(ut[i])
        for _ in range(calls):
            u0 = o.control(b.BOUNDS, x[i])
        out["u0"].append(u0)
        out["metric"].append(o.last()["metric"])
        out["ut"].append(o.get_ut())
    return out


@pytest.mark.gpu
def test_dump_of_the_last_timed_step(tmp_path):
    runs = []
    for steps in (3, 3, 8):
        out = tmp_path / str(len(runs))
        r = bench("--gpus", "1", "--steps", str(steps), "--warmup", "2", "--workload", "c2", "--dump-outputs", str(out))
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps
        runs.append((line, {n: np.load(out / f"{n}.npy") for n in ("u0", "metric", "ut")}))
    (line, dump), (_, again), (line8, _) = runs
    B, N = line["config"]["instances_total"], line["config"]["horizon_steps"]
    assert dump["u0"].shape == (B, 3) and dump["metric"].shape == (B,) and dump["ut"].shape == (B, N, 3)
    for name, a in dump.items():
        assert a.dtype == np.float64 and np.isfinite(a).all(), name
        np.testing.assert_array_equal(a, again[name], err_msg=f"{name} differs between two runs")
    assert line8["gpu_launches"] * 3 == line["gpu_launches"] * 8  # the same launches per timed step
    instances = np.random.default_rng(5).choice(B, 6, replace=False)
    for ln, d in ((line, dump), runs[2]):
        want = replay_last_step(ln, instances)
        for name in d:
            assert_abs_rel_close(d[name][instances], np.array(want[name]), f"--steps {ln['steps']}: {name}")
