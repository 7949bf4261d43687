"""The safe tick of B robots per GPU on several GPUs: eb_control_safe_batch_dev_gather_wait (the final twists stored
into every rank's gathered buffer over NVLink peer memory by the validation and fallback kernels, the last fallback CTA
waiting for every rank's flag) against what a user writes without it: eb_control_safe_batch_dev followed by one
dist.all_gather_into_tensor of u per tick.

Setup per GPU (the K4 setup of DESIGN.md): B = 4096 Omni robots (nb 10, 50 steps, per-instance entropy targets, warm
ut_), each on its own free map of 160..640 cells a side at 0.05 m (several hundred MB, more than the 126 MB of L2),
validate_control over 2 s at 0.1 s, the 3 x 8 x 5 window of explore_omni.yaml, vb = 0.  The failing fraction is steered
by obstacle rings 0.6..0.8 m around a share of the robots and counted from the checked tick's branches.

Both variants are driven through ctypes on device buffers on torch's current stream.  CUDA events around K strict
ticks after a warm-up, variants alternated per round (tools/per_instance_timing.time_rounds); every rank times the same
sequence, and the slowest rank's median is reported.  Before timing, one tick of each variant runs on clones of the
same controller and the gathered rows are compared bit for bit on every rank.

    python -m torch.distributed.run --nproc-per-node N tools/sharded_tick_timing.py [--batch B] [--steps K] [--rounds R]
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from per_instance_timing import card, gpu, time_rounds  # noqa: E402
from safe_control_timing import COL, DWA, RES, SAMPLES, VAL_DT, VAL_H  # noqa: E402

FRACTIONS = (0.0, 0.08)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=7)
    a = ap.parse_args()

    import torch
    import torch.distributed as dist

    import ergodic_exploration_b200 as eb
    from ergodic_exploration_b200 import capi
    from ergodic_exploration_b200.sharding import PeerGather

    if not torch.cuda.is_available():
        raise SystemExit("sharded_tick_timing needs CUDA devices")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", device_id=dev)
    lib = capi.load()
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rng = np.random.default_rng(rank)
    B = a.batch
    sides = rng.integers(160, 641, size=(B, 2))  # (ysize, xsize)
    origin = np.column_stack([rng.uniform(-50, 50, B), rng.uniform(-50, 50, B)])
    total_bytes = int(sum(int(ys) * int(xs) for ys, xs in sides))
    fx, fy = rng.uniform(0.2, 0.8, B), rng.uniform(0.2, 0.8, B)
    x_h = np.column_stack([origin[:, 0] + fx * sides[:, 1] * RES, origin[:, 1] + fy * sides[:, 0] * RES,
                           rng.uniform(-np.pi, np.pi, B)])
    free, ring = [], []
    for i, (ys, xs) in enumerate(sides):
        c = torch.zeros((int(ys), int(xs)), dtype=torch.int8, device=dev)
        free.append(c)
        cx = origin[i, 0] + (torch.arange(int(xs), device=dev, dtype=torch.float64) + 0.5) * RES
        cy = origin[i, 1] + (torch.arange(int(ys), device=dev, dtype=torch.float64) + 0.5) * RES
        d = torch.hypot(cx[None, :] - x_h[i, 0], cy[:, None] - x_h[i, 1])
        ring.append(torch.where((d > 0.6) & (d < 0.8), torch.tensor(100, dtype=torch.int8, device=dev), c))
    res_a, org_l = [RES] * B, [tuple(o) for o in origin]

    base = gpu(eb, B, 10)
    base.setMapTargets(free, res_a, org_l)
    base.set_ut(rng.uniform([-1.0, -1.0, -2.0], [1.0, 1.0, 2.0], size=(B, base.steps, 3)) * 0.5)
    gb = eb.GridMapBatch(B, device=rank)
    lib.eb_grid_batch_set_stream(gb._h, s)
    col, dwa = capi.EbCollision(*COL), capi.EbDwa(*DWA, *SAMPLES)
    x = torch.from_numpy(x_h).to(dev)
    vb = torch.zeros((B, 3), dtype=torch.float64, device=dev)
    u = torch.empty((B, 3), dtype=torch.float64, device=dev)
    full = torch.empty((world * B, 3), dtype=torch.float64, device=dev)
    br = torch.empty(B, dtype=torch.int32, device=dev)
    pg = PeerGather(base)
    P = lambda t: C.c_void_p(t.data_ptr())

    def ok(st):
        assert st == 0, lib.eb_last_error()

    def peer(c):  # (a)
        return lambda: ok(lib.eb_control_safe_batch_dev_gather_wait(c._h, pg._h, gb._h, col, dwa, VAL_DT, VAL_H, None,
                                                                    P(x), None, P(vb), P(br), None))

    def nccl(c):  # (b)
        def run():
            ok(lib.eb_control_safe_batch_dev(c._h, gb._h, col, dwa, VAL_DT, VAL_H, None, P(x), None, P(vb), P(u),
                                             P(br), None))
            dist.all_gather_into_tensor(full, u)
        return run

    def clone():
        c = base.clone()
        lib.eb_set_stream(c._h, s)
        return c

    perm = rng.permutation(B)
    results = []
    for f in FRACTIONS:
        inring = np.zeros(B, dtype=bool)
        inring[perm[:int(round(f * B))]] = True
        gb.set([ring[i] if inring[i] else free[i] for i in range(B)], res_a, org_l)
        # the checked tick: (a) and (b) on clones of the same controller, every rank's rows
        c1, c2 = clone(), clone()
        peer(c1)()
        got = pg.gathered(pg.steps).clone()
        nccl(c2)()
        torch.cuda.synchronize()
        same = torch.tensor([int(torch.equal(got.view(torch.int64), full.view(torch.int64)))], device=dev)
        failing = torch.tensor([int((br != 0).sum())], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        dist.all_reduce(failing)
        assert int(same.item()) == 1, f"fraction {f}: the gathered rows differ from the all_gather"
        t = time_rounds(torch, {"peer_gather_wait": peer(clone()), "safe_then_all_gather": nccl(clone())}, a.steps,
                        a.rounds)
        worst = torch.tensor([t["peer_gather_wait"], t["safe_then_all_gather"]], dtype=torch.float64, device=dev)
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        results.append({
            "target_fraction": f, "failing_fraction_checked": int(failing.item()) / (world * B),
            "outputs_bit_identical": True, "peer_gather_wait_us": float(worst[0]),
            "safe_then_all_gather_us": float(worst[1]), "saved_us": float(worst[1] - worst[0]),
        })
    if rank == 0:
        name, power = card()
        print(json.dumps({
            "card": name, "power_limit": power, "world": world, "batch_per_gpu": B, "steps": a.steps,
            "rounds": a.rounds,
            "maps": f"{B} free maps per GPU, sides uniform in [160, 640] cells at {RES} m, {total_bytes / 1e6:.0f} MB on "
                    "rank 0; obstacle rings 0.6..0.8 m around a share of the robots",
            "controller": f"Omni, nb 10, {base.steps} steps, per-instance entropy targets, warm ut_, no replay memory",
            "window": f"{SAMPLES[0]} x {SAMPLES[1]} x {SAMPLES[2]}, vb = 0; validate_control {VAL_H} s at {VAL_DT} s",
            "fractions": results,
        }))
    torch.cuda.synchronize()
    dist.barrier()
    pg.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
