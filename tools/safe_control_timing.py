"""The safe control tick of B robots on B maps (eb_control_safe_batch_dev) against the chain of calls it replaces:
eb_control_batch_dev, eb_validate_control_batch_dev, eb_opt_traj_dev, eb_dwa_control_traj_batch_dev over ALL robots and
two torch.where selections.  Also the mapping of the dynamic window: dwa_fallback_kernel (one CTA per failing robot)
against dwa_control_kernel<true> (one warp per robot) run on a grid batch of just the failing robots.

Setup: B = 4096 robots, each on its own free map of 160..640 cells a side at 0.05 m (several hundred MB, more than the
126 MB of L2), a per-instance Omni controller (nb 10, 50 steps) with the maps' entropy targets and a warm control
signal, robots inside their maps, vb = 0, validate_control over 2 s at 0.1 s, the 3 x 8 x 5 window of explore_omni.yaml.
The failing fraction is steered by putting an obstacle ring 0.6..0.8 m around a chosen share of the robots (a twist that
travels more than ~0.35 m collides; the window's slow candidates stay clear); the fraction that actually fails is
counted from the tick's branches and printed, before and after the timed calls (the solve moves ut_ on every call).

Every variant is driven through ctypes on device buffers on torch's current stream, so the host cost of enqueueing is
part of each time.  CUDA events around K back-to-back calls after a warm-up; variants alternated per round
(tools/per_instance_timing.time_rounds), medians reported.  The two window kernels are timed by torch.profiler (CUDA
activity, device time per launch) in a separate phase after the event timing.  Before timing, the outputs of the new
call and of the chain are compared bit for bit on clones of the same controller at every fraction.

    python tools/safe_control_timing.py [--batch B] [--steps K] [--rounds R]
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

COL = (0.2, 1.0, 0.05, 0.65)  # explore_omni.yaml radii
DWA = (0.1, 2.0, 0.2, 1.0, 1.0, 2.0, 1.0, -1.0, 1.0, -1.0, 2.0, -2.0)
SAMPLES = (3, 8, 5)
RES, VAL_DT, VAL_H = 0.05, 0.1, 2.0
FRACTIONS = (0.0, 0.01, 0.1, 1.0)


def kernel_us(prof, name):
    """mean device time per launch of the kernels whose name contains `name`, from a torch.profiler run"""
    tot, cnt = 0.0, 0
    for e in prof.key_averages():
        if name in e.key:
            t = getattr(e, "device_time_total", None)
            tot += t if t is not None else e.cuda_time_total
            cnt += e.count
    return tot / cnt if cnt else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()

    import torch

    import ergodic_exploration_b200 as eb
    from ergodic_exploration_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("safe_control_timing needs a CUDA device")
    lib = capi.load()
    dev = torch.device("cuda")
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rng = np.random.default_rng(0)
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
    N = base.steps
    gb = eb.GridMapBatch(B)
    lib.eb_grid_batch_set_stream(gb._h, s)
    col, dwa = capi.EbCollision(*COL), capi.EbDwa(*DWA, *SAMPLES)
    x = torch.from_numpy(x_h).to(dev)
    vb = torch.zeros((B, 3), dtype=torch.float64, device=dev)
    u0, ud, uc, us = (torch.empty((B, 3), dtype=torch.float64, device=dev) for _ in range(4))
    zeros = torch.zeros((B, 3), dtype=torch.float64, device=dev)
    valid, found, br = (torch.empty(B, dtype=torch.int32, device=dev) for _ in range(3))
    xt = torch.empty((B, N, 3), dtype=torch.float64, device=dev)
    P = lambda t: C.c_void_p(t.data_ptr())

    def ok(st):
        assert st == 0, lib.eb_last_error()

    def safe(c):
        return lambda: ok(lib.eb_control_safe_batch_dev(c._h, gb._h, col, dwa, VAL_DT, VAL_H, None, P(x), None, P(vb),
                                                        P(us), P(br), None))

    def chain(c):
        def run():
            ok(lib.eb_control_batch_dev(c._h, None, P(x), None, P(u0), None))
            ok(lib.eb_validate_control_batch_dev(gb._h, col, P(x), P(u0), 1, VAL_DT, VAL_H, P(valid)))
            ok(lib.eb_opt_traj_dev(c._h, P(xt)))
            ok(lib.eb_dwa_control_traj_batch_dev(gb._h, col, dwa, P(x), P(vb), P(xt), N, 1, base.timeStep(), P(found),
                                                 P(ud), None))
            torch.where(valid.bool()[:, None], u0, torch.where(found.bool()[:, None], ud, zeros), out=uc)
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
        # bit identity with the chain on clones of the same controller
        c1, c2 = clone(), clone()
        safe(c1)()
        chain(c2)()
        branch_chain = torch.where(valid.bool(), 0, torch.where(found.bool(), 1, 2)).to(torch.int32)
        torch.cuda.synchronize()
        same = bool(torch.equal(us.view(torch.int64), uc.view(torch.int64)) and torch.equal(br, branch_chain))
        assert same, f"fraction {f}: the safe tick and the chain differ"
        failing = torch.nonzero(br != 0).flatten()
        frac_before = failing.numel() / B
        # event timing, alternated
        ca, cb = clone(), clone()
        t = time_rounds(torch, {"safe": safe(ca), "chain": chain(cb)}, a.steps, a.rounds)
        ca2 = ca.clone()
        lib.eb_set_stream(ca2._h, s)
        safe(ca2)()
        torch.cuda.synchronize()
        frac_after = int((br != 0).sum()) / B
        # the window mappings on the same failing robots (those of the checked tick)
        mapping = {"failing_robots": int(failing.numel())}
        if failing.numel() > 0:
            idx = failing.cpu().numpy()
            nf = len(idx)
            sub = eb.GridMapBatch(nf)
            lib.eb_grid_batch_set_stream(sub._h, s)
            sub.set([ring[i] if inring[i] else free[i] for i in idx], [RES] * nf, [org_l[i] for i in idx])
            c3 = clone()
            ok(lib.eb_control_batch_dev(c3._h, None, P(x), None, P(u0), None))
            ok(lib.eb_opt_traj_dev(c3._h, P(xt)))
            ti = torch.from_numpy(idx).to(dev)
            xs_, vs_, xts = x[ti].contiguous(), vb[ti].contiguous(), xt[ti].contiguous()
            fs = torch.empty(nf, dtype=torch.int32, device=dev)
            uos = torch.empty((nf, 3), dtype=torch.float64, device=dev)
            warp = lambda: ok(lib.eb_dwa_control_traj_batch_dev(sub._h, col, dwa, P(xs_), P(vs_), P(xts), N, 1,
                                                                base.timeStep(), P(fs), P(uos), None))
            cp = clone()
            fb = safe(cp)
            for _ in range(3):
                warp()
                fb()
            torch.cuda.synchronize()
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for _ in range(a.steps):
                    fb()
                    warp()
                torch.cuda.synchronize()
            mapping.update({
                "fallback_cta_per_robot_kernel_us": kernel_us(prof, "dwa_fallback_kernel"),
                "dwa_control_kernel_warp_per_robot_us": kernel_us(prof, "dwa_control_kernel"),
                "warp_call_event_us": time_rounds(torch, {"warp": warp}, a.steps, a.rounds)["warp"],
            })
        results.append({
            "target_fraction": f, "failing_fraction_checked": frac_before, "failing_fraction_after_timing": frac_after,
            "outputs_bit_identical": same, "safe_us": t["safe"], "chain_us": t["chain"],
            "chain_over_safe": t["chain"] / t["safe"], "mapping": mapping,
        })
    name, power = card()
    print(json.dumps({
        "card": name, "power_limit": power, "batch": B, "steps": a.steps, "rounds": a.rounds,
        "maps": f"{B} free maps, sides uniform in [160, 640] cells at {RES} m, {total_bytes / 1e6:.0f} MB; obstacle "
                "rings 0.6..0.8 m around a share of the robots",
        "controller": f"Omni, nb 10, {N} steps, per-instance entropy targets, warm ut_, no replay memory",
        "window": f"{SAMPLES[0]} x {SAMPLES[1]} x {SAMPLES[2]}, vb = 0; validate_control {VAL_H} s at {VAL_DT} s",
        "fractions": results,
    }))


if __name__ == "__main__":
    main()
