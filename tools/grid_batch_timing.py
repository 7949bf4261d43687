"""Per-instance occupancy maps (eb_grid_batch): B robots, each on its own map, checked with one launch per call,
against (a) the loop over one eb_grid handle per robot that is the only per-map route without it, at a B that loop can
afford, and (b) the shared-grid call at the same B on one map of the same size (dilation off, so both walk circles).

Prints one JSON line.  CUDA events around K back-to-back calls after a warm-up; the variants of a group are alternated
in the same process (tools/per_instance_timing.time_rounds) and the median of the rounds is reported.  Every variant is
driven through ctypes on device buffers on torch's current stream, so the host cost of enqueueing is part of each time.
L2 is not flushed.  B = 4096 maps of 160..640 cells a side are several hundred MB, far more than the 126 MB of L2, so
the per-map probes come from HBM and the L2 gather peak (bench.py --workload collide) is not their bound; no share of
peak is quoted.  Probes per second use the algorithmic probe count of bench.py: the cells of the pruned circle walks
r_bnd .. min(r_max, r_col) per pose check (an upper bound: early exits probe less).

    python tools/grid_batch_timing.py [--batch B] [--loop-batch BL] [--steps K] [--rounds R]
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

from per_instance_timing import card, time_rounds  # noqa: E402

COL = (0.2, 1.0, 0.05, 0.65)  # explore_omni.yaml radii
DWA = (0.1, 2.0, 0.2, 1.0, 1.0, 2.0, 1.0, -1.0, 1.0, -1.0, 2.0, -2.0)
SAMPLES = (3, 8, 5)
RES = 0.05


def circle_cells(r):
    x, y, err, cnt = -r, 0, 2 - 2 * r, 0
    while x < 0:
        cnt += 4
        rr = err
        if rr <= y:
            y += 1
            err += 2 * y + 1
        if rr > x or err > y:
            x += 1
            err += 2 * x + 1
    return cnt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--loop-batch", type=int, default=256)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()

    import torch

    import ergodic_exploration_b200 as eb
    from ergodic_exploration_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("grid_batch_timing needs a CUDA device")
    lib = capi.load()
    dev = torch.device("cuda")
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rng = np.random.default_rng(0)
    B, BL = a.batch, a.loop_batch
    sides = rng.integers(160, 641, size=(B, 2))  # (ysize, xsize)
    gen = torch.Generator(device=dev).manual_seed(0)
    cells = []
    for ys, xs in sides:
        c = torch.zeros((int(ys), int(xs)), dtype=torch.int8, device=dev)
        c[torch.rand((int(ys), int(xs)), generator=gen, device=dev) < 0.004] = 100
        cells.append(c)
    cells_h = [c.cpu().numpy() for c in cells]
    origin = np.column_stack([rng.uniform(-50, 50, B), rng.uniform(-50, 50, B)])
    total_bytes = int(sum(int(ys) * int(xs) for ys, xs in sides))

    gb = eb.GridMapBatch(B)
    gb.set(cells_h, RES, origin)
    lib.eb_grid_batch_set_stream(gb._h, s)
    xs_a = np.ascontiguousarray(sides[:, 1], dtype=np.uint32)
    ys_a = np.ascontiguousarray(sides[:, 0], dtype=np.uint32)
    res_a = np.full(B, RES)
    ptr_d = (C.c_void_p * B)(*[c.data_ptr() for c in cells])
    ptr_h = (C.c_void_p * B)(*[c.ctypes.data for c in cells_h])
    few = np.zeros(B, dtype=np.int32)
    few[rng.choice(B, B // 10, replace=False)] = 1

    def set_call(fn, ptrs, upd):
        def run():
            st = fn(gb._h, C.addressof(ptrs), xs_a.ctypes.data, ys_a.ctypes.data, res_a.ctypes.data, origin.ctypes.data,
                    upd.ctypes.data if upd is not None else None)
            assert st == 0, lib.eb_last_error()
        return run

    set_times = time_rounds(torch, {
        "dev_all": set_call(lib.eb_grid_batch_set_maps_dev, ptr_d, None),
        "dev_10pct": set_call(lib.eb_grid_batch_set_maps_dev, ptr_d, few),
        "host_all": set_call(lib.eb_grid_batch_set_maps_host, ptr_h, None),
        "host_10pct": set_call(lib.eb_grid_batch_set_maps_host, ptr_h, few),
    }, max(1, a.steps // 2), a.rounds)

    # robots inside their maps; validate_control / DWA inputs
    fx = rng.uniform(0.1, 0.9, B)
    fy = rng.uniform(0.1, 0.9, B)
    x0_h = np.column_stack([origin[:, 0] + fx * sides[:, 1] * RES, origin[:, 1] + fy * sides[:, 0] * RES,
                            rng.uniform(-np.pi, np.pi, B)])
    u_h = np.column_stack([rng.uniform(-1, 1, B), rng.uniform(-1, 1, B), rng.uniform(-2, 2, B)])
    t = np.arange(50) * 0.1
    xt_h = x0_h[:, None, :] + np.stack([np.cos(0.7 * t), np.sin(0.9 * t), np.sin(0.5 * t)], axis=-1)[None] * 0.5
    x0, u, vb = (torch.from_numpy(np.ascontiguousarray(v)).to(dev) for v in (x0_h, u_h, u_h))
    xt = torch.from_numpy(np.ascontiguousarray(xt_h)).to(dev)
    out = torch.empty(B, dtype=torch.int32, device=dev)
    uo = torch.empty((B, 3), dtype=torch.float64, device=dev)
    col = capi.EbCollision(*COL)
    dwa = capi.EbDwa(*DWA, *SAMPLES)
    P = lambda x: C.c_void_p(x.data_ptr())

    # (b) one shared map of the median size, dilation off; the robots re-centred into it
    ys0, xs0 = (int(v) for v in np.median(sides, axis=0))
    shared = torch.zeros((ys0, xs0), dtype=torch.int8)
    shared[torch.rand((ys0, xs0)) < 0.004] = 100
    g_sh = eb.GridMap(0.0, xs0 * RES, 0.0, ys0 * RES, RES, shared.numpy())
    g_sh.dilation(1)
    lib.eb_grid_set_stream(g_sh._h, s)
    x0s_h = np.column_stack([fx * xs0 * RES, fy * ys0 * RES, x0_h[:, 2]])
    x0s = torch.from_numpy(x0s_h).to(dev)
    xts = torch.from_numpy(np.ascontiguousarray(xt_h - x0_h[:, None, :] + x0s_h[:, None, :])).to(dev)

    # (a) one eb_grid per robot, the first BL maps
    loop = []
    for i in range(BL):
        ys, xs = cells_h[i].shape
        g = eb.GridMap(origin[i, 0], origin[i, 0] + xs * RES, origin[i, 1], origin[i, 1] + ys * RES, RES, cells_h[i])
        g.dilation(1)
        lib.eb_grid_set_stream(g._h, s)
        loop.append(g)
    x0_p = [C.c_void_p(x0.data_ptr() + 24 * i) for i in range(BL)]
    u_p = [C.c_void_p(u.data_ptr() + 24 * i) for i in range(BL)]
    o_p = [C.c_void_p(out.data_ptr() + 4 * i) for i in range(BL)]
    uo_p = [C.c_void_p(uo.data_ptr() + 24 * i) for i in range(BL)]
    xt_p = [C.c_void_p(xt.data_ptr() + 8 * 150 * i) for i in range(BL)]

    def ok(st):
        assert st == 0, lib.eb_last_error()

    calls = {
        "collision_check": {
            "per_map": lambda: ok(lib.eb_collision_check_batch_dev(gb._h, col, P(x0), 1, P(out))),
            "shared": lambda: ok(lib.eb_collision_check_dev(g_sh._h, col, P(x0s), B, P(out))),
            "loop": lambda: [ok(lib.eb_collision_check_dev(loop[i]._h, col, x0_p[i], 1, o_p[i])) for i in range(BL)],
        },
        "validate_control": {
            "per_map": lambda: ok(lib.eb_validate_control_batch_dev(gb._h, col, P(x0), P(u), 1, 0.1, 0.5, P(out))),
            "shared": lambda: ok(lib.eb_validate_control_dev(g_sh._h, col, P(x0s), P(u), B, 0.1, 0.5, P(out))),
            "loop": lambda: [ok(lib.eb_validate_control_dev(loop[i]._h, col, x0_p[i], u_p[i], 1, 0.1, 0.5, o_p[i]))
                             for i in range(BL)],
        },
        "dwa_twist": {
            "per_map": lambda: ok(lib.eb_dwa_control_twist_batch_dev(gb._h, col, dwa, P(x0), P(vb), P(u), P(out), P(uo),
                                                                     None)),
            "shared": lambda: ok(lib.eb_dwa_control_twist_dev(g_sh._h, col, dwa, P(x0s), P(vb), P(u), B, P(out), P(uo),
                                                              None)),
            "loop": lambda: [ok(lib.eb_dwa_control_twist_dev(loop[i]._h, col, dwa, x0_p[i], u_p[i], u_p[i], 1, o_p[i],
                                                             uo_p[i], None)) for i in range(BL)],
        },
        "dwa_traj": {
            "per_map": lambda: ok(lib.eb_dwa_control_traj_batch_dev(gb._h, col, dwa, P(x0), P(vb), P(xt), 50, 1, 0.1,
                                                                    P(out), P(uo), None)),
            "shared": lambda: ok(lib.eb_dwa_control_traj_dev(g_sh._h, col, dwa, P(x0s), P(vb), P(xts), 50, 1, 0.1, B,
                                                             P(out), P(uo), None)),
            "loop": lambda: [ok(lib.eb_dwa_control_traj_dev(loop[i]._h, col, dwa, x0_p[i], u_p[i], xt_p[i], 50, 0, 0.1,
                                                            1, o_p[i], uo_p[i], None)) for i in range(BL)],
        },
    }
    r_bnd, r_col, r_max = int(COL[0] / RES), int((COL[0] + COL[2]) / RES), int(COL[1] / RES)
    probes_pose = sum(circle_cells(r) for r in range(r_bnd, min(r_max, r_col) + 1))
    poses = {"collision_check": 1, "validate_control": 5, "dwa_twist": 120 * 20, "dwa_traj": 120 * 20}
    checks = {}
    for name, fns in calls.items():
        us = time_rounds(torch, fns, a.steps, a.rounds)
        per_robot = {"per_map": us["per_map"] / B, "shared": us["shared"] / B, "loop": us["loop"] / BL}
        checks[name] = {
            "us_per_call": {"per_map_B": us["per_map"], "shared_B": us["shared"], "loop_BL": us["loop"]},
            "ns_per_robot": {k: v * 1e3 for k, v in per_robot.items()},
            "per_map_vs_loop_speedup_per_robot": per_robot["loop"] / per_robot["per_map"],
            "per_map_vs_shared_time_ratio": us["per_map"] / us["shared"],
            "per_map_gprobes_per_s": B * poses[name] * probes_pose / (us["per_map"] * 1e-6) / 1e9,
            "shared_gprobes_per_s": B * poses[name] * probes_pose / (us["shared"] * 1e-6) / 1e9,
        }
    name, power = card()
    print(json.dumps({
        "card": name, "power_limit": power, "batch": B, "loop_batch": BL, "steps": a.steps, "rounds": a.rounds,
        "maps": f"{B} maps, sides uniform in [160, 640] cells at {RES} m, 0.4 % occupied, {total_bytes / 1e6:.0f} MB",
        "shared_map": f"{xs0} x {ys0} cells at {RES} m ({xs0 * ys0 / 1e6:.2f} MB), dilation off",
        "l2": f"per-map working set {total_bytes / 1e6:.0f} MB > 126 MB L2: probes come from HBM; the shared map is "
              "L2-resident.  No share of peak is quoted.",
        "probes_per_pose": probes_pose, "set_maps_us": set_times, "checks": checks,
    }))


if __name__ == "__main__":
    main()
