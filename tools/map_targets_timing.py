"""Map-derived targets of a per-instance controller: the one-launch call (eb_set_map_targets_batch_dev) against the
route it replaces (one eb_map_target_execute_dev per map into its row, then eb_set_phik_batch_dev).

Prints one JSON line.  CUDA events around K back-to-back calls after a warm-up; the routes of one case are alternated
in the same process (rounds of new, old, new 10 %, old 10 %) and the median of the rounds is reported.  Both routes
are driven through ctypes with prepared pointer arrays, so the host cost of enqueueing is part of each time.  L2 is
not flushed: B = 64 maps (a few MB of cells) are read from L2 after the first pass, B >= 1024 maps (> 100 MB) and the
2048^2 maps are not.  FLOP count per call: F = sum_i (2 nx_i ny_i nb + 2 ny_i nb^2), over the maps of the call.

    python tools/map_targets_timing.py [--steps K] [--rounds R] [--quick]
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


def case(torch, eb, lib, shapes, nb, res, steps, rounds, rng, dmma_tflops):
    dev = torch.device("cuda")
    B = len(shapes)
    cells = [torch.from_numpy(rng.integers(-1, 101, size=(ny, nx)).astype(np.int8)).to(dev) for nx, ny in shapes]
    xs = np.array([nx for nx, _ in shapes], dtype=np.uint32)
    ys = np.array([ny for _, ny in shapes], dtype=np.uint32)
    rs = np.full(B, res)
    org = np.zeros((B, 2))
    ptrs = (C.c_void_p * B)(*[c.data_ptr() for c in cells])
    flag = np.zeros(B, dtype=np.int32)
    flag[rng.choice(B, max(1, B // 10), replace=False)] = 1
    new = gpu(eb, B, nb)
    old = gpu(eb, B, nb)
    s = torch.cuda.current_stream().cuda_stream
    for c in (new, old):
        c._lib.eb_set_stream(c._h, C.c_void_p(s))
    mts = [eb.MapTarget(nx, ny, res, nb) for nx, ny in shapes]
    for m in mts:
        lib.eb_map_target_set_stream(m._h, C.c_void_p(s))
    K = nb * nb
    rows = torch.empty((B, K), dtype=torch.float64, device=dev)
    ext = torch.tensor([[nx * res, ny * res] for nx, ny in shapes], dtype=torch.float64, device=dev)
    row_p = [rows[i].data_ptr() for i in range(B)]
    mt_h = [m._h for m in mts]
    cell_p = [c.data_ptr() for c in cells]
    flagged = np.flatnonzero(flag)

    def run_new(upd=None):
        st = lib.eb_set_map_targets_batch_dev(new._h, C.addressof(ptrs), xs.ctypes.data, ys.ctypes.data, rs.ctypes.data,
                                              org.ctypes.data, upd.ctypes.data if upd is not None else None)
        assert st == 0, lib.eb_last_error()

    def run_old(which):
        for i in which:
            lib.eb_map_target_execute_dev(mt_h[i], cell_p[i], row_p[i], None)
        assert lib.eb_set_phik_batch_dev(old._h, rows.data_ptr(), ext.data_ptr()) == 0, lib.eb_last_error()

    every = range(B)
    t = time_rounds(torch, {"new": run_new, "old": lambda: run_old(every), "new_10pct": lambda: run_new(flag),
                            "old_10pct": lambda: run_old(flagged)}, steps, rounds)
    # both routes give the same rows to rounding
    run_new()
    run_old(every)
    torch.cuda.synchronize()
    a, _ = new.get_phik_batch()
    b, _ = old.get_phik_batch()
    err = float(np.max(np.abs(a - b)))
    cells_n = float(sum(nx * ny for nx, ny in shapes))
    flop = float(sum(2.0 * nx * ny * nb + 2.0 * ny * nb * nb for nx, ny in shapes))
    fl10 = float(sum(2.0 * shapes[i][0] * shapes[i][1] * nb + 2.0 * shapes[i][1] * nb * nb for i in flagged))
    out = {"B": B, "nb": nb, "cells": cells_n, "max_abs_diff_new_vs_old": err}
    for k, v in t.items():
        out[f"{k}_us"] = round(v, 2)
    out["speedup"] = round(t["old"] / t["new"], 2)
    out["speedup_10pct"] = round(t["old_10pct"] / t["new_10pct"], 2)
    out["new_cells_per_s"] = cells_n / (t["new"] * 1e-6)
    out["new_tflops"] = flop / (t["new"] * 1e-6) / 1e12
    out["new_dmma_share"] = out["new_tflops"] / dmma_tflops
    out["new_10pct_tflops"] = fl10 / (t["new_10pct"] * 1e-6) / 1e12
    for m in mts:
        m.close()
    new.close()
    old.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--quick", action="store_true", help="one small case (smoke run of the tool)")
    args = ap.parse_args()
    import torch

    import ergodic_exploration_b200 as eb
    from ergodic_exploration_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("map_targets_timing: no CUDA device (the numbers are GPU times; there is no CPU fallback)")
    lib = capi.load()
    name, power = card()
    _, dmma = eb.fp64_peak()
    rng = np.random.default_rng(2024)
    res = {"card": name, "power_limit": power, "dmma_peak_tflops": dmma, "cases": []}
    sizes = [64] if args.quick else [64, 1024, 4096]
    nbs = [10] if args.quick else [10, 16, 32]
    for B in sizes:
        shapes = [tuple(int(v) for v in rng.integers(100, 401, 2)) for _ in range(B)]
        for nb in nbs:
            res["cases"].append(case(torch, eb, lib, shapes, nb, 0.05, args.steps, args.rounds, rng, dmma))
    if not args.quick:
        res["cases"].append(case(torch, eb, lib, [(2048, 2048)] * 8, 16, 0.05, args.steps, args.rounds, rng, dmma))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
