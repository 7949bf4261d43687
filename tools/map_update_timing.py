"""Map updates of B robots on B maps: (a) the whole-map flow, eb_grid_batch_set_maps_* followed by
eb_set_map_targets_batch_* of the same cells, against (b) the row-band flow, eb_grid_batch_set_rows_* followed by
eb_set_map_targets_from_grid_batch with the same bands declared, which recomputes only the 64-row units the bands meet.

K4 setup: B = 4096 maps of 160..640 cells a side at 0.05 m (several hundred MB, far more than the 126 MB of L2; L2 is
not flushed).  Each case updates 10 % or 100 % of the maps with one band of 64 or 256 rows (at most the map) at a
random row, through the _host or the _dev forms, at nb 10 and 16; (a) sends the same maps whole.  Also
eb_set_map_targets_from_grid_batch with NULL ranges (every unit of every map) against eb_set_map_targets_batch_dev.
CUDA events around K back-to-back flows after a warm-up, the two flows of a case alternated in rounds
(tools/per_instance_timing.time_rounds), medians in microseconds per flow.  Every call is made through ctypes on
torch's current stream, so the host cost of enqueueing and packing is part of each time.  Prints one JSON line with
the card's name and power limit.

    python tools/map_update_timing.py [--batch B] [--steps K] [--rounds R]
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

RES = 0.05


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()

    import torch

    import ergodic_exploration_b200 as eb
    from ergodic_exploration_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("map_update_timing needs a CUDA device")
    lib = capi.load()
    dev = torch.device("cuda")
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rng = np.random.default_rng(0)
    B = a.batch
    sides = rng.integers(160, 641, size=(B, 2))  # (ysize, xsize)
    gen = torch.Generator(device=dev).manual_seed(0)
    cells = [torch.randint(-1, 101, (int(ys), int(xs)), generator=gen, device=dev, dtype=torch.int8)
             for ys, xs in sides]
    cells_h = [c.cpu().numpy() for c in cells]
    origin = np.ascontiguousarray(np.column_stack([rng.uniform(-50, 50, B), rng.uniform(-50, 50, B)]))
    xs_a = np.ascontiguousarray(sides[:, 1], dtype=np.uint32)
    ys_a = np.ascontiguousarray(sides[:, 0], dtype=np.uint32)
    res_a = np.full(B, RES)
    ptr = {"dev": (C.c_void_p * B)(*[c.data_ptr() for c in cells]),
           "host": (C.c_void_p * B)(*[c.ctypes.data for c in cells_h])}
    units = int(sum((int(ys) + 63) // 64 for ys, _ in sides))

    def ok(st):
        assert st == 0, lib.eb_last_error()

    def flows(nb, path, band, frac):
        gba, gbb = eb.GridMapBatch(B), eb.GridMapBatch(B)
        ca, cb = gpu(eb, B, nb, buffer_size=1000), gpu(eb, B, nb, buffer_size=1000)
        for g in (gba, gbb):
            g.set(cells, RES, origin)
            lib.eb_grid_batch_set_stream(g._h, s)
        for c in (ca, cb):
            lib.eb_set_stream(c._h, s)
        cb.setMapTargets(gbb)
        upd = np.zeros(B, dtype=np.int32)
        upd[rng.choice(B, max(1, int(round(frac * B))), replace=False)] = 1
        rc = np.ascontiguousarray(np.where(upd == 1, np.minimum(band, sides[:, 0]), 0), dtype=np.uint32)
        rb = np.ascontiguousarray([int(rng.integers(0, ys - n + 1)) for (ys, _), n in zip(sides, rc)], dtype=np.uint32)
        if path == "dev":
            bands = (C.c_void_p * B)(*[cells[i][rb[i]:].data_ptr() for i in range(B)])
        else:
            bands = (C.c_void_p * B)(*[cells_h[i][rb[i]:].ctypes.data for i in range(B)])
        set_maps = lib.eb_grid_batch_set_maps_dev if path == "dev" else lib.eb_grid_batch_set_maps_host
        targets = lib.eb_set_map_targets_batch_dev if path == "dev" else lib.eb_set_map_targets_batch_host
        set_rows = lib.eb_grid_batch_set_rows_dev if path == "dev" else lib.eb_grid_batch_set_rows_host
        P = lambda v: v.ctypes.data  # noqa: E731

        def whole():
            ok(set_maps(gba._h, C.addressof(ptr[path]), P(xs_a), P(ys_a), P(res_a), P(origin), P(upd)))
            ok(targets(ca._h, C.addressof(ptr[path]), P(xs_a), P(ys_a), P(res_a), P(origin), P(upd)))

        def rows():
            ok(set_rows(gbb._h, C.addressof(bands), P(rb), P(rc), P(upd)))
            ok(lib.eb_set_map_targets_from_grid_batch(cb._h, gbb._h, P(rb), P(rc), P(upd)))

        t = time_rounds(torch, {"whole": whole, "rows": rows}, a.steps, a.rounds)
        recomputed = int(sum(((int(b) + int(n) - 1) // 64 - int(b) // 64 + 1) if n else 0 for b, n in zip(rb, rc)))
        return {"nb": nb, "path": path, "band": band, "maps_pct": int(round(100 * frac)), "whole_us": t["whole"],
                "rows_us": t["rows"], "speedup": t["whole"] / t["rows"], "units_recomputed": recomputed,
                "band_bytes": int(sum(int(n) * int(x) for n, x in zip(rc, xs_a))),
                "whole_bytes": int(sum(int(y) * int(x) for y, x, f in zip(ys_a, xs_a, upd) if f))}

    cases = []
    full = []
    for nb in (10, 16):
        for path in ("host", "dev"):
            for band in (64, 256):
                for frac in (0.1, 1.0):
                    cases.append(flows(nb, path, band, frac))
                    torch.cuda.empty_cache()
        # every unit of every map: the kept-block call with NULL ranges against the pointer call
        gb = eb.GridMapBatch(B)
        gb.set(cells, RES, origin)
        lib.eb_grid_batch_set_stream(gb._h, s)
        ca, cb = gpu(eb, B, nb, buffer_size=1000), gpu(eb, B, nb, buffer_size=1000)
        for c in (ca, cb):
            lib.eb_set_stream(c._h, s)
        t = time_rounds(torch, {
            "pointer_dev": lambda: ok(lib.eb_set_map_targets_batch_dev(
                ca._h, C.addressof(ptr["dev"]), xs_a.ctypes.data, ys_a.ctypes.data, res_a.ctypes.data,
                origin.ctypes.data, None)),
            "grid_batch_null_ranges": lambda: ok(lib.eb_set_map_targets_from_grid_batch(cb._h, gb._h, None, None,
                                                                                         None)),
        }, a.steps, a.rounds)
        full.append({"nb": nb, **{k + "_us": v for k, v in t.items()}})
        del gb, ca, cb
        torch.cuda.empty_cache()
    name, power = card()
    print(json.dumps({"card": name, "power_limit": power, "batch": B, "units": units,
                      "kept_block_bytes": {str(nb): units * nb * nb * 8 for nb in (10, 16, 32, 64)},
                      "steps": a.steps, "rounds": a.rounds, "cases": cases, "whole_maps": full}))


if __name__ == "__main__":
    main()
