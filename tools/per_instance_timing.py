"""Per-instance targets vs the shared target: step times of the solve at the C2 and C5 shapes, the cost of the frame
launch, and target_batch_kernel (configTarget of every instance) with all instances rebuilding.

Prints one JSON line.  CUDA events around K back-to-back steps after a warm-up; the variants of one shape are
alternated in the same process (rounds of A, B, C, ...) and the median of the rounds is reported.  L2 is not flushed:
the step working sets (C2: ~10 MB, C5: ~100 MB of ut / replay rows) are what a control loop touches every tick.

    python tools/per_instance_timing.py [--steps K] [--rounds R]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [v.strip() for v in out.split(",")]
        return name, power
    except Exception as e:  # the numbers are still reported, the card is named as unknown
        return f"unknown ({e})", "unknown"


def gpu(eb, B, nb, batch_size=100, buffer_size=1000000):
    R, umin, umax = np.diag([1.0, 1.0, 2.0]), [-1.0, -1.0, -2.0], [1.0, 1.0, 2.0]
    return eb.ErgodicControl(eb.Omni(), 0.1, 5.0, 0.1, 1.0, nb, buffer_size, batch_size, R, umin, umax, batch=B)


def time_rounds(torch, fns, steps, rounds):
    """fns: name -> callable(one step).  Alternated per round; returns name -> median us per step"""
    res = {k: [] for k in fns}
    for f in fns.values():
        for _ in range(3):
            f()
    torch.cuda.synchronize()
    for _ in range(rounds):
        for k, f in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps):
                f()
            b.record()
            b.synchronize()
            res[k].append(a.elapsed_time(b) * 1e3 / steps)
    return {k: float(np.median(v)) for k, v in res.items()}


def step_shape(torch, eb, B, nb, stored, steps, rounds, rng):
    """shared vs per-instance (replicated rows and frames / distinct frames), bounds None and bounds unchanged"""
    dev = torch.device("cuda")
    bounds = (0.0, 10.0, 0.0, 10.0)
    mk = lambda: gpu(eb, B, nb)  # noqa: E731
    shared, rep, dis = mk(), mk(), mk()
    mu, sg = [[2.5, 2.5], [8.5, 2.5]], [[1.5, 1.5], [1.5, 1.5]]
    shared.setTarget([eb.Gaussian(m, s) for m, s in zip(mu, sg)])
    shared.configTarget(bounds)
    ph, lx, ly = shared.get_phik()
    rep.set_phik_batch(torch.from_numpy(np.tile(ph, (B, 1))).to(dev), torch.tensor([[lx, ly]] * B, dtype=torch.float64, device=dev))
    bb = torch.tensor([bounds] * B, dtype=torch.float64, device=dev)
    # distinct frames: every instance its own origin and 10..12 m extent, the same two Gaussians in its frame
    off = rng.uniform(-20, 20, (B, 2))
    ext = 10.0 + np.round(rng.uniform(0, 2, (B, 2)), 1)
    bd = np.column_stack([off[:, 0], off[:, 0] + ext[:, 0], off[:, 1], off[:, 1] + ext[:, 1]])
    dis.setTargets([[eb.Gaussian(np.array(m) + off[i], s) for m, s in zip(mu, sg)] for i in range(B)])
    dis.configTargets(bd)
    bdd = torch.from_numpy(bd).to(dev)
    x = torch.from_numpy(np.column_stack([rng.uniform(1, 9, B), rng.uniform(1, 9, B), rng.uniform(-3, 3, B)])).to(dev)
    xd = x.clone()
    xd[:, 0] += bdd[:, 0]
    xd[:, 1] += bdd[:, 2]
    ut = rng.uniform([-1, -1, -2], [1, 1, 2], size=(B, shared.steps, 3)) * 0.5
    for c in (shared, rep, dis):
        c.set_ut(ut)
        for _ in range(stored):
            c.addStateMemory(x)
    u0 = torch.empty((B, 3), dtype=torch.float64, device=dev)
    # bit identity of the replicated mode at the timed size (one step each from the same state)
    a = shared.clone()
    b = rep.clone()
    ua, ub = torch.empty_like(u0), torch.empty_like(u0)
    ma, mb = torch.empty(B, dtype=torch.float64, device=dev), torch.empty(B, dtype=torch.float64, device=dev)
    a.control(bounds, x, u0=ua, metric=ma)
    b.control(None, x, u0=ub, metric=mb)
    torch.cuda.synchronize()
    identical = bool(torch.equal(ua, ub) and torch.equal(ma, mb) and np.array_equal(a.get_ut(), b.get_ut())
                     and np.array_equal(a.get_ck(), b.get_ck()))
    fns = {
        "shared": lambda: shared.control(bounds, x, u0=u0),
        "per_inst_replicated_bounds_none": lambda: rep.control(None, x, u0=u0),
        "per_inst_distinct_bounds_none": lambda: dis.control(None, xd, u0=u0),
        "per_inst_replicated_bounds_unchanged": lambda: rep.control(bb, x, u0=u0),
        "per_inst_distinct_bounds_unchanged": lambda: dis.control(bdd, xd, u0=u0),
    }
    t = time_rounds(torch, fns, steps, rounds)
    for c in (shared, rep, dis):
        c.check()
    out = {"B": B, "nb": nb, "N": shared.steps, "stored": stored, "us_per_step": t,
           "per_inst_vs_shared_bounds_none": t["per_inst_replicated_bounds_none"] / t["shared"],
           "bit_identical_replicated_vs_shared": identical}
    return out


def target_shape(torch, eb, capi, nb, steps, rng):
    """target_batch_kernel: 4096 instances on their own 10..30 m maps at 0.1 m, 2..4 Gaussians, every instance
    rebuilding on every call (the extents alternate between two values)"""
    B, res = 4096, 0.1
    dev = torch.device("cuda")
    c = gpu(eb, B, nb)
    ext = np.round(rng.uniform(10, 30, (B, 2)), 1)
    ng = rng.integers(2, 5, B)
    c.setTargets([[eb.Gaussian(rng.uniform(1, ext[i] - 1), rng.uniform(0.8, 2.5, 2)) for _ in range(ng[i])]
                  for i in range(B)])
    b0 = np.column_stack([np.zeros(B), ext[:, 0], np.zeros(B), ext[:, 1]])
    b1 = b0.copy()
    b1[:, 1] += res  # one more column: every instance rebuilds when the two alternate
    t0, t1 = torch.from_numpy(b0).to(dev), torch.from_numpy(b1).to(dev)
    lib = capi.load()
    c._sync_stream()

    def call(t):
        capi.check(lib.eb_config_target_batch_dev(c._h, C.c_void_p(t.data_ptr()), None))

    for _ in range(2):
        call(t0)
        call(t1)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for k in range(steps):
        call(t1 if k % 2 else t0)
    b.record()
    b.synchronize()
    c.check()
    ms = a.elapsed_time(b) / steps
    flops, exps = 0.0, 0.0
    for k in range(2):
        bb = b1 if k else b0
        nx = np.round((bb[:, 1] - bb[:, 0]) / res) + 1
        ny = np.round((bb[:, 3] - bb[:, 2]) / res) + 1
        flops += float(np.sum(2 * nx * ny * nb + 2 * ny * nb * nb)) / 2
        exps += float(np.sum(nx * ny * ng)) / 2
    dfma = C.c_double(0)
    dmma = C.c_double(0)
    capi.check(lib.eb_fp64_peak(0, C.byref(dfma), C.byref(dmma)))
    return {"B": B, "nb": nb, "ms_per_call": ms, "F_flop": flops, "exp_count": exps,
            "fp64_tflops": flops / (ms * 1e-3) / 1e12, "eb_fp64_peak_dfma_tflops": dfma.value,
            "share_of_dfma_peak": flops / (ms * 1e-3) / 1e12 / dfma.value if dfma.value > 0 else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    import torch

    import ergodic_exploration_b200 as eb
    from ergodic_exploration_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("per_instance_timing.py measures on the GPU; no CUDA device is visible")
    name, power = card()
    rng = np.random.default_rng(0)
    res = {"card": name, "power_limit": power, "method": "CUDA events, warm-up, K back-to-back steps, variants "
           "alternated per round, median of rounds; L2 not flushed", "steps": args.steps, "rounds": args.rounds}
    res["c2"] = step_shape(torch, eb, 4096, 10, 0, args.steps, args.rounds, rng)
    res["c5"] = step_shape(torch, eb, 65536, 16, 100, max(20, args.steps // 10), args.rounds, rng)
    res["target_batch"] = [target_shape(torch, eb, capi, nb, 20, rng) for nb in (10, 16)]
    print(json.dumps(res))


if __name__ == "__main__":
    main()
