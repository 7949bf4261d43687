#!/usr/bin/env python
"""bench.py -- ergodic control solves/sec and phi_k cells*bases/sec on B200 (BASELINE.json metrics).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload all|c2|c2big|c3|c4|c5|c5loop|entropy|collide|dwa] [--loop-steps L]
                    [--dump-outputs DIR]

One "step" = one batched ErgodicControl::control() iteration (ONE fused CUDA kernel) over the
workload's instances.  The PRIMARY line (`value`) is BASELINE.json configs[1] ("c2": Omni, 10x10 basis,
4096 instances per GPU, 50-step horizon, shared two-Gaussian target, warm control signals).  With
--workload all (the default) the same JSON line carries a `secondary` array with the other configs,
each with its own ms_per_step / roofline / e2e / clocks (and cpu_baseline at N = 1):
  c3      configs[2]: phi_k over an 8192 x 8192 density, 32 x 32 basis      (cells*bases/s; N > 1: rows sharded)
  c4      configs[3] shard: SimpleCart, 20 x 20 basis, 100-step horizon, 131072 instances per GPU (weak: 2^20 on 8 GPUs)
  c5      configs[4] step : Omni, 16 x 16 basis, 100 replay states, 65536 instances IN TOTAL (strong)
  c5loop  configs[4]      : the closed receding-horizon loop, 65536 instances IN TOTAL (strong), 1000 ticks
  entropy map-derived target (numerics.hpp:164-179): int8 occupancy grid -> density -> phi_k

Timing (N = world size, launched by torchrun: one process per GPU):
  * solve workloads: one CUDA-event pair per step on the launching stream, max over ranks.  N > 1: the pair
    also contains the gather of the first twists -- the step ends when EVERY rank's rows of this step have
    arrived in this rank's gathered buffer (P2P stores over NVLink + arrival flags, csrc/peer_gather.cuh).
  * c5loop: ONE event pair around the whole loop (addStateMemory + control + gather + wait + plant per tick).
  * e2e: the same metric through the host-buffer entry points with pinned host memory, copies inside the
    timed region.  N > 1: pinned x -> H2D -> control + fused gather -> wait -> D2H of the GATHERED twists.
--impl reference times the reference's own CPU implementation (oracle/_ref) on all host cores.
--dump-outputs DIR writes what the primary workload's timed path returned in its last timed step: u0.npy (first
twists), metric.npy and ut.npy (the warm-started control signals of the controller that step used), float64.  N > 1:
u0 holds the gathered rows of every rank, metric and ut rank 0's rows.  The inputs are seeded, so two builds run with
the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: model, nb, horizon, batch (per GPU for weak / total for strong scaling), memory states
    "c2": dict(model=1, nb=10, horizon=5.0, batch=4096, mem=0, scaling="weak",
               desc="configs[1]: Omni, 10x10 basis, 4096 instances, 50-step horizon"),
    "c2big": dict(model=1, nb=10, horizon=5.0, batch=262144, mem=0, scaling="weak",
                  desc="configs[1] shape at 64x the batch: Omni, 10x10 basis, 262144 instances, 50-step horizon"),
    "c4": dict(model=0, nb=20, horizon=10.0, batch=131072, mem=0, scaling="weak",
               desc="configs[3] shard: SimpleCart, 20x20 basis, 131072 instances/GPU, 100-step horizon"),
    "c5": dict(model=1, nb=16, horizon=5.0, batch=65536, mem=100, scaling="strong",
               desc="configs[4] step: Omni, 16x16 basis, 65536 instances in total, 50-step horizon, 100 replay states"),
}
BOUNDS = (0.0, 10.0, 0.0, 10.0)
MU = [[2.5, 2.5], [8.5, 2.5]]
SIGMA = [[1.5, 1.5], [1.5, 1.5]]
DT = 0.1
METRIC_SOLVE = "ergodic control solves/sec (batched)"


def model_params(model):
    if model == 1:
        return np.diag([1.0, 1.0, 2.0]), np.array([-1.0, -1.0, -2.0]), np.array([1.0, 1.0, 2.0])
    return np.diag([1.0, 0.0, 2.0]), np.array([-1.0, 0.0, -2.0]), np.array([1.0, 0.0, 2.0])


def flops_per_solve(K, N, M):
    """SURVEY.md section 8(d): algorithmic FP64 work of one control()"""
    return 2 * K * (N + M) + 4 * K * N + 2 * K + 200 * N


def bytes_per_solve(N, M):
    """SURVEY.md section 8(d): ut_ read + write, x, u0, metric, memory gather"""
    return 2 * 24 * N + 24 + 24 + 8 + 24 * M


def synth_inputs(wl, batch, seed):
    """synthetic inputs (SURVEY section 8d): x0 ~ U([0.5,9.5]^2 x [-pi,pi)), warm ut_ ~ 0.5 U(umin,umax)"""
    rng = np.random.default_rng(seed)
    _, umin, umax = model_params(wl["model"])
    steps = int(abs(wl["horizon"] / DT))
    x = np.column_stack([rng.uniform(0.5, 9.5, batch), rng.uniform(0.5, 9.5, batch),
                         rng.uniform(-np.pi, np.pi, batch)])
    ut = rng.uniform(umin, umax, size=(batch, steps, 3)) * 0.5
    mem = np.stack([np.column_stack([rng.uniform(0.5, 9.5, batch), rng.uniform(0.5, 9.5, batch),
                                     rng.uniform(-np.pi, np.pi, batch)]) for _ in range(wl["mem"])]) \
        if wl["mem"] else None
    return x, ut, mem


# --------------------------------------------------------------------------
# clocks: NVML polled from a thread (2 ms period), so that sub-millisecond timed regions still see samples
# --------------------------------------------------------------------------
class ClockSampler:
    """SM clock / throttle reasons of one GPU, sampled for the whole GPU arm; `region()` marks the
    timed regions, and the summary reports the samples that fell inside them ("under load")."""

    REASONS = (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40),
               ("sw_power_cap", 0x4), ("hw_power_brake", 0x80))

    def __init__(self, torch_device_index):
        self.idx = torch_device_index
        self.samples = []   # (t, sm_mhz, reasons_mask, power_w)
        self.regions = []   # (name, t0, t1)
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self._nvml = None

    def start(self):
        try:
            import pynvml
            import torch

            pynvml.nvmlInit()
            h = None
            try:
                uuid = str(torch.cuda.get_device_properties(self.idx).uuid)
                uuid = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
                h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, "encode") else uuid)
            except Exception:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES")
                phys = int(vis.split(",")[self.idx]) if vis and vis.split(",")[self.idx].isdigit() else self.idx
                h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self._nvml, self._h = pynvml, h
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._poll, daemon=True)
            self._thread.start()
        except Exception:
            self._nvml = None

    def _poll(self):
        nv, h = self._nvml, self._h
        reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop.is_set():
            try:
                t = time.perf_counter()
                mhz = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                mask = reasons(h)
                try:
                    pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                except Exception:
                    pw = None
                self.samples.append((t, float(mhz), int(mask), pw))
            except Exception:
                pass
            time.sleep(0.002)

    class _Region:
        def __init__(self, outer, name):
            self.o, self.name = outer, name

        def __enter__(self):
            self.t0 = time.perf_counter()

        def __exit__(self, *a):
            self.o.regions.append((self.name, self.t0, time.perf_counter()))

    def region(self, name):
        return ClockSampler._Region(self, name)

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=1.0)

    def summary(self, name=None):
        """clocks over the timed regions called `name` (all timed regions when None)"""
        regs = [(a, b) for n, a, b in self.regions if name is None or n == name]
        # NVML answers take ~1 ms: widen a short region by one polling period on either side
        inside = [s for s in self.samples if any(a - 0.004 <= s[0] <= b + 0.004 for a, b in regs)]
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0,
                    "source": "nvml" if self._nvml else "unavailable"}
        mask = 0
        for s in inside:
            mask |= s[2]
        pw = [s[3] for s in inside if s[3] is not None]
        return {"sm_mhz": float(np.median([s[1] for s in inside])), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(n for n, bit in self.REASONS if mask & bit), "samples": len(inside),
                "power_w_max": max(pw) if pw else None, "source": "nvml, 2 ms polling thread"}


# --------------------------------------------------------------------------
# CPU reference arm
# --------------------------------------------------------------------------
def cpu_reference_rate(wl, sample, steps, warmup, threads=None):
    """Times the reference's CPU control() (oracle/_ref when the compiled
    reference is available, else the C port) on `sample` instances of the
    workload, spread over all host cores, one controller object per instance."""
    import ctypes as C

    from oracle import pyoracle
    from oracle.pyoracle import Oracle, RefLib

    pyoracle.build()
    use_ref = RefLib.available()
    lib = RefLib if use_ref else Oracle
    threads = threads or os.cpu_count() or 1
    x, ut, mem = synth_inputs(wl, sample, seed=0xE16C0D1C + 2)
    R, umin, umax = model_params(wl["model"])
    ctrls = []
    for i in range(sample):
        c = lib.create(wl["model"], DT, wl["horizon"], 0.1, 1.0, wl["nb"], 1000000, 100, R, umin, umax)
        c.set_target(MU, SIGMA)
        c.set_ut(ut[i])
        if mem is not None:
            for m in mem:
                c.add_state_memory(m[i])
        ctrls.append(c)
    handles = (C.c_void_p * sample)(*[c._h for c in ctrls])
    u0 = np.zeros((sample, 3))
    clib = lib.lib()
    per = (sample + threads - 1) // threads
    chunks = [(lo, min(sample, lo + per)) for lo in range(0, sample, per)]
    b = [C.c_double(v) for v in BOUNDS]
    dp = C.POINTER(C.c_double)

    def work(lo, hi):
        hs = C.cast(C.byref(handles, lo * C.sizeof(C.c_void_p)), C.POINTER(C.c_void_p))
        xp = x[lo:hi].ctypes.data_as(dp)
        up = u0[lo:hi].ctypes.data_as(dp)
        if use_ref:
            clib.ref_control_many(hs, hi - lo, *b, C.c_double(0.1), xp, up)
        else:
            clib.eo_control_many(hs, hi - lo, *b, xp, up)

    def one_step():
        ts = [threading.Thread(target=work, args=ch) for ch in chunks]
        [t.start() for t in ts]
        [t.join() for t in ts]

    for _ in range(max(1, warmup)):  # first call builds phi_k (excluded, BASELINE.md section 3)
        one_step()
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    dt = time.perf_counter() - t0
    return {
        "value": sample * steps / dt,
        "unit": "solves/s",
        "cores": len(chunks),
        "kind": "reference" if use_ref else "port",
        "sample": f"{sample} instances x {steps} control() steps of the workload, {len(chunks)} host threads, "
                  f"one controller object per instance"
                  + ("" if use_ref else " (C port: compiled reference oracle/_ref not present)"),
        "ms_per_step": dt / steps * 1e3,
    }


def run_reference(args, rank, world):
    if rank != 0:
        return
    key = "c2" if args.workload == "all" else args.workload
    if key == "c5loop":
        key = "c5"
    if key not in WORKLOADS:
        print(json.dumps({"impl": "reference", "unavailable": f"no CPU reference arm for workload {key}"}), flush=True)
        return
    wl = WORKLOADS[key]
    sample = min(wl["batch"], args.ref_sample)
    r = cpu_reference_rate(wl, sample, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC_SOLVE, "value": r["value"],
        "unit": "solves/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        # the GPU arm's workload keys, same names and values (bench_solve); the CPU arm's own facts go under other keys
        "config": {"workload": wl["desc"], "instances_per_gpu": wl["batch"] if wl["scaling"] == "weak" else -(-wl["batch"] // world),
                   "instances_total": wl["batch"] * world if wl["scaling"] == "weak" else wl["batch"],
                   "num_basis": wl["nb"], "horizon_steps": int(abs(wl["horizon"] / DT)), "replay_states": wl["mem"],
                   "instances_per_step": sample,
                   "note": "reference CPU path (single-threaded per instance), all host cores; each step is a bounded "
                           "sample of the workload's instances"},
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r["value"], "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------
class Ctx:
    """per-process state of the GPU arm: rank / device, torch.distributed, measured peaks, clock sampler"""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        import ergodic_exploration_b200 as eb

        self.torch, self.dist, self.eb, self.args = torch, dist, eb, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.clocks = ClockSampler(self.local_rank)
        if self.rank == 0:
            self.clocks.start()
        self._flush = None
        self._peak64 = None
        self.outputs = None  # --dump-outputs: the arrays bench_solve kept from its last timed step
        try:
            self.peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            self.peaks = {}
        self.hbm_peak = self.peaks.get("hbm_gbs", 6650.0)
        self.hbm_source = "MEASURED_PEAKS.json (hbm_gbs, of measured)" if self.peaks else "fallback 6650 GB/s (of fallback)"

    def flush_l2(self):
        """writes 256 MiB (> 126 MB L2): evicts the previous step's working set; enqueued OUTSIDE the event pairs"""
        if self._flush is None:
            self._flush = self.torch.empty(256 << 20, dtype=self.torch.uint8, device=self.dev)
        self._flush.zero_()

    def fp64_peak(self):
        if self._peak64 is None:
            self._peak64 = self.eb.fp64_peak(self.local_rank)
        return self._peak64

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        if self.world == 1:
            return list(vals)
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def traffic(self, key):
        try:
            return json.load(open(os.path.join(ROOT, "profiles", "solve_traffic.json")))[key]["bytes"]
        except Exception:
            return None

    def close(self):
        self.clocks.stop()
        if self.world > 1:
            self.dist.destroy_process_group()


def fp64_roofline(ctx, F, solves_per_launch, k_ms, key, N, M, note=None):
    dfma, dmma = ctx.fp64_peak()
    peak = max(dfma, dmma)
    achieved = F * solves_per_launch / (k_ms * 1e-3) / 1e12
    bps = bytes_per_solve(N, M)
    r = {"kernel": "solve_kernel", "bound": "fp64", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
         "frac": achieved / peak, "traffic": ctx.traffic(key), "flops_per_solve": F, "kernel_ms": k_ms,
         "solves_per_launch": solves_per_launch,
         "peak_source": f"measured live by eb_fp64_peak (DFMA {dfma:.2f}, DMMA {dmma:.2f} TFLOP/s; DFMA and DMMA share "
                        "one pipe on B200, tools/microbench/mix_probe.cu); MEASURED_PEAKS.json has no FP64 figure",
         "hbm": {"achieved": bps * solves_per_launch / (k_ms * 1e-3) / 1e9, "peak": ctx.hbm_peak, "unit": "GB/s",
                 "bytes_per_solve": bps, "peak_source": ctx.hbm_source}}
    if note:
        r["note"] = note
    return r


def bench_solve(ctx, key, steps, warmup, with_cpu=True, keep_outputs=False):
    """one batched control() per step over this rank's instances; returns the result dict (rank 0) or None.
    keep_outputs: rank 0 keeps in ctx.outputs what the last step of the run `value` reports returned"""
    torch, dist, eb = ctx.torch, ctx.dist, ctx.eb
    wl = WORKLOADS[key]
    world, rank = ctx.world, ctx.rank
    strong = wl["scaling"] == "strong" and world > 1
    B = wl["batch"] // world if strong else wl["batch"]
    R, umin, umax = model_params(wl["model"])
    N = int(abs(wl["horizon"] / DT))
    K = wl["nb"] ** 2
    M = min(wl["mem"], 100)
    working_set = 2 * 24 * N * B + 24 * max(M, 0) * B
    # A batch whose state (ut_ ping-pong + replay rows) fits into the 126 MB L2 would be served from L2 when the same
    # buffers are stepped again and again: such workloads ROTATE over enough independent batches (controllers) that
    # their combined state is 2.2 x L2 -- by the time a batch comes round again it has been evicted ("inputs larger
    # than L2"), and the K timed steps can run back to back inside ONE event pair.
    small_state = working_set < 2 * 126e6
    n_rot = max(2, int(np.ceil(2.2 * 126e6 / working_set))) if small_state else 1
    x, ut, mem = synth_inputs(wl, B, seed=0xE16C0D1C + 2 + rank)
    ctls = []
    for r_ in range(n_rot):
        c_ = eb.ErgodicControl(wl["model"], DT, wl["horizon"], 0.1, 1.0, wl["nb"], 1000000, 100, R, umin, umax,
                               batch=B, device=ctx.local_rank)
        c_.setTarget([eb.Gaussian(m, s) for m, s in zip(MU, SIGMA)])
        c_.set_ut(ut if r_ == 0 else synth_inputs(dict(wl, mem=0), B, seed=0xE16C0D1C + 1000 * (r_ + 1) + rank)[1])
        c_.keep_ck(False)  # control() returns u0 (+ metric); the K x B c_k dump is a debugging by-product
        if mem is not None:
            for m in mem:
                c_.addStateMemory(m)
        ctls.append(c_)
    ctl = ctls[0]

    xd = torch.from_numpy(x).to(ctx.dev)
    u0d = torch.empty((B, 3), dtype=torch.float64, device=ctx.dev)
    metd = torch.empty(B, dtype=torch.float64, device=ctx.dev)

    # N > 1: the gather of the first twists is fused with the solve (P2P stores into every rank's gathered
    # buffer over NVLink peer memory, csrc/peer_gather.cuh); a step ends when every rank's rows are here
    pg, gather_kind = None, "none (single GPU)"
    if world > 1:
        from ergodic_exploration_b200.sharding import PeerGather
        pg = PeerGather(ctl)
        # the branch eb_control_dev_gather_wait (the strict, timed call) takes for this batch
        gather_kind = ("fused into the solve kernel (every warp stores its row into all ranks' gathered buffers: P2P stores "
                       "over NVLink peer memory; arrival flags raised by the launch's last warp), then peer_wait_kernel on "
                       "the same stream") if pg.fused() else \
                      ("solve kernel writes u0 locally; peer_publish_wait_kernel right behind it on the SAME stream "
                       "(programmatic dependent launch) copies the block to all ranks over NVLink peer memory, raises "
                       "the arrival flags and waits for every rank's flags")

    def step_dev(i):
        c_ = ctls[i % n_rot]
        if pg is not None:
            pg.control_wait(BOUNDS, xd, metric=metd, ctl=c_)  # solve + gather + wait for every rank's rows
        else:
            c_.control(BOUNDS, xd, u0=u0d, metric=metd)

    def launch_total():
        return sum(c_.launch_count() for c_ in ctls)

    def last_step_outputs(u0):
        # read before any untimed call reuses u0d / metd or steps the controller again
        return {"u0": u0.cpu().numpy(), "metric": metd.cpu().numpy(), "ut": ctls[(steps - 1) % n_rot].get_ut()}

    W = max(3, warmup)
    for i in range(max(W, n_rot)):  # every batch has built its phi_k (first call) before the clock starts
        step_dev(i)
    for c_ in ctls:
        c_.check()
    if n_rot == 1:
        ctx.flush_l2()  # one batch larger than L2; with rotating batches the rotation itself has evicted batch 0's state
    ctx.barrier()
    launches0 = launch_total()
    ea, eb_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ctx.clocks.region(key):
        # the host enqueues ahead of the device (a step costs ~11 us of host time): no launch bubble inside the pair
        torch.cuda._sleep(int(min(steps, 400) * 15e-6 * 1.9e9))
        if pg is not None:
            step_dev(n_rot - 1)  # untimed: its wait for every rank's rows lines the ranks up ON THE DEVICE (host skew
            #                      after the barrier would otherwise be charged to the first timed steps: K is small)
        ea.record()
        for i in range(steps):
            step_dev(i)
        eb_.record()
        torch.cuda.synchronize()
    ctx.barrier()
    launches = launch_total() - launches0
    for c_ in ctls:
        c_.check()
    t_ms = ea.elapsed_time(eb_)
    if keep_outputs and pg is None and rank == 0:
        ctx.outputs = last_step_outputs(u0d)

    # N > 1, beside the strict number: the same K steps with the gather PIPELINED -- nothing in step i + 1 of a rank
    # depends on other ranks' rows (independent instances), so the solve of step i + 1 is launched while the rows of
    # step i are still travelling; every publication is launched and lands inside the event pair, whose end waits for
    # every rank's rows of the last step (a rank publishes in step order, so of every step)
    pipe_ms = 0.0
    if pg is not None:
        for i in range(W):
            pg.control(BOUNDS, xd, metric=metd, ctl=ctls[i % n_rot])
        pg.wait()
        ctx.barrier()
        pa, pb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ctx.clocks.region(key):
            torch.cuda._sleep(int(min(steps, 400) * 15e-6 * 1.9e9))
            step_dev(n_rot - 1)  # untimed, lines the ranks up on the device
            launches0 = launch_total()  # `value` is this run at N > 1: gpu_launches counts its launches
            pa.record()
            for i in range(steps):
                pg.control(BOUNDS, xd, metric=metd, ctl=ctls[i % n_rot])
            pg.wait()
            pb.record()
            torch.cuda.synchronize()
        ctx.barrier()
        launches = launch_total() - launches0
        for c_ in ctls:
            c_.check()
        pipe_ms = pa.elapsed_time(pb)
        if keep_outputs and rank == 0:
            ctx.outputs = last_step_outputs(pg.gathered())

    gather_ok = None
    if pg is not None:
        # the fused gather against a collective: every rank's copy must equal the all_gather of the row blocks
        mine = pg.gathered()[rank * B:(rank + 1) * B].clone()
        ref = torch.empty((world * B, 3), dtype=torch.float64, device=ctx.dev)
        dist.all_gather_into_tensor(ref, mine)
        gather_ok = bool(torch.equal(ref, pg.gathered()))
        if not gather_ok:
            raise SystemExit("bench.py: fused peer gather disagrees with NCCL all_gather")

    # the kernel alone (roofline): at N = 1 that is what the timed region holds (K launches back to back)
    k_ms = t_ms / steps
    if pg is not None:
        ctx.flush_l2()
        ka, kb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ka.record()
        for i in range(steps):
            ctls[i % n_rot].control(BOUNDS, xd, u0=u0d, metric=metd)
        kb.record()
        torch.cuda.synchronize()
        k_ms = ka.elapsed_time(kb) / steps
    # round-1 protocol beside it (N = 1): one event pair per step on ONE batch, L2 flushed between the pairs
    pairs_ms = None
    if pg is None and small_state:
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        torch.cuda._sleep(int(min(steps, 400) * 150e-6 * 1.9e9))  # the host enqueues ahead of the device
        for a, b in ev:
            ctx.flush_l2()
            a.record()
            ctl.control(BOUNDS, xd, u0=u0d, metric=metd)
            b.record()
        torch.cuda.synchronize()
        pairs_ms = sum(a.elapsed_time(b) for a, b in ev) / steps

    # end to end through the host-buffer entry points
    xh = torch.from_numpy(x).pin_memory()
    e2e_steps = max(3, min(steps, 200))
    if pg is None:
        u0h = torch.empty((B, 3), dtype=torch.float64).pin_memory()
        xh_np, u0h_np = xh.numpy(), u0h.numpy()

        def step_e2e():
            ctl.control(BOUNDS, xh_np, u0=u0h_np)  # H2D x (or zero-copy), kernel, D2H u0 + status, sync
        d2h = B * 24 + 4
        path = ("eb_control_host with pinned host buffers: the fused kernel reads x and writes u0 in place over "
                "PCIe (zero-copy, batch <= 16384), fault flag in mapped memory, stream sync") if B <= 16384 else \
            "eb_control_host: pinned host x -> H2D -> fused kernel -> D2H u0 + fault flag -> sync"
    else:
        gh = torch.empty((world * B, 3), dtype=torch.float64).pin_memory()

        def step_e2e():
            xd.copy_(xh, non_blocking=True)
            s = pg.control_wait(BOUNDS, xd, metric=metd)
            gh.copy_(pg.gathered(s), non_blocking=True)
            torch.cuda.current_stream().synchronize()
        d2h = world * B * 24
        path = ("pinned host x -> H2D -> solve kernel + fused gather (P2P stores over NVLink) -> wait for every rank's "
                "rows -> D2H of the GATHERED first twists (world x batch x 3) -> sync")
    for _ in range(3):
        step_e2e()
    ctx.barrier()
    with ctx.clocks.region(key):
        e0 = time.perf_counter()
        for _ in range(e2e_steps):
            step_e2e()
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - e0
    if pg is not None:
        pg.close()
    t_ms, e2e_s, k_ms, pipe_ms = ctx.max_over_ranks(t_ms, e2e_s, k_ms, pipe_ms)
    for c_ in ctls:
        c_.close()
    if rank != 0:
        return None

    total = world * B
    F = flops_per_solve(K, N, M)
    # N > 1: `value` is the run with the gather pipelined under the next step (every publication launched and landed
    # inside the event pair); the run with a barrier across the ranks inside every step is reported as `strict_barrier`
    strict_ms = t_ms
    if world > 1:
        t_ms = pipe_ms
    res = {
        "workload": key, "metric": METRIC_SOLVE, "value": total * steps / (t_ms * 1e-3), "unit": "solves/s",
        "n_gpus": world, "steps": steps, "warmup": W, "ms_per_step": t_ms / steps, "higher_is_better": True,
        "scaling": "strong" if strong else "weak", "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["desc"], "instances_per_gpu": B, "instances_total": total, "num_basis": wl["nb"],
                   "horizon_steps": N, "replay_states": M,
                   "l2": (f"inputs larger than L2: the steps rotate over {n_rot} independent batches of {B} instances "
                          f"({n_rot * working_set / 1e6:.0f} MB of controller state against a 126 MB L2), flushed once before the clock starts")
                   if small_state else
                   f"no flush: the per-step working set ({working_set / 1e6:.0f} MB of ut_ + replay rows) exceeds the 126 MB L2",
                   "timing": ("ONE CUDA-event pair around the K steps (one kernel launch per step, back to back) on the launching "
                              "stream, barrier + synchronize on both sides, max over ranks"
                              + ("; every step launches the solve AND the publication of its first twists to all ranks "
                                 "(eb_control_dev_gather); step i + 1 does not wait for the other ranks' rows of step i "
                                 "(independent instances), the pair ends with the wait for every rank's rows of the last "
                                 "step, i.e. all K gathers complete inside it.  strict_barrier = the same K steps with "
                                 "eb_control_dev_gather_wait: every step ends with the wait for all ranks' rows of THAT "
                                 "step (a barrier across the ranks per step)" if world > 1 else "")),
                   "ck_by_product": "off",
                   "parallelism": (f"instances sharded over {world} GPUs ({'strong' if strong else 'weak'} scaling), no data-path "
                                   f"collective; gather of u0 (timed run): {pg_mode(B)}; verified equal to an NCCL "
                                   f"all_gather: {gather_ok}")
                   if world > 1 else "single GPU"},
        "e2e": {"value": total * e2e_steps / e2e_s, "unit": "solves/s", "h2d_bytes_per_step": B * 24,
                "d2h_bytes_per_step": d2h, "ms_per_step": e2e_s / e2e_steps * 1e3, "steps": e2e_steps, "path": path},
        "gpu_launches": int(launches),
        "clocks": ctx.clocks.summary(key),
        "roofline": fp64_roofline(ctx, F, B, k_ms, key, N, M),
    }
    if world > 1:
        res["strict_barrier"] = {
            "value": total * steps / (strict_ms * 1e-3), "unit": "solves/s", "ms_per_step": strict_ms / steps,
            "note": "same K steps, one event pair, max over ranks, every step waits for all ranks' rows of that step before "
                    "the next solve is launched (" + gather_kind + "); the difference to `value` is the per-step NVLink "
                    "publish + flag round trip + rank skew that the pipelined gather hides under the next solve"}
    if pairs_ms is not None:
        res["ms_per_step_round1_protocol"] = pairs_ms
        res["config"]["round1_protocol"] = ("ms_per_step_round1_protocol = one event pair per step on ONE batch, 256 MiB L2 flush "
                                            "between the pairs (how BENCH_r01 was timed; each pair also holds ~5 us of "
                                            "launch + event overhead, measured with an empty kernel)")
    if world == 1 and with_cpu:
        sample = min(B, 4096 if key == "c2" else 1024)
        res["cpu_baseline"] = {k: v for k, v in cpu_reference_rate(wl, sample, 3, 1).items() if k != "ms_per_step"}
    return res


def bench_loop(ctx, loop_steps, warmup):
    """configs[4]: the full receding-horizon loop -- per tick addStateMemory(x) (exploration.hpp:209), control()
    (:232), and the plant x <- integrate_twist(x, u0, 0.1) with the angle wrap (numerics.hpp:273-298, the
    reference's own constant-twist integrator) -- 65536 Omni instances IN TOTAL (strong scaling), 16x16 basis,
    replay batch 100 drawn by the on-device sampler once more than 100 states are stored.  Everything stays on
    the device; ONE event pair brackets the whole loop.  N > 1: every rank loops over its own instances, the
    first twists of every tick are published to all ranks (fused gather) and each rank waits for the COMPLETE
    tick before it moves its robots -- the gather is on the critical path of every tick."""
    torch, eb = ctx.torch, ctx.eb
    world, rank = ctx.world, ctx.rank
    wl = WORKLOADS["c5"]
    B = int(os.environ.get("EB_C5_TOTAL", wl["batch"])) // world  # EB_C5_TOTAL: tuning runs at other sizes
    steps, warm = loop_steps, max(3, min(warmup, 10))
    R, umin, umax = model_params(wl["model"])
    N, K = int(abs(wl["horizon"] / DT)), wl["nb"] ** 2
    x, ut, _ = synth_inputs(dict(wl, mem=0), B, seed=0xE16C0D1C + 5 + rank)
    e2e_ticks = 50
    ctl = eb.ErgodicControl(wl["model"], DT, wl["horizon"], 0.1, 1.0, wl["nb"], steps + warm + e2e_ticks + 16, 100, R,
                            umin, umax, batch=B, device=ctx.local_rank)
    ctl.setTarget([eb.Gaussian(m, s) for m, s in zip(MU, SIGMA)])
    ctl.set_ut(ut)
    ctl.keep_ck(False)
    ctl.reserve_memory(steps + warm + e2e_ticks + 16)  # the replay buffer never re-allocates inside the loop
    xd = torch.from_numpy(x).to(ctx.dev)
    u0d = torch.empty((B, 3), dtype=torch.float64, device=ctx.dev)
    metd = torch.empty(B, dtype=torch.float64, device=ctx.dev)
    pg = None
    if world > 1:
        from ergodic_exploration_b200.sharding import PeerGather
        pg = PeerGather(ctl)

    def tick():
        ctl.addStateMemory(xd)  # exploration.hpp:209
        if pg is not None:
            step = pg.control_wait(BOUNDS, xd, metric=metd)
            mine = pg.gathered(step)[rank * B:(rank + 1) * B]
            eb.integrate_twist(xd, mine, DT, out=xd)
            return step
        ctl.control(BOUNDS, xd, u0=u0d, metric=metd)
        eb.integrate_twist(xd, u0d, DT, out=xd)
        return 0

    for _ in range(warm):
        tick()
    ctl.check()
    ctx.barrier()
    l0 = ctl.launch_count()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ctx.clocks.region("c5loop"):
        a.record()
        for _ in range(steps):
            tick()
        b.record()
        torch.cuda.synchronize()
    ctx.barrier()
    t_ms = a.elapsed_time(b)
    launches = ctl.launch_count() - l0 + steps  # + one integrate_twist kernel per tick
    ctl.check()
    metric_now = float(metd.mean())
    inside = bool(((xd[:, 0] > -1) & (xd[:, 0] < 11) & (xd[:, 1] > -1) & (xd[:, 1] < 11)).all())

    # end to end: the robots' poses live on the HOST.  Per tick: pinned x -> H2D, addStateMemory + control
    # (+ gather + wait) + plant on the device, u0 (the gathered block at N > 1) and the new poses -> D2H, sync.
    xh = xd.cpu().pin_memory()
    uh = torch.empty((world * B, 3), dtype=torch.float64).pin_memory()

    def tick_e2e():
        xd.copy_(xh, non_blocking=True)
        s = tick()
        uh.copy_(pg.gathered(s) if pg is not None else u0d, non_blocking=True)
        xh.copy_(xd, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for _ in range(2):
        tick_e2e()
    ctx.barrier()
    with ctx.clocks.region("c5loop"):
        e0 = time.perf_counter()
        for _ in range(e2e_ticks):
            tick_e2e()
        e2e_s = time.perf_counter() - e0
    ctl.check()
    if pg is not None:
        pg.close()
    t_ms, e2e_s = ctx.max_over_ranks(t_ms, e2e_s)
    ctl.close()
    if rank != 0:
        return None
    # replay states per solve: all stored (<= 100) early on, 100 sampled afterwards
    m_avg = sum(min(warm + i + 1, 100) for i in range(steps)) / steps
    F = flops_per_solve(K, N, m_avg)
    total = world * B
    roof = fp64_roofline(ctx, F, B, t_ms / steps, "c5", N, int(round(m_avg)),
                         note="per tick: addStateMemory copy + solve kernel (+ publish / wait at N > 1) + plant kernel -- "
                              "the whole loop, not the solve kernel alone")
    return {
        "workload": "c5loop", "metric": METRIC_SOLVE, "value": total * steps / (t_ms * 1e-3), "unit": "solves/s",
        "n_gpus": world, "steps": steps, "warmup": warm, "ms_per_step": t_ms / steps, "loop_ms": t_ms,
        "higher_is_better": True, "scaling": "strong" if world > 1 else "weak", "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"configs[4]: full receding-horizon loop, {steps} ticks, {total} Omni instances in total "
                               f"({B} per GPU), 16x16 basis, replay batch 100 (device sampler), plant = integrate_twist",
                   "instances_per_gpu": B, "instances_total": total,
                   "l2": "closed loop, no flush" + (": per-tick working set (2 x 157 MB of ut_) exceeds L2" if B >= 32768 else
                                                  f": per-tick working set {2 * 24 * N * B / 1e6:.0f} MB (ut_ ping-pong) + replay rows"),
                   "timing": "ONE CUDA-event pair around the whole loop (every tick's gather + wait inside), max over ranks",
                   "mean_ergodic_metric_at_end": metric_now, "robots_inside_map": inside,
                   "parallelism": (f"instances sharded over {world} GPUs (strong scaling: {total} in total); u0 of every tick "
                                   f"published to all ranks ({pg_mode(B)}), each rank waits for the complete tick before the plant step")
                   if world > 1 else "single GPU"},
        "gpu_launches": int(launches), "clocks": ctx.clocks.summary("c5loop"),
        "e2e": {"value": total * e2e_ticks / e2e_s, "unit": "solves/s", "h2d_bytes_per_step": B * 24,
                "d2h_bytes_per_step": world * B * 24 + B * 24, "ms_per_step": e2e_s / e2e_ticks * 1e3, "steps": e2e_ticks,
                "path": "per tick: pinned host poses -> H2D -> addStateMemory + control (+ fused gather + wait) + plant -> "
                        "D2H of the first twists (gathered block at N > 1) and of the new poses -> sync"},
        "roofline": roof,
    }


def pg_mode(batch):
    from ergodic_exploration_b200.sharding import gather_mode_for_batch
    return gather_mode_for_batch(batch)


def bench_phik(ctx, steps, warmup, with_cpu=True):
    """secondary metric: phi_k grid cells*bases/sec (configs[2]: 8192^2 grid, 32x32 basis).
    N > 1: the grid is row-sharded (strong scaling of the one contraction), every rank
    contracts its row block and one all_reduce of the raw 32x32 block finishes it."""
    torch, dist, eb = ctx.torch, ctx.dist, ctx.eb
    from ergodic_exploration_b200.sharding import finish_phik, shard_bounds

    world, rank = ctx.world, ctx.rank
    nx = ny = 8192
    nb, res = 32, 0.1
    lx = ly = (nx - 1) * res
    lo, hi = shard_bounds(ny, world, rank)
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from c3_density import c3_density_torch  # un-normalised mixture of 8 Gaussians (SURVEY section 8d C3), closed form

    phi = c3_density_torch(ctx.dev, nx, res, lo, hi)
    algo = int(os.environ.get("EB_PHIK_ALGO", "0"))
    plan = eb.PhikPlan(nx, hi - lo, res, lx, ly, nb, device=ctx.local_rank, algo=algo, row_begin=lo, ny_total=ny)
    fold, fold_dev = plan.fold()
    fold = fold and algo != 3
    raw = torch.empty((32, 32), dtype=torch.float64, device=ctx.dev)
    out = torch.empty(nb * nb, dtype=torch.float64, device=ctx.dev)
    # N > 1: the all-reduce of the ranks' 32 x 32 blocks is fused into the tile kernel (P2P over NVLink, PhikAllReduce);
    # NCCL (finish_phik) only when the peer mapping is unavailable
    par, reduce_kind = None, "none (single GPU)"
    if world > 1:
        try:
            from ergodic_exploration_b200.sharding import PhikAllReduce
            par = PhikAllReduce(plan)
            reduce_kind = "fused into the tile kernel: P2P stores of the raw 32x32 blocks over NVLink peer memory + arrival flags"
        except Exception as exc:
            reduce_kind = f"NCCL all_reduce of the raw 32x32 block (peer mapping failed: {exc})"

    def step():
        if par is not None:
            return par.execute(phi, out)
        if world > 1:
            plan.execute_raw(phi, raw)
            return finish_phik(raw, nb)[0]
        return plan.execute(phi, out)

    W = max(3, warmup)
    for _ in range(W):
        step()
    ctx.barrier()
    l0 = plan.launch_count()
    ea, eb_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ctx.clocks.region("c3"):
        torch.cuda._sleep(int(min(steps, 400) * 100e-6 * 1.9e9))  # host enqueues ahead of the device
        ea.record()
        for _ in range(steps):
            step()
        eb_.record()
        torch.cuda.synchronize()
    ctx.barrier()
    launches = plan.launch_count() - l0
    ms = ea.elapsed_time(eb_) / steps

    # parity at full size: the committed golden coefficients of this exact density (tests/golden/make_golden_c3.py)
    parity = None
    gpath = os.path.join(ROOT, "tests", "golden", "c3_phik_8192.npz")
    if os.path.exists(gpath):
        want = np.load(gpath)["phik"]
        got = step().cpu().numpy()
        parity = {"max_rel_err_vs_golden": float(np.max(np.abs(got - want)) / np.max(np.abs(want))), "tolerance": 1e-9,
                  "golden": "tests/golden/c3_phik_8192.npz (CPU oracle eo_phik_rows over the same closed-form density, "
                            "tests/golden/make_golden_c3.py)"}

    # end to end (N = 1): pinned host density in, phi_k out, through eb_phik_execute_host
    e2e = None
    if world == 1:
        phih = phi.cpu().pin_memory()
        phin = phih.numpy()
        plan.execute(phin)
        reps = max(2, min(steps, 5))
        with ctx.clocks.region("c3"):
            t0 = time.perf_counter()
            for _ in range(reps):
                plan.execute(phin)
            e2e_s = (time.perf_counter() - t0) / reps
        e2e = {"value": nx * ny * nb * nb / e2e_s, "unit": "cell*bases/s", "h2d_bytes_per_step": 8 * nx * ny,
               "d2h_bytes_per_step": 8 * nb * nb + 8, "ms_per_step": e2e_s * 1e3, "steps": reps,
               "path": "eb_phik_execute_host: pinned host density -> H2D (512 MiB, PCIe-bound) -> tile kernel -> D2H phi_k"}
        del phih
    else:
        # N > 1: every rank's row block starts in ITS pinned host buffer; H2D, tile kernel with the fused all-reduce,
        # D2H of the finished coefficients on every rank; wall clock between barriers, max over ranks
        phih = phi.cpu().pin_memory()
        outh = torch.empty(nb * nb, dtype=torch.float64).pin_memory()

        def step_host():
            phi.copy_(phih, non_blocking=True)
            outh.copy_(step(), non_blocking=True)
            torch.cuda.current_stream().synchronize()

        step_host()
        reps = max(2, min(steps, 5))
        ctx.barrier()
        with ctx.clocks.region("c3"):
            t0 = time.perf_counter()
            for _ in range(reps):
                step_host()
            e2e_s = (time.perf_counter() - t0) / reps
        ctx.barrier()
        (e2e_s,) = ctx.max_over_ranks(e2e_s)
        e2e = {"value": nx * ny * nb * nb / e2e_s, "unit": "cell*bases/s", "h2d_bytes_per_step": 8 * nx * (hi - lo),
               "d2h_bytes_per_step": 8 * nb * nb, "ms_per_step": e2e_s * 1e3, "steps": reps,
               "path": f"per rank: pinned host row block ({8 * nx * (hi - lo) >> 20} MiB) -> H2D -> tile kernel with the "
                       f"fused all-reduce -> D2H phi_k; bytes are per rank"}
        del phih
    (ms,) = ctx.max_over_ranks(ms)
    phis = phi[:384, :384].cpu().numpy() if (world == 1 and with_cpu) else None
    del phi
    if par is not None:
        par.close()
    plan.close()
    if rank != 0:
        return None
    dfma, dmma = ctx.fp64_peak()
    peak64 = max(dfma, dmma)
    flops = 2.0 * nx * ny * nb + 2.0 * ny * nb * nb  # SURVEY section 8(d) algorithmic count (unfolded)
    done_flops = flops / 2 if fold else flops        # the fold halves the DMMA work actually issued
    hbm = {"achieved": 8.0 * nx * ny / world / (ms * 1e-3) / 1e9, "peak": ctx.hbm_peak, "unit": "GB/s",
           "frac": 8.0 * nx * ny / world / (ms * 1e-3) / 1e9 / ctx.hbm_peak, "peak_source": ctx.hbm_source}
    f64 = {"achieved": done_flops / world / (ms * 1e-3) / 1e12, "peak": peak64, "unit": "TFLOP/s",
           "frac": done_flops / world / (ms * 1e-3) / 1e12 / peak64,
           "flops_issued_over_algorithmic": 0.5 if fold else 1.0,
           "peak_source": f"measured live by eb_fp64_peak (DFMA {dfma:.2f}, DMMA {dmma:.2f} TFLOP/s)"}
    main_ = hbm if fold else f64
    out_d = {
        "workload": "c3", "metric": "phi_k grid cells*bases/sec", "value": nx * ny * nb * nb / (ms * 1e-3),
        "unit": "cell*bases/s", "n_gpus": world, "steps": steps, "warmup": W, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong" if world > 1 else "weak", "dtype": "f64", "data": "synthetic",
        "config": {"workload": "configs[2]: phi_k over 8192x8192 Gaussian-mixture grid, 32x32 basis",
                   "l2": "input (512 MiB per step) larger than L2", "mirror_fold": bool(fold),
                   "timing": "one CUDA-event pair around the K steps (one kernel launch per step), max over ranks",
                   "table_asymmetry": fold_dev,
                   "parallelism": f"rows sharded over {world} GPUs (strong scaling); reduction: {reduce_kind}" if world > 1
                   else "single GPU"},
        "gpu_launches": int(launches), "clocks": ctx.clocks.summary("c3"),
        "roofline": {"kernel": "phik_tile_kernel", "bound": "hbm" if fold else "fp64", "achieved": main_["achieved"],
                     "peak": main_["peak"], "unit": main_["unit"], "frac": main_["frac"], "traffic": ctx.traffic("c3"),
                     "kernel_ms": ms, "hbm": hbm, "fp64": f64},
    }
    if parity:
        out_d["parity"] = parity
    if e2e:
        out_d["e2e"] = e2e
    if phis is not None:
        # CPU beside it: the reference's spatialCoeff arithmetic (2K cosines per cell; its K x G temporary would
        # be 550 TB at this size) as streamed by the C restatement, on a bounded sub-grid, one core
        from oracle import pyoracle
        from oracle.pyoracle import Oracle

        pyoracle.build()
        sub = 384
        t0 = time.perf_counter()
        Oracle.phik_from_grid(phis, res, (sub - 1) * res, (sub - 1) * res, nb)
        dt_cpu = time.perf_counter() - t0
        out_d["cpu_baseline"] = {"value": sub * sub * nb * nb / dt_cpu, "unit": "cell*bases/s", "cores": 1, "kind": "port",
                               "sample": f"{sub}x{sub} corner of the grid, 32x32 basis, Basis::spatialCoeff arithmetic "
                                         f"(basis.cpp:122-133) streamed by oracle/ergodic_oracle.c, single thread"}
    return out_d


def bench_avoid(ctx, mode, steps, warmup):
    """widened rows (SURVEY section 8f-2/3): the collision side of the tick that follows control().
    collide: validate_control of one twist per robot; dwa: DynamicWindow::control (3 x 8 x 5 window,
    2 s rollouts) per robot.  One shared 4000 x 4000 map (16 MB int8, L2-resident), explore_omni.yaml
    radii and limits, 2^18 robots per GPU; the robots are block-partitioned over the ranks with no exchange."""
    torch, eb = ctx.torch, ctx.eb
    world, rank = ctx.world, ctx.rank
    dwa_mode = mode == "dwa"
    rng = np.random.default_rng(0xE16C0D1C + 7 + rank)
    n, res, B = 4000, 0.05, 1 << 18
    mrng = np.random.default_rng(0xE16C0D1C + 8)  # the same map on every rank
    data = np.zeros((n, n), dtype=np.int8)
    data[mrng.random((n, n)) < 0.002] = 100
    data[mrng.random((n, n)) < 0.01] = -1
    colp = (0.7, 1.0, 0.2, 0.8)  # explore_omni.yaml:35-38
    grid = eb.GridMap(-100.0, 100.0, -100.0, 100.0, res, data, device=ctx.local_rank)
    col = eb.Collision(*colp)
    x0 = np.column_stack([rng.uniform(-98, 98, B), rng.uniform(-98, 98, B), rng.uniform(-np.pi, np.pi, B)])
    u = np.column_stack([rng.uniform(-1, 1, B), rng.uniform(-1, 1, B), rng.uniform(-2, 2, B)])
    xd, ud = torch.from_numpy(x0).to(ctx.dev), torch.from_numpy(u).to(ctx.dev)
    dwa_cfg = (0.1, 2.0, 0.2, 2.5, 2.5, 1.0, 1.0, -1.0, 1.0, -1.0, 2.0, -2.0)  # explore_omni.yaml:15-28,65-70
    dwa = eb.DynamicWindow(col, *dwa_cfg, 3, 8, 5)
    vref = torch.zeros_like(ud)

    def step():
        if dwa_mode:
            return dwa.control(grid, xd, ud, vref=vref)[0]
        return eb.validate_control(col, grid, xd, ud, 0.1, 0.5)

    xh = torch.from_numpy(x0).pin_memory().numpy()
    uh = torch.from_numpy(u).pin_memory().numpy()
    vh = torch.zeros((B, 3), dtype=torch.float64).pin_memory().numpy()
    fh = torch.zeros(B, dtype=torch.int32).pin_memory().numpy()
    oh = torch.zeros((B, 3), dtype=torch.float64).pin_memory().numpy()

    def step_host():
        if dwa_mode:
            return dwa.control(grid, xh, uh, vref=vh, out=(fh, oh))[0]
        return eb.validate_control(col, grid, xh, uh, 0.1, 0.5)

    W = max(3, warmup)
    for _ in range(W):
        out = step()
    torch.cuda.synchronize()
    free_frac = float(out.float().mean())
    ctx.barrier()
    l0 = grid.launch_count()
    steps = min(steps, 100)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    with ctx.clocks.region(mode):
        for a, b in ev:
            ctx.flush_l2()  # the map and the poses leave L2 between steps
            a.record()
            step()
            b.record()
        torch.cuda.synchronize()
    ctx.barrier()
    launches = grid.launch_count() - l0
    ms = sum(a.elapsed_time(b) for a, b in ev) / steps
    # the pre-dilated map is built once per map update; time one rebuild + step beside the steady state
    build_ms = None
    if dwa_mode:
        grid.update(data)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step()
        b.record()
        torch.cuda.synchronize()
        build_ms = a.elapsed_time(b) - ms
    # end to end: pinned host poses / twists in, flags (+ twists) out
    step_host()
    reps = 5
    with ctx.clocks.region(mode):
        t0 = time.perf_counter()
        for _ in range(reps):
            step_host()
        e2e_s = (time.perf_counter() - t0) / reps
    ms, e2e_s = ctx.max_over_ranks(ms, e2e_s)
    if rank != 0:
        return None

    # algorithmic probes of one full (collision-free) check: the reference's circle walk, pruned radii
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
    r_bnd, r_col, r_max = int(colp[0] / res), int((colp[0] + colp[2]) / res), int(colp[1] / res)
    probes_pose = sum(circle_cells(r) for r in range(r_bnd, min(r_max, r_col) + 1))
    probes_ref = sum(circle_cells(r) for r in range(r_bnd, r_max + 1))
    rollouts = 120 if dwa_mode else 1
    nsteps = 20 if dwa_mode else 5
    unit = "DWA decisions/s" if dwa_mode else "validated twists/s"
    # Roofline of the byte-gather kernels.  Every pose check is (dwa: dilated map) ONE 1-byte lookup or (collide)
    # a circle walk of 1-byte probes; a probe moves one 32-byte L2 sector.  The map (16 MB) is L2-resident, so the
    # bound is the L2 -> SM sector rate; the denominator is the MEASURED L2 random-sector bandwidth (eb_l2_gather_peak,
    # a kernel of the same access shape: 1-byte loads at random addresses of a 16 MB buffer).
    lookups_per_pose = 1 if dwa_mode else probes_pose
    sectors = B * rollouts * nsteps * lookups_per_pose
    l2_peak = None
    try:
        l2_peak = eb.l2_gather_peak(ctx.local_rank)  # G sectors/s
    except Exception:
        pass
    ach = sectors / (ms * 1e-3) / 1e9
    res_d = {
        "workload": mode,
        "metric": ("DynamicWindow::control decisions/sec (batched)" if dwa_mode else "validate_control twists/sec (batched)"),
        "value": world * B / (ms * 1e-3), "unit": unit, "n_gpus": world, "steps": steps, "warmup": W,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "dtype": "int8/f64", "data": "synthetic",
        "config": {"workload": ("DynamicWindow 3x8x5 window, 2 s rollouts" if dwa_mode else "validate_control, 0.5 s rollout")
                   + f", {B} robots per GPU on one 4000x4000 map @ 0.05 m, explore_omni.yaml radii",
                   "collision_free_fraction": free_frac, "l2": "flushed between timed steps",
                   "dilated_map": ("pose checks are single lookups into a pre-dilated map, rebuilt per map update: "
                                   f"{build_ms:.2f} ms for this map (outside the timed steps)") if dwa_mode else
                                  "not used at this pose count (circle walks)",
                   "parallelism": f"robots block-partitioned over {world} GPU(s), no exchange"},
        "e2e": {"value": world * B / e2e_s, "unit": unit, "h2d_bytes_per_step": (3 if dwa_mode else 2) * B * 24,
                "d2h_bytes_per_step": B * (4 + (24 if dwa_mode else 0)), "ms_per_step": e2e_s * 1e3, "steps": reps,
                "path": ("pinned host poses + twists + reference twists -> H2D -> kernel -> D2H flags + twists, in 32768-robot "
                         "slices alternating between two streams (copies of one slice overlap the kernel of the other)")
                if dwa_mode else "pinned host poses + twists -> H2D -> kernel -> D2H flags"},
        "gpu_launches": int(launches), "clocks": ctx.clocks.summary(mode),
        "roofline": {"kernel": "dwa_control_kernel" if dwa_mode else "validate_control_kernel",
                     "bound": "l2 (random 32-byte sectors of an L2-resident int8 map)",
                     "achieved": ach, "peak": l2_peak, "unit": "G sectors/s (upper bound on the probes: early exits probe less)",
                     "frac": (ach / l2_peak) if l2_peak else None, "traffic": None,
                     "probes_per_pose": lookups_per_pose, "probes_per_pose_reference_unpruned": probes_ref,
                     "peak_source": "measured live by eb_l2_gather_peak (random 1-byte loads over a 16 MB buffer)"},
    }
    if world == 1:
        from oracle import pyoracle
        from oracle.pyoracle import Oracle, RefLib

        pyoracle.build()
        lib = RefLib if RefLib.available() else Oracle
        sample = 2048 if dwa_mode else 200000
        sub = slice(0, sample)
        t0 = time.perf_counter()
        if dwa_mode:
            lib.dwa_control(data, res, -100.0, -100.0, colp, dwa_cfg, (3, 8, 5), x0[sub], u[sub], vref=np.zeros((sample, 3)))
        else:
            lib.validate_control(data, res, -100.0, -100.0, colp, x0[sub], u[sub], 0.1, 0.5)
        dt_cpu = time.perf_counter() - t0
        res_d["cpu_baseline"] = {"value": sample / dt_cpu, "unit": unit, "cores": 1,
                                 "kind": "reference" if lib is RefLib else "port",
                                 "sample": f"{sample} robots of the same workload, the reference's own "
                                           f"{'DynamicWindow::control' if dwa_mode else 'validate_control'} on one core "
                                           "(includes one GridMap construction)"}
    return res_d


def peer_stress(ctx, steps=48):
    """N > 1, untimed: the flag / fence protocol of the fused gather under skew.  Both publication branches (a
    single-wave batch on the side stream, a multi-wave batch from inside the solve kernel); every step ONE rank is
    held back by a ~1 ms spin kernel and NO collective runs between steps, so the fast ranks run ahead until the
    4-buffer reuse guard stops them.  Every step's gathered block is copied after its wait; at the end the copies
    must equal an NCCL all_gather of the ranks' own rows, bit for bit, on every rank."""
    torch, dist, eb = ctx.torch, ctx.dist, ctx.eb
    from ergodic_exploration_b200.sharding import PeerGather

    world, rank = ctx.world, ctx.rank
    results = {}
    for name, B in (("side_stream", 1024), ("in_kernel", 40000)):
        wl = WORKLOADS["c2"]
        R, umin, umax = model_params(wl["model"])
        x, ut, _ = synth_inputs(wl, B, seed=0xE16C0D1C + 40 + rank)
        ctl = eb.ErgodicControl(wl["model"], DT, wl["horizon"], 0.1, 1.0, wl["nb"], 1000, 100, R, umin, umax, batch=B,
                                device=ctx.local_rank)
        ctl.setTarget([eb.Gaussian(m, s) for m, s in zip(MU, SIGMA)])
        ctl.set_ut(ut)
        ctl.keep_ck(False)
        xd = torch.from_numpy(x).to(ctx.dev)
        pg = PeerGather(ctl)
        mine = torch.empty((steps, B, 3), dtype=torch.float64, device=ctx.dev)
        seen = torch.empty((steps, world * B, 3), dtype=torch.float64, device=ctx.dev)
        ctx.barrier()
        for s_ in range(steps):
            if s_ % world == rank:
                torch.cuda._sleep(2_000_000)  # ~1 ms: this rank falls behind
            st = pg.control(BOUNDS, xd)
            pg.wait(st)
            g = pg.gathered(st)
            seen[s_].copy_(g)
            mine[s_].copy_(g[rank * B:(rank + 1) * B])
        ctl.check()
        ctx.barrier()
        allm = torch.empty((world, steps, B, 3), dtype=torch.float64, device=ctx.dev)
        dist.all_gather_into_tensor(allm, mine)
        want = allm.permute(1, 0, 2, 3).reshape(steps, world * B, 3)
        ok = torch.tensor([1 if torch.equal(want, seen) else 0], dtype=torch.int32, device=ctx.dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        results[name] = {"batch_per_gpu": B, "steps": steps, "branch": pg.mode()[:40], "bit_identical_on_all_ranks": bool(ok.item())}
        pg.close()
        ctl.close()
        if not ok.item():
            raise SystemExit(f"bench.py: peer gather stress ({name}) disagrees with NCCL all_gather")
    return results


def primary_line(res):
    """the driver's contract: the primary workload's result at the top level of the JSON line"""
    line = {k: res[k] for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                                "scaling") if k in res}
    line["vs_baseline"] = None  # BASELINE.md holds no published number for this metric
    for k in ("dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline", "parity", "loop_ms", "strict_barrier"):
        if k in res:
            line[k] = res[k]
    return line


DUMP_BYTES = 60 * 10**6  # a dump stays under 64 MB, .npy headers included


def dump_outputs(path, arrays):
    """<path>/<name>.npy in float64.  Beyond DUMP_BYTES in all, every array keeps the same fraction of its rows, a
    seeded sorted sample: the same rows in every run of the same arguments, and the same rows of arrays of equal length
    (u0, metric and ut of one instance stay together)."""
    os.makedirs(path, exist_ok=True)
    arrays = {name: np.asarray(a, dtype=np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            a = a[np.sort(np.random.default_rng(0).choice(len(a), len(a) * DUMP_BYTES // total, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def run_ours(args):
    ctx = Ctx(args)
    order = ["c2", "c3", "c4", "c5", "c5loop", "entropy"] if args.workload == "all" else [args.workload]
    results = []
    for key in order:
        try:
            if key == "c3":
                # secondary line of the full run: at least 100 steps (10 ms) inside its one event pair, whatever K the
                # primary was given -- the pair's own cost would otherwise be several per cent of 20 x 0.1 ms
                r = bench_phik(ctx, max(args.steps, 100) if args.workload == "all" else args.steps, args.warmup)
            elif key == "c5loop":
                r = bench_loop(ctx, args.loop_steps, args.warmup)
            elif key in ("collide", "dwa"):
                r = bench_avoid(ctx, key, args.steps, args.warmup)
            elif key == "entropy":
                r = bench_entropy(ctx, max(args.steps, 100) if args.workload == "all" else args.steps, args.warmup)
            else:
                r = bench_solve(ctx, key, args.steps, args.warmup,
                                keep_outputs=args.dump_outputs is not None and key == order[0])
        except SystemExit:
            raise
        except Exception as exc:  # a secondary must not take the primary line down with it
            if key == order[0]:
                raise
            r = {"workload": key, "error": f"{type(exc).__name__}: {exc}"} if ctx.rank == 0 else None
        results.append(r)
        ctx.torch.cuda.empty_cache()
    stress = peer_stress(ctx) if (ctx.world > 1 and args.workload == "all") else None
    if ctx.rank == 0:
        if args.dump_outputs is not None:
            dump_outputs(args.dump_outputs, ctx.outputs)
        line = primary_line(results[0])
        if stress is not None:
            line["peer_stress"] = stress
        if len(results) > 1:
            line["secondary"] = [r for r in results[1:] if r is not None]
            line["clocks_all_timed_regions"] = ctx.clocks.summary(None)
        print(json.dumps(line), flush=True)
    ctx.close()


def bench_entropy(ctx, steps, warmup):
    """SURVEY section 8f-4: map-derived target.  int8 occupancy grid -> per-cell entropy (numerics.hpp:164-179)
    -> normalised density -> phi_k, all on the device (eb_target_from_map_dev); one step = one map update."""
    torch, eb = ctx.torch, ctx.eb
    world, rank = ctx.world, ctx.rank
    if not hasattr(eb, "MapTarget"):
        return {"workload": "entropy", "error": "not built"} if rank == 0 else None
    n, res, nb = 4096, 0.05, 16
    rng = np.random.default_rng(0xE16C0D1C + 9)
    data = rng.integers(-1, 101, size=(n, n)).astype(np.int8)
    dd = torch.from_numpy(data).to(ctx.dev)
    mt = eb.MapTarget(n, n, res, nb, device=ctx.local_rank)
    out = torch.empty(nb * nb, dtype=torch.float64, device=ctx.dev)
    W = max(3, warmup)
    for _ in range(W):
        mt.execute(dd, out)
    ctx.barrier()
    l0 = mt.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    with ctx.clocks.region("entropy"):
        for a, b in ev:
            ctx.flush_l2()
            a.record()
            mt.execute(dd, out)
            b.record()
        torch.cuda.synchronize()
    ctx.barrier()
    launches = mt.launch_count() - l0
    ms = sum(a.elapsed_time(b) for a, b in ev) / steps
    dh = torch.from_numpy(data).pin_memory().numpy()
    mt.execute(dh)
    reps = 5
    t0 = time.perf_counter()
    for _ in range(reps):
        mt.execute(dh)
    e2e_s = (time.perf_counter() - t0) / reps
    ms, e2e_s = ctx.max_over_ranks(ms, e2e_s)
    mt.close()
    if rank != 0:
        return None
    cells = n * n
    per_step = launches / max(1, steps)
    fused = per_step < 1.5
    if fused:
        # ONE kernel (TMA-staged bytes, table lookup in shared memory, folded DMMA tiles): 1 B per cell of HBM traffic,
        # bound by the FP64 pipe: 2 nx ny nb + 2 ny nb^2 algorithmic flops (the fold issues half of them)
        dfma, dmma = ctx.fp64_peak()
        peak64 = max(dfma, dmma)
        flops = 2.0 * cells * nb + 2.0 * n * nb * nb
        ach64 = 0.5 * flops / (ms * 1e-3) / 1e12
        roof = {"kernel": "phik_tma_kernel<fold, u8> (entropy table lookup fused into the tile kernel)", "bound": "fp64",
                "achieved": ach64, "peak": peak64, "unit": "TFLOP/s", "frac": ach64 / peak64, "traffic": None,
                "flops_issued_over_algorithmic": 0.5, "bytes_per_cell": 1,
                "hbm": {"achieved": cells / (ms * 1e-3) / 1e9, "peak": ctx.hbm_peak, "unit": "GB/s"},
                "peak_source": f"measured live by eb_fp64_peak (DFMA {dfma:.2f}, DMMA {dmma:.2f} TFLOP/s)"}
    else:
        # entropy kernel: 1 B read + 8 B written per cell; contraction: 8 B read per cell
        ach = cells * (1 + 8 + 8) / (ms * 1e-3) / 1e9
        roof = {"kernel": "entropy_density_kernel + phi_k tile kernel", "bound": "hbm", "achieved": ach, "peak": ctx.hbm_peak,
                "unit": "GB/s", "frac": ach / ctx.hbm_peak, "traffic": None, "bytes_per_cell": 17,
                "peak_source": ctx.hbm_source}
    res_d = {
        "workload": "entropy", "metric": "map-derived target: occupancy cells/sec (entropy -> density -> phi_k)",
        "value": world * cells / (ms * 1e-3), "unit": "cells/s", "n_gpus": world, "steps": steps, "warmup": W,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "dtype": "int8 -> f64", "data": "synthetic",
        "config": {"workload": f"{n}x{n} int8 occupancy grid (uniform random -1..100), {nb}x{nb} basis: entropy per cell "
                               "(numerics.hpp:164-179), then phi_k of the entropy density", "l2": "flushed between timed steps",
                   "parallelism": f"replicas only: every rank processes its own map ({world} GPU(s))"},
        "e2e": {"value": world * cells / e2e_s, "unit": "cells/s", "h2d_bytes_per_step": cells, "d2h_bytes_per_step": 8 * nb * nb,
                "ms_per_step": e2e_s * 1e3, "steps": reps, "path": "pinned host int8 map -> H2D -> entropy lookup + phi_k (one fused kernel) -> D2H phi_k"},
        "gpu_launches": int(launches), "clocks": ctx.clocks.summary("entropy"),
        "roofline": roof,
    }
    if world == 1:
        from oracle import pyoracle
        from oracle.pyoracle import Oracle

        pyoracle.build()
        sub = 512
        t0 = time.perf_counter()
        Oracle.entropy_grid(data[:sub, :sub])
        dt_cpu = time.perf_counter() - t0
        res_d["cpu_baseline"] = {"value": sub * sub / dt_cpu, "unit": "cells/s", "cores": 1, "kind": "port",
                                 "sample": f"{sub}x{sub} corner, entropy() per cell only (numerics.hpp:164-179), one core"}
    return res_d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-sample", type=int, default=4096, help="instances per step of the CPU reference arm")
    ap.add_argument("--loop-steps", type=int, default=1000, help="ticks of the configs[4] closed loop")
    ap.add_argument("--workload", default="all",
                    choices=["all"] + sorted(WORKLOADS) + ["c3", "c5loop", "collide", "dwa", "entropy"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the primary workload's outputs of its last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs is not None and (args.impl != "ours" or args.workload not in ["all"] + sorted(WORKLOADS)):
        ap.error("--dump-outputs needs the GPU arm with a control() workload as the primary: all, "
                 + ", ".join(sorted(WORKLOADS)))
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    run_ours(args)


if __name__ == "__main__":
    main()
