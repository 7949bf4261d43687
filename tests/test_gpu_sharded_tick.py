"""-m gpu: per-instance control() and the safe tick on several GPUs (eb_control_batch_dev_gather[_wait],
eb_control_safe_batch_dev_gather[_wait], PeerGather.control_batch / control_safe).  On one GPU the peer group has a
single member (the kernels store into its own gathered buffer and raise its own flag) and every step's rows equal, bit
for bit, what a clone() of the controller returns from the single-GPU call; with two or more GPUs a torch.distributed
run checks the rows that arrive over NVLink against an NCCL all_gather of those single-GPU outputs."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import MODEL_OMNI, make_gpu, plant, warm_ut
from test_dwa_cpu import COL, DWA_OMNI
from test_gpu_grid_batch import mixed_maps, robots, set_maps
from test_gpu_safe_control import VAL_DT, VAL_H, _assert_same, _obstacles, _own_bounds, _setup

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GEOMS = [(160, 200, 0.05, -1.0, 2.0), (120, 90, 0.1, 0.0, 0.0), (200, 200, 0.05, -5.0, -5.0), (90, 130, 0.2, 3.3, -7.1)]


def _dev(a):
    import torch

    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _moved(bounds, i):
    """instance i's frame shifted by (0.5, -0.25): its extent and phi_k stay, its replay cosines are re-derived"""
    out = bounds.copy()
    out[i] += (0.5, 0.5, -0.25, -0.25)
    return out


@pytest.mark.parametrize("fuse_min_batch", ["0", "1000000"])  # publish from inside the kernel / from the side stream
def test_plain_per_instance_gather_matches_control(fuse_min_batch, monkeypatch):
    import torch

    from ergodic_exploration_b200.sharding import PeerGather

    monkeypatch.setenv("EB_GATHER_FUSE_MIN_BATCH", fuse_min_batch)
    rng = np.random.default_rng(81)
    maps = mixed_maps(rng, copies=5, geoms=GEOMS)
    B = len(maps)
    x, _ = robots(rng, maps)
    a = make_gpu(MODEL_OMNI, B)
    a.set_ut(warm_ut(rng, B, a.steps, MODEL_OMNI))
    a.setMapTargets([m[0] for m in maps], [m[1] for m in maps], [(m[2], m[3]) for m in maps])
    b = a.clone()
    pg = PeerGather(a)
    fused = pg.fused()
    assert fused == (fuse_min_batch == "0")
    bounds = _own_bounds(maps)
    for step in range(1, 14):  # 13 steps: the four buffers wrap three times
        bd = bounds if step == 1 else (_moved(bounds, 3) if step == 7 else None)
        xd = _dev(x)
        a.addStateMemory(xd)
        b.addStateMemory(xd)
        md = torch.empty(B, dtype=torch.float64, device="cuda")
        n = a.launch_count()
        if step % 2:
            assert pg.control_batch(_dev(bd), xd, metric=md) == step
            # as eb_control_dev_gather: the solve (+ side-stream publication), + the frame launch with bounds
            assert a.launch_count() == n + (1 if fused else 2) + (bd is not None)
            pg.wait(step)
        else:
            assert pg.control_batch_wait(_dev(bd), xd, metric=md) == step
            assert a.launch_count() == n + 2 + (bd is not None)  # solve + publish-and-wait / wait kernel
        assert pg.steps == step
        got = pg.gathered(step).clone()
        mb = torch.empty(B, dtype=torch.float64, device="cuda")
        want = b.control(_dev(bd), xd, metric=mb)
        _assert_same(got, want, f"step {step} u0")
        _assert_same(md, mb, f"step {step} metric")
        x = plant(x, want.cpu().numpy())
    _assert_same(a.get_ut(), b.get_ut(), "ut_")
    pg.close()


def _safe_setup(rng, copies=4):
    maps = mixed_maps(rng, copies=copies, geoms=GEOMS)
    x0, vb = robots(rng, maps)
    vb[1::2] = 0.0
    vb[:, 1] *= 0.3
    maps = _obstacles(maps, x0)
    ctl, gb = _setup(MODEL_OMNI, 10, rng, maps, x0)
    return maps, x0, vb, ctl, gb


@pytest.mark.parametrize("fuse_min_batch,side_stream", [("0", False), ("1000000", False), ("1000000", True)])
def test_safe_gather_matches_control_safe(fuse_min_batch, side_stream, monkeypatch):
    import torch

    import ergodic_exploration_b200 as eb
    from ergodic_exploration_b200.sharding import PeerGather

    monkeypatch.setenv("EB_GATHER_FUSE_MIN_BATCH", fuse_min_batch)
    rng = np.random.default_rng(91)
    maps, x0, vb, ctl, gb = _safe_setup(rng)
    B = len(maps)
    ref = ctl.clone()
    pg = PeerGather(ctl)
    dwa = eb.DynamicWindow(eb.Collision(*COL), *DWA_OMNI, 3, 8, 5)
    bounds = _own_bounds(maps)
    stream = torch.cuda.Stream() if side_stream else torch.cuda.current_stream()
    counts = np.zeros(3, dtype=np.int64)
    with torch.cuda.stream(stream):
        x, v = _dev(x0), _dev(vb)
        for step in range(1, 14):
            bd = _dev(bounds) if step in (1, 9) else None
            md = torch.empty(B, dtype=torch.float64, device="cuda")
            n = ctl.launch_count()
            if step % 4 == 3:  # a plain gather between safe ones, on the same group
                assert pg.control_batch(bd, x, metric=md) == step
                pg.wait(step)
                got = pg.gathered(step).clone()
                mw = torch.empty(B, dtype=torch.float64, device="cuda")
                want = ref.control(bd, x, metric=mw)
                _assert_same(got, want, f"step {step} u0")
                _assert_same(md, mw, f"step {step} metric")
                continue
            if step % 2:
                st, branch = pg.control_safe(gb, dwa, x, v, VAL_DT, VAL_H, bounds=bd, metric=md)
                assert ctl.launch_count() == n + 3 + (bd is not None)  # solve, validation, window (+ frames)
                pg.wait(st)
            else:
                st, branch = pg.control_safe_wait(gb, dwa, x, v, VAL_DT, VAL_H, bounds=bd, metric=md)
                assert ctl.launch_count() == n + 3 + (bd is not None)
            assert st == step == pg.steps
            got = pg.gathered(step).clone()
            mw = torch.empty(B, dtype=torch.float64, device="cuda")
            uw, bw = ref.control_safe(gb, dwa, x, v, VAL_DT, VAL_H, bounds=bd, metric=mw)
            _assert_same(got, uw, f"step {step} u")
            _assert_same(branch, bw, f"step {step} branch")
            _assert_same(md, mw, f"step {step} metric")
            counts += np.bincount(branch.cpu().numpy(), minlength=3)
            v = uw
    stream.synchronize()
    assert (counts > 0).all(), counts  # every branch: valid twists, window twists, boxed-in robots
    _assert_same(ctl.get_ut(), ref.get_ut(), "ut_")
    pg.close()


def test_refusals_leave_group_and_controller_unchanged():
    import torch

    import ergodic_exploration_b200 as eb
    from ergodic_exploration_b200 import capi
    from ergodic_exploration_b200.sharding import PeerGather

    lib = capi.load()
    rng = np.random.default_rng(95)
    maps, x0, vb, ctl, gb = _safe_setup(rng, copies=2)
    B = len(maps)
    ref = ctl.clone()
    pg = PeerGather(ctl)
    dwa = eb.DynamicWindow(eb.Collision(*COL), *DWA_OMNI, 3, 8, 5)
    X, V = _dev(x0), _dev(vb)
    Bo = torch.empty(B, dtype=torch.int32, device="cuda")
    P = lambda t: C.c_void_p(t.data_ptr())
    col, cfg = C.byref(dwa.collision.cfg), C.byref(dwa.cfg)
    bad = capi.EB_ERR_INVALID_ARGUMENT
    sg, sgw = lib.eb_control_safe_batch_dev_gather, lib.eb_control_safe_batch_dev_gather_wait
    pb, pbw = lib.eb_control_batch_dev_gather, lib.eb_control_batch_dev_gather_wait

    unconnected = C.c_void_p()
    assert lib.eb_peer_group_create(0, 0, 1, 3 * B, C.byref(unconnected)) == capi.EB_OK
    small = PeerGather(make_gpu(MODEL_OMNI, B - 1))  # a group sized for another batch
    other_b = eb.GridMapBatch(B - 1)
    set_maps(other_b, maps[:-1])
    shared = make_gpu(MODEL_OMNI, B)  # a shared target, and no frame configured for bounds NULL
    groups = {"pg": pg._h, "unconnected": unconnected, "small": small._h}

    def safe_cases(fn):
        a = dict(c=ctl._h, pg=pg._h, g=gb._h, col=col, cfg=cfg, x=P(X), vb=P(V), br=P(Bo))
        out = []
        for k in a:
            out.append(dict(a, **{k: None}))  # each NULL argument
        out.append(dict(a, c=shared._h))
        out.append(dict(a, pg=groups["unconnected"]))
        out.append(dict(a, pg=groups["small"]))
        out.append(dict(a, g=other_b._h))
        return [fn(d["c"], d["pg"], d["g"], d["col"], d["cfg"], VAL_DT, VAL_H, None, d["x"], None, d["vb"], d["br"],
                   None) for d in out]

    def plain_cases(fn):
        return [fn(None, pg._h, None, P(X), None, None), fn(ctl._h, None, None, P(X), None, None),
                fn(ctl._h, pg._h, None, None, None, None), fn(shared._h, pg._h, None, P(X), None, None),
                fn(ctl._h, unconnected, None, P(X), None, None), fn(ctl._h, small._h, None, P(X), None, None)]

    for step in range(2):  # before the first step and after one
        n = ctl.launch_count()
        for fn in (sg, sgw):
            assert safe_cases(fn) == [bad] * 12
        for fn in (pb, pbw):
            assert plain_cases(fn) == [bad] * 6
        if torch.cuda.device_count() > 1:  # a group on another device than the controller
            other_dev = C.c_void_p()
            assert lib.eb_peer_group_create(1, 0, 1, 3 * B, C.byref(other_dev)) == capi.EB_OK
            assert lib.eb_peer_group_connect(other_dev, None) == capi.EB_OK
            assert sg(ctl._h, other_dev, gb._h, col, cfg, VAL_DT, VAL_H, None, P(X), None, P(V), P(Bo), None) == bad
            assert pb(ctl._h, other_dev, None, P(X), None, None) == bad
            lib.eb_peer_group_destroy(other_dev)
        assert pg.steps == step and ctl.launch_count() == n
        # the next valid call: the same bits as a clone that never saw the refused calls
        st, branch = pg.control_safe_wait(gb, dwa, X, V, VAL_DT, VAL_H)
        assert st == step + 1
        uw, bw = ref.control_safe(gb, dwa, X, V, VAL_DT, VAL_H)
        _assert_same(pg.gathered(st), uw, "u after refusals")
        _assert_same(branch, bw, "branch after refusals")
    # the shared-target gathers keep refusing a per-instance controller
    assert lib.eb_control_dev_gather(ctl._h, pg._h, 0.0, 1.0, 0.0, 1.0, P(X), None, None) == capi.EB_ERR_UNSUPPORTED
    assert pg.steps == 2
    _assert_same(ctl.get_ut(), ref.get_ut(), "ut_")
    lib.eb_peer_group_destroy(unconnected)
    small.close()
    pg.close()


WORKER = r"""
import os, sys, time
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
import ergodic_exploration_b200 as eb
from helpers import MODEL_OMNI, make_gpu, warm_ut
from test_dwa_cpu import COL, DWA_OMNI
from test_gpu_grid_batch import mixed_maps, robots, set_maps
from test_gpu_safe_control import _obstacles
from ergodic_exploration_b200.sharding import PeerGather
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
rng = np.random.default_rng(200 + rank)
geoms = [(80, 100, 0.05, -1.0, 2.0), (60, 45, 0.1, 0.0, 0.0), (100, 100, 0.05, -5.0, -5.0), (45, 65, 0.2, 3.3, -7.1)]
maps = mixed_maps(rng, copies=128, geoms=geoms)   # 512 robots, each on its own map
B = len(maps)
x0, vb = robots(rng, maps)
vb[:, 1] *= 0.3
maps = _obstacles(maps, x0)                        # a third boxed in, a third in a ring: some twists fail
ctl = make_gpu(MODEL_OMNI, B, device=rank)
ctl.set_ut(warm_ut(rng, B, ctl.steps, MODEL_OMNI))
ctl.setMapTargets([m[0] for m in maps], [m[1] for m in maps], [(m[2], m[3]) for m in maps])
gb = eb.GridMapBatch(B, device=rank)
set_maps(gb, maps)
ref = ctl.clone()
pg = PeerGather(ctl)
dwa = eb.DynamicWindow(eb.Collision(*COL), *DWA_OMNI, 3, 8, 5)
x = torch.from_numpy(x0).cuda()
v = torch.from_numpy(vb).cuda()
got, want, fails = [], [], 0
for step in range(1, 14):
    if step % 3 == rank % 3:
        time.sleep(0.001)   # this rank launches late: the others' reuse guards wait for it
    kind = step % 4
    if kind == 1:
        st, br = pg.control_safe(gb, dwa, x, v, 0.1, 2.0)
        pg.wait(st)
    elif kind == 2:
        st, br = pg.control_safe_wait(gb, dwa, x, v, 0.1, 2.0)
    elif kind == 3:
        st = pg.control_batch(None, x)
        pg.wait(st)
    else:
        st = pg.control_batch_wait(None, x)
    assert st == step
    got.append(pg.gathered(step).clone())   # read before the next step is launched
    if kind in (1, 2):
        u, bw = ref.control_safe(gb, dwa, x, v, 0.1, 2.0)
        assert torch.equal(br, bw), f"rank {rank} step {step}: branch"
        fails += int((bw != 0).sum())
        v = u
    else:
        u = ref.control(None, x)
    want.append(u.clone())
torch.cuda.synchronize()
assert fails > 0
for step, (g, u) in enumerate(zip(got, want), 1):
    full = torch.empty((world * B, 3), dtype=torch.float64, device="cuda")
    dist.all_gather_into_tensor(full, u)
    assert torch.equal(full, g), f"rank {rank} step {step}: gathered rows differ from all_gather"
pg.close()
dist.destroy_process_group()
print("TICK_OK", rank)
"""


@pytest.mark.parametrize("world,port", [(2, 29541), ("all", 29543)])
@pytest.mark.parametrize("fuse_min_batch", ["0", "1000000"])
def test_ranks_over_nvlink(tmp_path, world, port, fuse_min_batch):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    if world == "all":
        world = min(torch.cuda.device_count(), 8)
        if world <= 2:
            pytest.skip("needs more than two GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                        "--master-addr", "127.0.0.1", "--master-port", str(port + (fuse_min_batch == "0") * 4),
                        str(script), ROOT], capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, EB_GATHER_FUSE_MIN_BATCH=fuse_min_batch))
    assert r.returncode == 0 and r.stdout.count("TICK_OK") == world, r.stdout[-2000:] + r.stderr[-3000:]
