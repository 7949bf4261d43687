"""-m gpu: the safe control tick of B robots on B maps (ErgodicControl.control_safe / eb_control_safe_batch_*).  Every
output equals, bit for bit, the composition of the calls it replaces -- control(), validate_control on each robot's
map, optTraj() and DynamicWindow.control on the robots whose twist collides, then the selection -- run on a clone()
of the same controller; a small batch is also checked against the oracle."""
import copy
import ctypes as C

import numpy as np
import pytest

from helpers import MODEL_OMNI, MODEL_SIMPLE_CART, make_gpu, plant, warm_ut
from oracle.pyoracle import Oracle
from test_dwa_cpu import COL, DWA_CART, DWA_OMNI
from test_gpu_grid_batch import SAMPLES, mixed_maps, robots, set_maps

pytestmark = pytest.mark.gpu
VAL_DT, VAL_H = 0.1, 2.0


def _bits(a):
    a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
    return np.ascontiguousarray(a).view(np.int64 if a.dtype == np.float64 else np.int32)


def _assert_same(got, want, what):
    np.testing.assert_array_equal(_bits(got), _bits(want), what)


def _obstacles(maps, x0):
    """robot i % 3 == 0: inside a filled disc (nothing is free: branch 2); i % 3 == 1: in a ring 0.6-0.8 m away (a
    fast twist collides, a slow one does not); i % 3 == 2: the map as it is"""
    out = []
    for i, (data, res, xmin, ymin) in enumerate(maps):
        data = data.copy()
        ys, xs = data.shape
        cx = xmin + (np.arange(xs) + 0.5) * res
        cy = ymin + (np.arange(ys) + 0.5) * res
        d = np.hypot(cx[None, :] - x0[i, 0], cy[:, None] - x0[i, 1])
        if i % 3 == 0:
            data[d < 0.5] = 100
        elif i % 3 == 1:
            data[(d > 0.6) & (d < 0.8)] = 100
        out.append((data, res, xmin, ymin))
    return out


def _setup(model, nb, rng, maps, x0):
    import ergodic_exploration_b200 as eb

    ctl = make_gpu(model, len(maps), nb=nb)
    ctl.set_ut(warm_ut(rng, len(maps), ctl.steps, model))
    ctl.setMapTargets([m[0] for m in maps], [m[1] for m in maps], [(m[2], m[3]) for m in maps])
    gb = eb.GridMapBatch(len(maps))
    set_maps(gb, maps)
    for _ in range(3):
        ctl.addStateMemory(x0 + rng.normal(0.0, 0.05, x0.shape))
    return ctl, gb


def _own_bounds(maps):
    return np.array([(m[2], m[2] + m[0].shape[1] * m[1], m[3], m[3] + m[0].shape[0] * m[1]) for m in maps])


def composed(ctl, gb, dwa, x, vb, bounds=None, collision=None, val_dt=VAL_DT, val_h=VAL_H):
    """the chain the safe tick replaces, on torch's current stream: (u, branch, metric, u0, ok)"""
    import torch

    import ergodic_exploration_b200 as eb

    dev = torch.device("cuda")
    T = lambda a: a if torch.is_tensor(a) else torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    xd, vbd = T(x), T(vb)
    metric = torch.empty(ctl.batch, dtype=torch.float64, device=dev)
    u0 = ctl.control(T(bounds) if bounds is not None else None, xd, metric=metric)
    if collision is not None:  # the tick's Collision serves the validation and the window
        dwa = copy.copy(dwa)
        dwa.collision = collision
    ok = eb.validate_control(dwa.collision, gb, xd, u0, val_dt, val_h)
    xt = torch.empty((ctl.batch, ctl.steps, 3), dtype=torch.float64, device=dev)
    ctl.optTraj(out=xt)
    found, ud = dwa.control(gb, xd, vbd, xt_ref=xt, dt_ref=ctl.timeStep())
    okb, fb = ok.bool(), found.bool()
    u = torch.where(okb[:, None], u0, torch.where(fb[:, None], ud, torch.zeros_like(ud)))
    branch = torch.where(okb, 0, torch.where(fb, 1, 2)).to(torch.int32)
    return u, branch, metric, u0, ok


def safe(ctl, gb, dwa, x, vb, bounds=None, **kw):
    import torch

    dev = torch.device("cuda")
    T = lambda a: a if torch.is_tensor(a) else torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    metric = torch.empty(ctl.batch, dtype=torch.float64, device=dev)
    u, branch = ctl.control_safe(gb, dwa, T(x), T(vb), kw.pop("val_dt", VAL_DT), kw.pop("val_h", VAL_H),
                                 bounds=T(bounds) if bounds is not None else None, metric=metric, **kw)
    return u, branch, metric


def _check_tick(ctl, gb, dwa, x, vb, bounds=None, tag="", val_h=VAL_H, collision=None):
    ref = ctl.clone()
    got = safe(ctl, gb, dwa, x, vb, bounds, val_h=val_h, collision=collision)
    want = composed(ref, gb, dwa, x, vb, bounds, collision=collision, val_h=val_h)
    for name, g, w in zip(("u", "branch", "metric"), got, want[:3]):
        _assert_same(g, w, f"{tag} {name}")
    _assert_same(ctl.get_ut(), ref.get_ut(), f"{tag} ut_")
    return got[1].cpu().numpy()


@pytest.mark.parametrize("model,nb", [(MODEL_OMNI, 10), (MODEL_SIMPLE_CART, 10), (MODEL_OMNI, 40),
                                      (MODEL_SIMPLE_CART, 40)])
@pytest.mark.parametrize("with_bounds", [False, True])
def test_bit_identical_to_composed_calls(model, nb, with_bounds):
    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(7 + nb + 2 * model + int(with_bounds))
    maps = mixed_maps(rng, copies=2, geoms=[(160, 200, 0.05, -1.0, 2.0), (120, 90, 0.1, 0.0, 0.0),
                                           (200, 200, 0.05, -5.0, -5.0), (90, 130, 0.2, 3.3, -7.1)])
    x0, _ = robots(rng, maps)
    vb = np.zeros((len(maps), 3))
    vb[1::2] = np.column_stack([rng.uniform(-0.5, 0.5, len(maps) // 2), np.zeros(len(maps) // 2),
                                rng.uniform(-1, 1, len(maps) // 2)])
    maps = _obstacles(maps, x0)
    ctl, gb = _setup(model, nb, rng, maps, x0)
    seen = set()
    for cfg, samples in SAMPLES:
        cfg = DWA_CART if model == MODEL_SIMPLE_CART else cfg
        dwa = eb.DynamicWindow(eb.Collision(*COL), *cfg, *samples)
        branch = _check_tick(ctl, gb, dwa, x0, vb, _own_bounds(maps) if with_bounds else None, f"{samples}")
        assert (branch[0::3] == 2).all(), branch  # boxed in
        seen |= set(branch.tolist())
    assert seen == {0, 1, 2}, seen


def test_failing_robots_match_the_oracle():
    import torch

    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(12)
    maps = mixed_maps(rng, copies=1, geoms=[(160, 200, 0.05, -1.0, 2.0), (120, 90, 0.1, 0.0, 0.0),
                                           (200, 200, 0.05, -5.0, -5.0), (90, 130, 0.2, 3.3, -7.1)] * 3)
    x0, _ = robots(rng, maps)
    vb = np.zeros((len(maps), 3))
    maps = _obstacles(maps, x0)
    ctl, gb = _setup(MODEL_OMNI, 10, rng, maps, x0)
    dwa = eb.DynamicWindow(eb.Collision(*COL), *DWA_OMNI, 3, 8, 5)
    ref = ctl.clone()
    u, branch, _ = safe(ctl, gb, dwa, x0, vb)
    u, branch = u.cpu().numpy(), branch.cpu().numpy()
    u0 = ref.control(None, torch.from_numpy(x0).cuda()).cpu().numpy()
    xt = ref.optTraj()
    for i, (data, res, xmin, ymin) in enumerate(maps):
        ok = Oracle.validate_control(data, res, xmin, ymin, COL, x0[i:i + 1], u0[i:i + 1], VAL_DT, VAL_H)[0]
        if ok:
            assert branch[i] == 0, i
            np.testing.assert_array_equal(u[i], u0[i])
            continue
        fo, uo, _ = Oracle.dwa_control(data, res, xmin, ymin, COL, DWA_OMNI, (3, 8, 5), x0[i:i + 1], vb[i:i + 1],
                                       xt_ref=xt[i], dt_ref=ctl.timeStep())
        assert branch[i] == (1 if fo[0] else 2), i
        np.testing.assert_array_equal(u[i], uo[0] if fo[0] else np.zeros(3), f"robot {i}")
    assert {0, 1, 2} <= set(branch.tolist())


def _open_maps(rng, B):
    return [(np.zeros((100, 100), dtype=np.int8), 0.1, float(rng.uniform(-5, 5)), float(rng.uniform(-5, 5)))
            for _ in range(B)]


def _centred(maps):
    return np.array([(m[2] + 5.0, m[3] + 5.0, 0.3 * i) for i, m in enumerate(maps)])


def test_no_robot_fails_and_every_robot_fails():
    import torch

    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(21)
    B = 40
    maps = _open_maps(rng, B)
    x0 = _centred(maps)
    ctl, gb = _setup(MODEL_OMNI, 10, rng, maps, x0)
    dwa = eb.DynamicWindow(eb.Collision(*COL), *DWA_OMNI, 3, 8, 5)
    ref = ctl.clone()
    u, branch, _ = safe(ctl, gb, dwa, x0, np.zeros((B, 3)))
    want = composed(ref, gb, dwa, x0, np.zeros((B, 3)))
    assert (branch.cpu().numpy() == 0).all()
    _assert_same(u, want[3], "u == u0")
    # every robot fails: an obstacle disc covers the pose its twist reaches at the end of the validation horizon
    # (the solve of the tick gives the twist a clone computes now).  Where that pose is far from the start, the
    # window's slow candidates stay clear (branch 1); a robot whose twist barely moves it sits in the disc (branch 2).
    # The tick's Collision is given explicitly, with the values of the window's own.
    u0 = ctl.clone().control(None, torch.from_numpy(x0).cuda()).cpu().numpy()
    end = x0.copy()
    for _ in range(int(VAL_H / VAL_DT)):
        end = plant(end, u0, VAL_DT)
    boxed = [(m[0].copy(), m[1], m[2], m[3]) for m in maps]
    for (data, res, xmin, ymin), e in zip(boxed, end):
        cx, cy = xmin + (np.arange(100) + 0.5) * res, ymin + (np.arange(100) + 0.5) * res
        data[np.hypot(cx[None, :] - e[0], cy[:, None] - e[1]) < 0.3] = 100
    set_maps(gb, boxed)
    branch = _check_tick(ctl, gb, dwa, x0, np.zeros((B, 3)), tag="all fail", collision=eb.Collision(*COL))
    assert (branch != 0).all(), branch
    assert (branch == 1).any(), branch


def test_boxed_in_robots_get_the_zero_twist():
    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(22)
    B = 16
    maps = _open_maps(rng, B)
    x0 = _centred(maps)
    for data, *_ in maps:
        data[40:60, 40:60] = 100  # the robot sits in the middle of an obstacle
    ctl, gb = _setup(MODEL_OMNI, 10, rng, maps, x0)
    dwa = eb.DynamicWindow(eb.Collision(*COL), *DWA_OMNI, 7, 7, 7)
    branch = _check_tick(ctl, gb, dwa, x0, np.zeros((B, 3)), tag="boxed")
    assert (branch == 2).all()
    u, _, _ = safe(ctl.clone(), gb, dwa, x0, np.zeros((B, 3)))
    _assert_same(u, np.zeros((B, 3)), "zero twist")


@pytest.mark.parametrize("model", [MODEL_OMNI, MODEL_SIMPLE_CART])
def test_closed_loop_20_ticks(model):
    import torch

    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(30 + model)
    maps = mixed_maps(rng, copies=3, geoms=[(160, 200, 0.05, -1.0, 2.0), (120, 90, 0.1, 0.0, 0.0),
                                           (90, 130, 0.2, 3.3, -7.1)])
    B = len(maps)
    x0, _ = robots(rng, maps)
    maps = _obstacles(maps, x0)
    ctl, gb = _setup(model, 10, rng, maps, x0)
    ref = ctl.clone()
    dwa = eb.DynamicWindow(eb.Collision(*COL), *(DWA_CART if model == MODEL_SIMPLE_CART else DWA_OMNI), 3, 8, 5)
    xa = torch.from_numpy(x0).cuda()
    xb = xa.clone()
    va = torch.zeros((B, 3), dtype=torch.float64, device="cuda")
    vb = va.clone()
    seen = set()
    for tick in range(20):
        ctl.addStateMemory(xa)
        ref.addStateMemory(xb)
        u, branch, metric = safe(ctl, gb, dwa, xa, va)
        uw, bw, mw, _, _ = composed(ref, gb, dwa, xb, vb)
        for name, g, w in (("u", u, uw), ("branch", branch, bw), ("metric", metric, mw)):
            _assert_same(g, w, f"tick {tick} {name}")
        seen |= set(branch.cpu().numpy().tolist())
        xa = eb.integrate_twist(xa, u, 0.1)
        xb = eb.integrate_twist(xb, uw, 0.1)
        va, vb = u.clone(), uw.clone()
    _assert_same(ctl.get_ut(), ref.get_ut(), "ut_ after 20 ticks")
    assert len(seen) >= 2, seen


def test_host_path_equals_device_path():
    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(40)
    maps = mixed_maps(rng, copies=2, geoms=[(160, 200, 0.05, -1.0, 2.0), (120, 90, 0.1, 0.0, 0.0),
                                           (90, 130, 0.2, 3.3, -7.1)])
    B = len(maps)
    x0, vb = robots(rng, maps)
    vb[:, 1] *= 0.3
    maps = _obstacles(maps, x0)
    ctl, gb = _setup(MODEL_OMNI, 10, rng, maps, x0)
    dwa = eb.DynamicWindow(eb.Collision(*COL), *DWA_OMNI, 3, 8, 5)
    ref = ctl.clone()
    bounds = _own_bounds(maps)
    metric = np.empty(B)
    u, branch = ctl.control_safe(gb, dwa, x0, vb, VAL_DT, VAL_H, bounds=bounds, metric=metric)
    assert isinstance(u, np.ndarray) and u.shape == (B, 3) and branch.dtype == np.int32
    ud, bd, md = safe(ref, gb, dwa, x0, vb, bounds)
    for name, g, w in (("u", u, ud), ("branch", branch, bd), ("metric", metric, md)):
        _assert_same(g, w, name)
    _assert_same(ctl.get_ut(), ref.get_ut(), "ut_")


def test_side_stream_and_device_map_updates_need_no_sync():
    import torch

    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(50)
    geoms = [(120, 160, 0.05, -1.0, 2.0), (80, 90, 0.1, 0.0, 0.0), (60, 60, 0.1, 3.0, -2.0)] * 4
    maps = mixed_maps(rng, copies=1, geoms=geoms)
    B = len(maps)
    x0, _ = robots(rng, maps)
    maps = _obstacles(maps, x0)
    ctl, gb_ref = _setup(MODEL_OMNI, 10, rng, maps, x0)
    ref = ctl.clone()
    dwa = eb.DynamicWindow(eb.Collision(*COL), *DWA_OMNI, 3, 8, 5)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        gb = eb.GridMapBatch(B)
        gb.set([torch.from_numpy(m[0]).cuda() for m in maps], [m[1] for m in maps], [(m[2], m[3]) for m in maps])
        x = torch.from_numpy(x0).cuda()
        v = torch.zeros((B, 3), dtype=torch.float64, device="cuda")
        outs = []
        for tick in range(4):
            if tick in (1, 3):  # new cells for robots 0 and 4; at tick 3 robot 4's map grows: every map moves
                upd = np.zeros(B, dtype=bool)
                upd[[0, 4]] = True
                new = list(maps)
                new[0] = (np.where(rng.random(maps[0][0].shape) < 0.01, 100, maps[0][0]).astype(np.int8),) + maps[0][1:]
                if tick == 3:
                    d4 = np.zeros((200, 220), dtype=np.int8)
                    d4[:maps[4][0].shape[0], :maps[4][0].shape[1]] = maps[4][0]
                    new[4] = (d4,) + maps[4][1:]
                maps = new
                cells = [torch.from_numpy(m[0]).cuda() if f else None for m, f in zip(maps, upd)]
                gb.set(cells, [m[1] for m in maps], [(m[2], m[3]) for m in maps], upd)
            u, branch, metric = safe(ctl, gb, dwa, x, v)
            outs.append((maps, x.clone(), v.clone(), u.clone(), branch.clone(), metric.clone()))
            x = eb.integrate_twist(x, u, 0.1)
            v = u
    side.synchronize()
    for tick, (mp, xt, vt, u, branch, metric) in enumerate(outs):
        set_maps(gb_ref, mp)
        want = composed(ref, gb_ref, dwa, xt.cpu().numpy(), vt.cpu().numpy())
        torch.cuda.synchronize()
        for name, g, w in (("u", u, want[0]), ("branch", branch, want[1]), ("metric", metric, want[2])):
            _assert_same(g, w, f"tick {tick} {name}")


def test_launch_count():
    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(60)
    maps = mixed_maps(rng, copies=1, geoms=[(160, 200, 0.05, -1.0, 2.0), (120, 90, 0.1, 0.0, 0.0)] * 3)
    x0, vb = robots(rng, maps)
    maps = _obstacles(maps, x0)
    ctl, gb = _setup(MODEL_OMNI, 10, rng, maps, x0)
    dwa = eb.DynamicWindow(eb.Collision(*COL), *DWA_OMNI, 3, 8, 5)
    for bounds, launches in ((None, 3), (_own_bounds(maps), 4)):
        for path in ("dev", "host"):
            n, ng = ctl.launch_count(), gb.launch_count()
            if path == "dev":
                safe(ctl, gb, dwa, x0, vb, bounds)
            else:
                ctl.control_safe(gb, dwa, x0, vb, VAL_DT, VAL_H, bounds=bounds)
            assert ctl.launch_count() == n + launches, (path, bounds is None)
            assert gb.launch_count() == ng


def test_scale_4096_robots():
    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(4096)
    B = 4096
    maps = []
    for _ in range(B):
        ys, xs = int(rng.integers(40, 160)), int(rng.integers(40, 160))
        data = np.zeros((ys, xs), dtype=np.int8)
        data[rng.random((ys, xs)) < 0.01] = 100
        maps.append((data, float(rng.choice([0.05, 0.1])), float(rng.uniform(-20, 20)), float(rng.uniform(-20, 20))))
    x0, vb = robots(rng, maps)
    vb *= 0.3
    ctl, gb = _setup(MODEL_OMNI, 10, rng, maps, x0)
    dwa = eb.DynamicWindow(eb.Collision(*COL), *DWA_OMNI, 3, 8, 5)
    branch = _check_tick(ctl, gb, dwa, x0, vb, tag="4096")
    assert 0 < (branch != 0).sum() < B


def test_errors_leave_the_controller_unchanged():
    import torch

    import ergodic_exploration_b200 as eb
    from ergodic_exploration_b200 import capi
    from test_gpu_grid_batch import _raw_collision

    lib = capi.load()
    rng = np.random.default_rng(70)
    maps = mixed_maps(rng, copies=1, geoms=[(160, 200, 0.05, -1.0, 2.0), (120, 90, 0.1, 0.0, 0.0)] * 2)
    B = len(maps)
    x0, vb = robots(rng, maps)
    ctl, gb = _setup(MODEL_OMNI, 10, rng, maps, x0)
    dwa = eb.DynamicWindow(eb.Collision(*COL), *DWA_OMNI, 3, 8, 5)
    ut0, xt0, mem0 = ctl.get_ut(), ctl.optTraj(), ctl.memory_size()
    launches = [ctl.launch_count()]

    def unchanged():
        assert ctl.launch_count() == launches[0]  # nothing was launched
        _assert_same(ctl.get_ut(), ut0, "ut_")
        _assert_same(ctl.optTraj(), xt0, "pose (optTraj)")
        assert ctl.memory_size() == mem0
        launches[0] = ctl.launch_count()

    X, V = torch.from_numpy(x0).cuda(), torch.from_numpy(vb).cuda()
    U = torch.empty((B, 3), dtype=torch.float64, device="cuda")
    Bo = torch.empty(B, dtype=torch.int32, device="cuda")
    P = lambda t: C.c_void_p(t.data_ptr())
    col, cfg = C.byref(dwa.collision.cfg), C.byref(dwa.cfg)
    bad, oor = capi.EB_ERR_INVALID_ARGUMENT, capi.EB_ERR_OUT_OF_RANGE
    dev = lib.eb_control_safe_batch_dev
    host = lib.eb_control_safe_batch_host
    xh, vh, uh, bh = x0.copy(), vb.copy(), np.empty((B, 3)), np.empty(B, dtype=np.int32)
    cases = [
        (dev(None, gb._h, col, cfg, 0.1, 1.0, None, P(X), None, P(V), P(U), P(Bo), None), bad),
        (dev(ctl._h, None, col, cfg, 0.1, 1.0, None, P(X), None, P(V), P(U), P(Bo), None), bad),
        (dev(ctl._h, gb._h, None, cfg, 0.1, 1.0, None, P(X), None, P(V), P(U), P(Bo), None), bad),
        (dev(ctl._h, gb._h, col, None, 0.1, 1.0, None, P(X), None, P(V), P(U), P(Bo), None), bad),
        (dev(ctl._h, gb._h, col, cfg, 0.1, 1.0, None, None, None, P(V), P(U), P(Bo), None), bad),
        (dev(ctl._h, gb._h, col, cfg, 0.1, 1.0, None, P(X), None, None, P(U), P(Bo), None), bad),
        (dev(ctl._h, gb._h, col, cfg, 0.1, 1.0, None, P(X), None, P(V), None, P(Bo), None), bad),
        (dev(ctl._h, gb._h, col, cfg, 0.1, 1.0, None, P(X), None, P(V), P(U), None, None), bad),
        (dev(ctl._h, gb._h, col, cfg, 0.0, 1.0, None, P(X), None, P(V), P(U), P(Bo), None), bad),  # val_dt 0
        (host(ctl._h, gb._h, col, cfg, 0.0, 1.0, None, xh.ctypes.data, None, vh.ctypes.data, uh.ctypes.data,
              bh.ctypes.data, None), bad),
    ]
    for radii in ((0.5, 0.2, 0.0, 0.5), (0.1, 0.2, 0.0, 101.0)):  # Collision constructor rules
        cases.append((dev(ctl._h, gb._h, C.byref(_raw_collision(*radii).cfg), cfg, 0.1, 1.0, None, P(X), None, P(V),
                          P(U), P(Bo), None), bad))
    zero_dt = eb.DynamicWindow(eb.Collision(*COL), 0.0, *DWA_OMNI[1:], 3, 8, 5)
    cases.append((dev(ctl._h, gb._h, col, C.byref(zero_dt.cfg), 0.1, 1.0, None, P(X), None, P(V), P(U), P(Bo), None),
                  bad))
    long_dwa = eb.DynamicWindow(eb.Collision(*COL), 0.1, 6.0, *DWA_OMNI[2:], 3, 8, 5)  # 6 s rollout, 5 s optTraj
    cases.append((dev(ctl._h, gb._h, col, C.byref(long_dwa.cfg), 0.1, 1.0, None, P(X), None, P(V), P(U), P(Bo), None),
                  oor))
    cases.append((host(ctl._h, gb._h, col, C.byref(long_dwa.cfg), 0.1, 1.0, None, xh.ctypes.data, None,
                       vh.ctypes.data, uh.ctypes.data, bh.ctypes.data, None), oor))
    other_b = eb.GridMapBatch(B - 1)
    set_maps(other_b, maps[:-1])
    cases.append((dev(ctl._h, other_b._h, col, cfg, 0.1, 1.0, None, P(X), None, P(V), P(U), P(Bo), None), bad))
    unmapped = eb.GridMapBatch(B)
    unmapped.set([m[0] for m in maps], [m[1] for m in maps], [(m[2], m[3]) for m in maps],
                 np.arange(B) != 2)  # instance 2 never got a map
    cases.append((dev(ctl._h, unmapped._h, col, cfg, 0.1, 1.0, None, P(X), None, P(V), P(U), P(Bo), None), bad))
    shared = make_gpu(MODEL_OMNI, B)  # shared target: not a per-instance controller
    cases.append((dev(shared._h, gb._h, col, cfg, 0.1, 1.0, None, P(X), None, P(V), P(U), P(Bo), None), bad))
    for k, (st, want) in enumerate(cases):
        assert st == want, (k, st, lib.eb_last_error())
    unchanged()
    if torch.cuda.device_count() > 1:  # a grid batch on another device
        other_dev = eb.GridMapBatch(B, device=1)
        set_maps(other_dev, maps)
        assert dev(ctl._h, other_dev._h, col, cfg, 0.1, 1.0, None, P(X), None, P(V), P(U), P(Bo), None) == bad
        unchanged()
    with pytest.raises(ValueError, match="val_dt"):
        ctl.control_safe(gb, dwa, x0, vb, 0.0, 1.0)
    with pytest.raises(eb.ErgodicB200Error) as e:
        ctl.control_safe(gb, long_dwa, x0, vb, 0.1, 1.0)
    assert e.value.status == oor
    unchanged()
