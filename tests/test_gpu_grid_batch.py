"""-m gpu: per-instance occupancy maps (GridMapBatch / eb_grid_batch_*).  Instance i's collision checks,
validate_control and DynamicWindow run against map i: against the CPU restatement with each instance's own map, and
bit for bit against the shared-grid calls (GridMap with dilation(1)) on that map."""
import numpy as np
import pytest

from helpers import assert_abs_rel_close
from oracle.pyoracle import Oracle
from test_collision_cpu import CASES, random_map
from test_dwa_cpu import COL, DWA_CART, DWA_OMNI

pytestmark = pytest.mark.gpu

# (ysize, xsize, res, xmin, ymin): the maps of test_collision_cpu.CASES, a 1 x 1 map and two thin ones
GEOMS = [c[:5] for c in CASES] + [(1, 1, 0.1, 0.3, -0.2), (3, 250, 0.07, -2.0, 1.0), (210, 7, 0.05, 1.0, 1.0)]
SAMPLES = [(DWA_OMNI, (3, 8, 5)), (DWA_CART, (5, 1, 9)), (DWA_OMNI, (0, 2, 1)), (DWA_OMNI, (7, 7, 7))]


def mixed_maps(rng, copies=3, geoms=GEOMS):
    maps = []
    for _ in range(copies):
        for ys, xs, res, xmin, ymin in geoms:
            maps.append((random_map(rng, ys, xs, p_occ=0.004), res, xmin, ymin))
    return maps


def set_maps(gb, maps, update=None):
    gb.set([m[0] for m in maps], [m[1] for m in maps], [(m[2], m[3]) for m in maps], update)


def poses_for(rng, maps, per, margin=0.7):
    out = np.empty((len(maps), per, 3))
    for i, (data, res, xmin, ymin) in enumerate(maps):
        ys, xs = data.shape
        out[i, :, 0] = rng.uniform(xmin - margin, xmin + xs * res + margin, per)
        out[i, :, 1] = rng.uniform(ymin - margin, ymin + ys * res + margin, per)
        out[i, :, 2] = rng.uniform(-3.1, 3.1, per)
        out[i, 0, :2] = (xmin + xs * res, ymin + ys * res)  # exactly on the upper edge (grid.cpp:148-156)
        if per > 1:
            out[i, 1, :2] = (xmin, ymin)
    return out


def twists(rng, shape):
    u = np.stack([rng.uniform(-1, 1, shape), rng.uniform(-1, 1, shape), rng.uniform(-2, 2, shape)], axis=-1)
    u.reshape(-1, 3)[::5, 2] = 0.0  # the no-rotation branch of integrate_twist
    return u


def reference_trajectory(rng, maps, n=50):
    t = np.arange(n) * 0.1
    xt = np.empty((len(maps), n, 3))
    for i, (data, res, xmin, ymin) in enumerate(maps):
        ys, xs = data.shape
        cx, cy = xmin + xs * res / 2, ymin + ys * res / 2
        xt[i] = np.column_stack([cx + 0.3 * xs * res * np.cos(0.7 * t), cy + 0.3 * ys * res * np.sin(0.9 * t),
                                 4.0 * np.sin(0.5 * t)])
    return xt


def robots(rng, maps):
    x0 = np.empty((len(maps), 3))
    for i, (data, res, xmin, ymin) in enumerate(maps):
        ys, xs = data.shape
        x0[i] = (xmin + rng.uniform(0.2, 0.8) * xs * res, ymin + rng.uniform(0.2, 0.8) * ys * res, rng.uniform(-3, 3))
    vb = np.column_stack([rng.uniform(-1, 1, len(maps)), rng.uniform(-1, 1, len(maps)), rng.uniform(-2, 2, len(maps))])
    return x0, vb


@pytest.mark.parametrize("case", CASES)
def test_collision_and_validate_match_oracle_mixed_maps(case):
    import ergodic_exploration_b200 as eb

    col = case[5]
    rng = np.random.default_rng(int(col[0] * 1000) + 7)
    maps = mixed_maps(rng)
    gb, c = eb.GridMapBatch(len(maps)), eb.Collision(*col)
    set_maps(gb, maps)
    for per in (1, 37):
        poses = poses_for(rng, maps, per)
        got = c.collisionCheck(gb, poses[:, 0] if per == 1 else poses)
        assert got.shape == ((len(maps),) if per == 1 else (len(maps), per)) and got.dtype == np.int32
        got = got.reshape(len(maps), per)
        for i, (data, res, xmin, ymin) in enumerate(maps):
            np.testing.assert_array_equal(got[i], Oracle.collision_check(data, res, xmin, ymin, col, poses[i]), f"map {i}")
    per = 20
    x0 = poses_for(rng, maps, per, margin=0.0)
    u = twists(rng, (len(maps), per))
    for dt, horizon in ((0.1, 0.5), (0.1, 2.0), (0.05, 0.33)):
        got = eb.validate_control(c, gb, x0, u, dt, horizon)
        for i, (data, res, xmin, ymin) in enumerate(maps):
            np.testing.assert_array_equal(got[i], Oracle.validate_control(data, res, xmin, ymin, col, x0[i], u[i], dt,
                                                                          horizon), f"map {i}")


@pytest.mark.parametrize("cfg,samples", SAMPLES)
def test_dwa_twist_matches_oracle_mixed_maps(cfg, samples):
    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(11 + sum(samples))
    maps = mixed_maps(rng, copies=4)
    gb = eb.GridMapBatch(len(maps))
    set_maps(gb, maps)
    x0, vb = robots(rng, maps)
    vref = twists(rng, (len(maps),))
    dwa = eb.DynamicWindow(eb.Collision(*COL), *cfg, *samples)
    cost = np.empty(len(maps))
    found, u = dwa.control(gb, x0, vb, vref=vref, min_cost=cost)
    for i, (data, res, xmin, ymin) in enumerate(maps):
        fo, uo, co = Oracle.dwa_control(data, res, xmin, ymin, COL, cfg, samples, x0[i:i + 1], vb[i:i + 1],
                                        vref=vref[i:i + 1])
        assert found[i] == fo[0], f"map {i}"
        np.testing.assert_array_equal(u[i], uo[0], f"map {i}")
        if fo[0]:
            assert_abs_rel_close(cost[i:i + 1], co, f"map {i} min cost")
    assert 0 < found.sum()


@pytest.mark.parametrize("per_instance", [False, True])
def test_dwa_trajectory_matches_oracle_mixed_maps(per_instance):
    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(29)
    maps = mixed_maps(rng, copies=4)
    gb = eb.GridMapBatch(len(maps))
    set_maps(gb, maps)
    x0, vb = robots(rng, maps)
    xt = reference_trajectory(rng, maps)
    if not per_instance:
        xt = xt[0]
    dwa = eb.DynamicWindow(eb.Collision(*COL), *DWA_OMNI, 3, 8, 5)
    cost = np.empty(len(maps))
    found, u = dwa.control(gb, x0, vb, xt_ref=xt, dt_ref=0.1, min_cost=cost)
    for i, (data, res, xmin, ymin) in enumerate(maps):
        fo, uo, co = Oracle.dwa_control(data, res, xmin, ymin, COL, DWA_OMNI, (3, 8, 5), x0[i:i + 1], vb[i:i + 1],
                                        xt_ref=xt[i] if per_instance else xt, dt_ref=0.1)
        assert found[i] == fo[0], f"map {i}"
        np.testing.assert_array_equal(u[i], uo[0], f"map {i}")
        if fo[0]:
            assert_abs_rel_close(cost[i:i + 1], co, f"map {i} min cost")


def _all_outputs(gb, maps, seed):
    """every check of one instance set: collision (per 5), validate (per 4), DWA twist and traj with costs"""
    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(seed)
    c = eb.Collision(*COL)
    poses = poses_for(rng, maps, 5)
    x0v = poses_for(rng, maps, 4, margin=0.0)
    u = twists(rng, (len(maps), 4))
    x0, vb = robots(rng, maps)
    vref = twists(rng, (len(maps),))
    xt = reference_trajectory(rng, maps)
    dwa = eb.DynamicWindow(c, *DWA_OMNI, 3, 8, 5)
    ct, cj = np.empty(len(maps)), np.empty(len(maps))
    ft, ut = dwa.control(gb, x0, vb, vref=vref, min_cost=ct)
    fj, uj = dwa.control(gb, x0, vb, xt_ref=xt, dt_ref=0.1, min_cost=cj)
    inputs = dict(poses=poses, x0v=x0v, u=u, x0=x0, vb=vb, vref=vref, xt=xt)
    return inputs, dict(hit=c.collisionCheck(gb, poses), valid=eb.validate_control(c, gb, x0v, u, 0.1, 2.0), ft=ft,
                        ut=ut, ct=ct, fj=fj, uj=uj, cj=cj)


def _shared_outputs(m, inp, i):
    """the same checks of instance i through a GridMap of its own map with dilation(1)"""
    import ergodic_exploration_b200 as eb

    data, res, xmin, ymin = m
    ys, xs = data.shape
    g = eb.GridMap(xmin, xmin + xs * res, ymin, ymin + ys * res, res, data)
    g.dilation(1)
    c = eb.Collision(*COL)
    dwa = eb.DynamicWindow(c, *DWA_OMNI, 3, 8, 5)
    ct, cj = np.empty(1), np.empty(1)
    ft, ut = dwa.control(g, inp["x0"][i:i + 1], inp["vb"][i:i + 1], vref=inp["vref"][i:i + 1], min_cost=ct)
    fj, uj = dwa.control(g, inp["x0"][i:i + 1], inp["vb"][i:i + 1], xt_ref=inp["xt"][i], dt_ref=0.1, min_cost=cj)
    return dict(hit=c.collisionCheck(g, inp["poses"][i]), valid=eb.validate_control(c, g, inp["x0v"][i], inp["u"][i],
                                                                                    0.1, 2.0),
                ft=ft[0], ut=ut[0], ct=ct[0], fj=fj[0], uj=uj[0], cj=cj[0])


def test_bit_identical_to_shared_grid_and_permutation_invariant():
    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(64)
    geoms = [(int(rng.integers(1, 120)), int(rng.integers(1, 120)), float(rng.choice([0.05, 0.07, 0.1, 0.2])),
              float(rng.uniform(-5, 5)), float(rng.uniform(-5, 5))) for _ in range(64)]
    maps = mixed_maps(rng, copies=1, geoms=geoms)
    gb = eb.GridMapBatch(64)
    set_maps(gb, maps)
    inp, out = _all_outputs(gb, maps, 1)
    for i in range(64):
        want = _shared_outputs(maps[i], inp, i)
        for k, v in want.items():
            np.testing.assert_array_equal(out[k][i], v, f"{k} of instance {i}")
    # maps and inputs permuted together: the outputs permute, nothing else changes
    perm = rng.permutation(64)
    gp = eb.GridMapBatch(64)
    set_maps(gp, [maps[p] for p in perm])
    inp_p = {k: v[perm] for k, v in inp.items()}
    c = eb.Collision(*COL)
    np.testing.assert_array_equal(c.collisionCheck(gp, inp_p["poses"]), out["hit"][perm])
    np.testing.assert_array_equal(eb.validate_control(c, gp, inp_p["x0v"], inp_p["u"], 0.1, 2.0), out["valid"][perm])
    dwa = eb.DynamicWindow(c, *DWA_OMNI, 3, 8, 5)
    cost = np.empty(64)
    f, u = dwa.control(gp, inp_p["x0"], inp_p["vb"], xt_ref=inp_p["xt"], dt_ref=0.1, min_cost=cost)
    np.testing.assert_array_equal(f, out["fj"][perm])
    np.testing.assert_array_equal(u, out["uj"][perm])
    np.testing.assert_array_equal(cost, out["cj"][perm])
    # B = 1 is the shared call
    g1 = eb.GridMapBatch(1)
    set_maps(g1, maps[5:6])
    inp1, o1 = _all_outputs(g1, maps[5:6], 2)
    w1 = _shared_outputs(maps[5], inp1, 0)
    for k, v in w1.items():
        np.testing.assert_array_equal(o1[k][0], v, k)


def test_update_mask_and_relayout():
    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(3)
    maps = mixed_maps(rng, copies=1, geoms=[(60, 80, 0.05, 0.0, 0.0), (90, 90, 0.1, -3.0, 2.0), (40, 70, 0.07, 1.0, 1.0),
                                            (50, 50, 0.05, 2.0, -1.0), (1, 1, 0.1, 0.0, 0.0), (30, 120, 0.2, -9.0, 4.0)])
    gb = eb.GridMapBatch(len(maps))
    set_maps(gb, maps)
    inp, before = _all_outputs(gb, maps, 5)
    new = list(maps)
    new[0] = (random_map(rng, 150, 170, p_occ=0.004), 0.05, -1.0, 0.5)  # outgrows its slot: every map moves
    new[1] = (random_map(rng, 20, 30, p_occ=0.004), 0.1, -3.0, 2.0)     # shrinks
    new[2] = (random_map(rng, 40, 70, p_occ=0.05), 0.07, 1.0, 1.0)      # new cells only
    upd = np.array([True, True, True, False, False, False])
    cells = [m[0] if f else None for m, f in zip(new, upd)]
    gb.set(cells, [m[1] for m in new], [(m[2], m[3]) for m in new], upd)
    inp2, after = _all_outputs(gb, new, 5)
    for i in range(len(maps)):
        if upd[i]:
            want = _shared_outputs(new[i], inp2, i)
            data, res, xmin, ymin = new[i]
            np.testing.assert_array_equal(after["hit"][i], Oracle.collision_check(data, res, xmin, ymin, COL,
                                                                                  inp2["poses"][i]))
        else:
            want = {k: v[i] for k, v in before.items()}
            assert all(np.array_equal(inp[k][i], inp2[k][i]) for k in ("poses", "x0v", "u", "x0", "vb", "vref"))
        for k, v in want.items():
            np.testing.assert_array_equal(after[k][i], v, f"{k} of instance {i}")


def test_launch_counts():
    import torch

    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(4)
    maps = mixed_maps(rng, copies=1)
    gb = eb.GridMapBatch(len(maps))
    n0 = gb.launch_count()
    set_maps(gb, maps)
    assert gb.launch_count() == n0 + 1
    upd = np.zeros(len(maps), dtype=bool)
    upd[2] = True
    gb.set([m[0] for m in maps], [m[1] for m in maps], [(m[2], m[3]) for m in maps], upd)
    assert gb.launch_count() == n0 + 2
    c = eb.Collision(*COL)
    dwa = eb.DynamicWindow(c, *DWA_OMNI, 3, 8, 5)
    x0, vb = robots(rng, maps)
    calls = [lambda: c.collisionCheck(gb, x0), lambda: eb.validate_control(c, gb, x0, vb, 0.1, 1.0),
             lambda: dwa.control(gb, x0, vb, vref=vb), lambda: dwa.control(gb, x0, vb, xt_ref=reference_trajectory(
                 rng, maps), dt_ref=0.1)]
    xd, vd = torch.from_numpy(x0).cuda(), torch.from_numpy(vb).cuda()
    calls += [lambda: c.collisionCheck(gb, xd), lambda: eb.validate_control(c, gb, xd, vd, 0.1, 1.0),
              lambda: dwa.control(gb, xd, vd, vref=vd)]
    for call in calls:
        n = gb.launch_count()
        call()
        assert gb.launch_count() == n + 1


def test_device_path_equals_host_path_on_a_side_stream():
    import torch

    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(6)
    maps = mixed_maps(rng, copies=4)
    B = len(maps)
    host = eb.GridMapBatch(B)
    set_maps(host, maps)
    c = eb.Collision(*COL)
    dwa = eb.DynamicWindow(c, *DWA_OMNI, 3, 8, 5)
    poses = poses_for(rng, maps, 9)
    u = twists(rng, (B, 9))
    x0, vb = robots(rng, maps)
    xt = reference_trajectory(rng, maps)
    want = (c.collisionCheck(host, poses), eb.validate_control(c, host, poses, u, 0.1, 1.0),
            *dwa.control(host, x0, vb, vref=vb), *dwa.control(host, x0, vb, xt_ref=xt, dt_ref=0.1))
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        dev = eb.GridMapBatch(B)
        cells = [torch.from_numpy(m[0]).cuda() for m in maps]  # on the side stream, no synchronisation after
        dev.set(cells, [m[1] for m in maps], [(m[2], m[3]) for m in maps])
        T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        got = (c.collisionCheck(dev, T(poses)), eb.validate_control(c, dev, T(poses), T(u), 0.1, 1.0),
               *dwa.control(dev, T(x0), T(vb), vref=T(vb)), *dwa.control(dev, T(x0), T(vb), xt_ref=T(xt), dt_ref=0.1))
        got = [g.cpu().numpy() for g in got]
    for w, g in zip(want, got):
        np.testing.assert_array_equal(g, w)


def test_scale_4096_maps_sampled_against_oracle():
    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(4096)
    B = 4096
    maps = []
    for _ in range(B):
        ys, xs = int(rng.integers(40, 200)), int(rng.integers(40, 200))
        data = np.zeros((ys, xs), dtype=np.int8)
        data[rng.random((ys, xs)) < 0.004] = 100
        data[ys // 3: ys // 3 + 2, xs // 5: 4 * xs // 5] = 100
        maps.append((data, float(rng.choice([0.05, 0.1])), float(rng.uniform(-20, 20)), float(rng.uniform(-20, 20))))
    gb = eb.GridMapBatch(B)
    set_maps(gb, maps)
    c = eb.Collision(*COL)
    dwa = eb.DynamicWindow(c, *DWA_OMNI, 3, 8, 5)
    poses = poses_for(rng, maps, 4)
    u = twists(rng, (B, 4))
    x0, vb = robots(rng, maps)
    hit = c.collisionCheck(gb, poses)
    valid = eb.validate_control(c, gb, poses, u, 0.1, 0.5)
    found, uo = dwa.control(gb, x0, vb, vref=vb)
    for i in np.sort(rng.choice(B, 200, replace=False)):
        data, res, xmin, ymin = maps[i]
        np.testing.assert_array_equal(hit[i], Oracle.collision_check(data, res, xmin, ymin, COL, poses[i]))
        np.testing.assert_array_equal(valid[i], Oracle.validate_control(data, res, xmin, ymin, COL, poses[i], u[i], 0.1,
                                                                         0.5))
        fo, ua, _ = Oracle.dwa_control(data, res, xmin, ymin, COL, DWA_OMNI, (3, 8, 5), x0[i:i + 1], vb[i:i + 1],
                                       vref=vb[i:i + 1])
        assert found[i] == fo[0]
        np.testing.assert_array_equal(uo[i], ua[0])


def test_errors():
    import ctypes as C

    import ergodic_exploration_b200 as eb
    from ergodic_exploration_b200 import capi

    lib = capi.load()
    rng = np.random.default_rng(8)
    maps = mixed_maps(rng, copies=1, geoms=GEOMS[:3])
    gb = eb.GridMapBatch(3)
    cells, res, org = [m[0] for m in maps], [m[1] for m in maps], [(m[2], m[3]) for m in maps]
    c = eb.Collision(*COL)
    x = np.zeros((3, 3))
    gb.set(cells, res, org, update=[True, False, True])
    with pytest.raises(ValueError, match="no map"):  # a check before every instance has a map
        c.collisionCheck(gb, x)
    n = gb.launch_count()
    for bad_res in ([0.1, 0.0, 0.1], [0.1, -1.0, 0.1], [0.1, np.nan, 0.1], [0.1, np.inf, 0.1]):
        with pytest.raises(ValueError, match="resolution"):
            gb.set(cells, bad_res, org)
    with pytest.raises(ValueError, match="map 1"):  # a flagged instance without cells
        gb.set([cells[0], None, cells[2]], res, org)
    with pytest.raises(ValueError, match="xsize"):
        gb.set([cells[0], np.zeros((0, 4), dtype=np.int8), cells[2]], res, org)
    rr, oo = np.array(res), np.zeros((3, 2))
    xs, ys = (C.c_uint * 3)(4, 4, 4), (C.c_uint * 3)(4, 4, 4)
    for fn in (lib.eb_grid_batch_set_maps_host, lib.eb_grid_batch_set_maps_dev):  # NULL cells of a flagged map
        ptrs = (C.c_void_p * 3)(1, None, 1)
        assert fn(gb._h, C.addressof(ptrs), xs, ys, rr.ctypes.data, oo.ctypes.data, None) == capi.EB_ERR_INVALID_ARGUMENT
        assert b"NULL" in lib.eb_last_error()
    # more than 2^31 - 1 cells: refused before any cell is read
    ptrs = (C.c_void_p * 3)(1, 1, 1)
    xs, ys = (C.c_uint * 3)(4, 65536, 4), (C.c_uint * 3)(4, 32768, 4)
    assert lib.eb_grid_batch_set_maps_host(gb._h, C.addressof(ptrs), xs, ys, rr.ctypes.data, oo.ctypes.data,
                                           None) == capi.EB_ERR_INVALID_ARGUMENT
    assert b"2^31" in lib.eb_last_error()
    assert gb.launch_count() == n  # nothing was launched
    gb.set(cells, res, org)
    for radii in ((0.5, 0.2, 0.0, 0.5), (0.1, 0.2, 0.0, 101.0)):  # Collision constructor rules (collision.cpp:52-62)
        with pytest.raises(ValueError):
            _raw_collision(*radii).collisionCheck(gb, x)
        with pytest.raises(ValueError):
            eb.validate_control(_raw_collision(*radii), gb, x, x, 0.1, 1.0)
    out = np.empty(12, dtype=np.int32)
    pose = np.zeros((12, 3))
    for per in (0, -1, 1 << 30):  # per < 1, per * B beyond INT_MAX
        assert lib.eb_collision_check_batch_host(gb._h, C.byref(c.cfg), pose.ctypes.data, per,
                                                 out.ctypes.data) == capi.EB_ERR_INVALID_ARGUMENT
        assert lib.eb_validate_control_batch_host(gb._h, C.byref(c.cfg), pose.ctypes.data, pose.ctypes.data, per, 0.1,
                                                  1.0, out.ctypes.data) == capi.EB_ERR_INVALID_ARGUMENT
    assert gb.launch_count() == n + 1
    # DWA traj: the rollout (2 s) outlasts a 1 s reference trajectory -> EB_ERR_OUT_OF_RANGE
    dwa = eb.DynamicWindow(c, *DWA_OMNI, 3, 8, 5)
    x0, vb = robots(rng, maps)
    with pytest.raises(eb.ErgodicB200Error) as e:
        dwa.control(gb, x0, vb, xt_ref=np.zeros((10, 3)), dt_ref=0.1)
    assert e.value.status == capi.EB_ERR_OUT_OF_RANGE


def _raw_collision(*radii):
    """a Collision whose arguments the Python constructor would refuse, to reach the library's own checks"""
    import ergodic_exploration_b200 as eb
    from ergodic_exploration_b200.capi import EbCollision

    c = object.__new__(eb.Collision)
    c.cfg = EbCollision(*[float(r) for r in radii])
    return c
