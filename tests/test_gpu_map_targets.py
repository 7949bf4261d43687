"""-m gpu: map-derived (entropy) targets per instance in one launch (eb_set_map_targets_batch_*): every instance gets
the phi_k row of its own occupancy map and that map's frame.  Rows are checked against the CPU oracle's entropy +
spatialCoeff, against the single-map MapTarget, for composition invariance, and in closed loops; tolerances from
tests/helpers.py."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import MODEL_OMNI, assert_abs_rel_close, assert_coeff_close, make_gpu, make_oracle, warm_ut
from oracle.pyoracle import Oracle
from test_gpu_map_target import centre_phik

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
MAZE = (-8.350015, -13.950030)
# (xsize, ysize): single cell, single row, single column, odd widths, and one map on the fused single-map route
SHAPES = [(1, 1), (1, 37), (37, 1), (17, 333), (120, 90), (200, 200), (333, 257), (640, 512)]


def _maps(rng, shapes):
    cells = [rng.integers(-1, 101, size=(ny, nx)).astype(np.int8) for nx, ny in shapes]
    res = np.array([0.05 if i % 2 == 0 else 0.1 for i in range(len(shapes))])
    origin = np.array([MAZE if i % 3 == 0 else (0.0, 0.0) if i % 3 == 1 else tuple(rng.uniform(-20, 20, 2))
                       for i in range(len(shapes))])
    return cells, res, origin


def _mixed(rng, B=25):
    shapes = list(SHAPES) + [tuple(rng.integers(20, 300, 2)) for _ in range(B - len(SHAPES))]
    return _maps(rng, shapes)


def _dev(cells):
    import torch

    return [torch.from_numpy(c).cuda() for c in cells]


def _bounds(cells, res, origin):
    return np.array([(o[0], o[0] + c.shape[1] * r, o[1], o[1] + c.shape[0] * r) for c, r, o in zip(cells, res, origin)])


def _states(rng, bounds):
    x = np.empty((len(bounds), 3))
    for i, (x0, x1, y0, y1) in enumerate(bounds):
        x[i] = rng.uniform(x0, x1), rng.uniform(y0, y1), rng.uniform(-np.pi, np.pi)
    return x


@pytest.mark.parametrize("nb", [1, 7, 10, 16, 20, 32, 40, 64])
def test_parity_mixed_shapes(nb):
    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(300 + nb)
    cells, res, origin = _mixed(rng)
    B = len(cells)
    gpu = make_gpu(MODEL_OMNI, B, nb=nb)
    gpu.setMapTargets(_dev(cells), res, origin)
    phik, ext = gpu.get_phik_batch()
    want_ext = np.array([(c.shape[1] * r, c.shape[0] * r) for c, r in zip(cells, res)])
    assert np.array_equal(ext, want_ext)
    for i, c in enumerate(cells):
        ny, nx = c.shape
        mt = eb.MapTarget(nx, ny, res[i], nb)
        assert_coeff_close(phik[i], mt.execute(c), f"nb={nb} map {i} ({nx}x{ny}) vs MapTarget", rtol=1e-12)
        if nx * ny * nb * nb <= 4_000_000:
            assert_coeff_close(phik[i], centre_phik(Oracle.entropy_grid(c), res[i], nb), f"nb={nb} map {i} vs oracle")
    # the host path runs the same kernel: the same bits
    host = make_gpu(MODEL_OMNI, B, nb=nb)
    host.setMapTargets(cells, res, origin)
    ph2, ext2 = host.get_phik_batch()
    assert np.array_equal(ph2, phik) and np.array_equal(ext2, ext)


def test_composition_invariance_and_determinism():
    rng = np.random.default_rng(7)
    nb = 16
    cells, res, origin = _mixed(rng, 12)
    B = len(cells)
    gpu = make_gpu(MODEL_OMNI, B, nb=nb)
    gpu.setMapTargets(_dev(cells), res, origin)
    ph_a, _ = gpu.get_phik_batch()
    gpu.setMapTargets(_dev(cells), res, origin)
    ph_b, _ = gpu.get_phik_batch()
    assert np.array_equal(ph_a, ph_b), "two identical calls"
    for i in (0, 5, 7, 11):
        one = make_gpu(MODEL_OMNI, 1, nb=nb)
        one.setMapTargets([cells[i]], res[i:i + 1], origin[i:i + 1])
        assert np.array_equal(one.get_phik_batch()[0][0], ph_a[i]), f"map {i}: B = 1 vs the mixed batch"
    # the other maps change (new cells and shapes): row 7 keeps its bits
    other, ores, oorg = _mixed(np.random.default_rng(8), 12)
    other[7], ores[7], oorg[7] = cells[7], res[7], origin[7]
    gpu.setMapTargets(_dev(other), ores, oorg)
    assert np.array_equal(gpu.get_phik_batch()[0][7], ph_a[7])


def test_update_mask():
    from helpers import TARGET_MU, TARGET_SIGMA

    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(9)
    nb, B = 10, 9
    cells, res, origin = _maps(rng, [tuple(rng.integers(30, 200, 2)) for _ in range(B)])
    gpu = make_gpu(MODEL_OMNI, B, nb=nb)
    gpu.setTargets([[eb.Gaussian(m, s) for m, s in zip(TARGET_MU, TARGET_SIGMA)]] * B)
    bounds = np.array([(0.0, 10.0 + i, -1.0, 9.0 + 0.5 * i) for i in range(B)])
    assert gpu.configTargets(bounds).all()
    ph0, ext0 = gpu.get_phik_batch()
    upd = np.arange(B) % 3 == 1
    launches = gpu.launch_count()
    gpu.setMapTargets([c if u else None for c, u in zip(_dev(cells), upd)], res, origin, update=upd)
    assert gpu.launch_count() - launches == 1
    ph1, ext1 = gpu.get_phik_batch()
    assert np.array_equal(ph1[~upd], ph0[~upd]) and np.array_equal(ext1[~upd], ext0[~upd])
    full = make_gpu(MODEL_OMNI, B, nb=nb)
    full.setMapTargets(cells, res, origin)
    phf, extf = full.get_phik_batch()
    assert np.array_equal(ph1[upd], phf[upd]) and np.array_equal(ext1[upd], extf[upd])
    assert not np.array_equal(ph1[upd], ph0[upd])
    # the unflagged instances keep their Gaussian frames: configure with the old bounds rebuilds nothing there
    x = _states(rng, bounds)
    gpu.set_ut(warm_ut(rng, B, gpu.steps, MODEL_OMNI))
    b2 = bounds.copy()
    b2[upd] = _bounds(cells, res, origin)[upd]
    rebuilt = gpu.configTargets(b2)
    assert not rebuilt.any()
    gpu.control(None, x)


def _oracles(cells, res, nb, batch_size):
    out = []
    for c, r in zip(cells, res):
        o = make_oracle(MODEL_OMNI, nb=nb, batch_size=batch_size)
        o.set_phik(centre_phik(Oracle.entropy_grid(c), r, nb), c.shape[1] * r, c.shape[0] * r)
        out.append(o)
    return out


@pytest.mark.parametrize("stored", [0, 150])
def test_closed_loop_against_oracle(stored):
    rng = np.random.default_rng(40 + stored)
    nb = 10
    cells, res, origin = _maps(rng, [(60, 45), (90, 120), (33, 71), (150, 100), (77, 77)])
    B = len(cells)
    gpu = make_gpu(MODEL_OMNI, B, nb=nb, batch_size=100)
    gpu.setMapTargets(_dev(cells), res, origin)
    oracles = _oracles(cells, res, nb, 100)
    bounds = _bounds(cells, res, origin)
    for _ in range(stored):
        m = _states(rng, bounds)
        gpu.addStateMemory(m)
        for i, o in enumerate(oracles):
            o.add_state_memory(m[i])
    idx = rng.integers(0, stored, size=(B, 100)).astype(np.int32) if stored > 100 else None

    def step(grid, tag):
        x = _states(rng, bounds)
        ut = warm_ut(rng, B, gpu.steps, MODEL_OMNI)
        gpu.set_ut(ut)
        metric = np.empty(B)
        u0 = gpu.control(grid, x, mem_idx=idx, metric=metric)
        gut, gck = gpu.get_ut(), gpu.get_ck()
        for i, o in enumerate(oracles):
            o.set_ut(ut[i])
            ou = o.control(tuple(bounds[i]), x[i], mem_idx=idx[i] if idx is not None else None)
            assert_abs_rel_close(u0[i], ou, f"{tag} u0[{i}]")
            assert_abs_rel_close(gut[i], o.get_ut(), f"{tag} ut[{i}]")
            assert_coeff_close(gck[i], o.last()["ck"], f"{tag} c_k[{i}]")
            assert_abs_rel_close(metric[i], o.last()["metric"], f"{tag} metric[{i}]")

    step(bounds, "bounds of the maps")
    step(None, "bounds None")
    # map 2 grows: new cells and a larger xsize; its replay cosines follow the new frame
    grown = rng.integers(-1, 101, size=(71, 60)).astype(np.int8)
    cells[2] = grown
    upd = np.zeros(B, dtype=bool)
    upd[2] = True
    gpu.setMapTargets([c if u else None for c, u in zip(_dev(cells), upd)], res, origin, update=upd)
    oracles[2].set_phik(centre_phik(Oracle.entropy_grid(grown), res[2], nb), 60 * res[2], 71 * res[2])
    bounds = _bounds(cells, res, origin)
    step(None, "after growth, bounds None")
    step(bounds, "after growth, bounds of the maps")


@pytest.mark.skipif(os.environ.get("EB_REPLAY_COS") == "0", reason="already the uncached run")
def test_closed_loop_without_replay_cosine_cache():
    env = dict(os.environ, EB_REPLAY_COS="0")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", os.path.abspath(__file__),
                        "-k", "test_closed_loop_against_oracle and 150"], cwd=HERE, env=env, capture_output=True,
                       text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


def test_against_map_target_loop():
    import torch

    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(12)
    nb = 12
    cells, res, origin = _mixed(rng, 10)
    B = len(cells)
    new = make_gpu(MODEL_OMNI, B, nb=nb)
    new.setMapTargets(_dev(cells), res, origin)
    old = make_gpu(MODEL_OMNI, B, nb=nb)
    rows = torch.empty((B, nb * nb), dtype=torch.float64, device="cuda")
    ext = torch.empty((B, 2), dtype=torch.float64, device="cuda")
    for i, c in enumerate(cells):
        mt = eb.MapTarget(c.shape[1], c.shape[0], res[i], nb)
        mt.execute(torch.from_numpy(c).cuda(), phik=rows[i])
        ext[i, 0], ext[i, 1] = mt.lx, mt.ly
    old.set_phik_batch(rows, ext)
    bounds = _bounds(cells, res, origin)
    x = _states(rng, bounds)
    ut = warm_ut(rng, B, new.steps, MODEL_OMNI)
    new.set_ut(ut)
    old.set_ut(ut)
    u_new = new.control(bounds, x)
    u_old = old.control(bounds, x)
    assert_abs_rel_close(u_new, u_old, "u0: one launch vs the MapTarget loop", rtol=1e-12)


def test_one_launch_per_call():
    rng = np.random.default_rng(13)
    cells, res, origin = _mixed(rng, 16)
    gpu = make_gpu(MODEL_OMNI, len(cells), nb=10)
    dev = _dev(cells)
    for nb_calls in range(3):
        l0 = gpu.launch_count()
        gpu.setMapTargets(dev, res, origin)
        assert gpu.launch_count() - l0 == 1


def test_scale_4096_maps():
    rng = np.random.default_rng(4096)
    B, nb = 4096, 10
    shapes = [tuple(rng.integers(100, 301, 2)) for _ in range(B)]
    cells, res, origin = _maps(rng, shapes)
    gpu = make_gpu(MODEL_OMNI, B, nb=nb)
    gpu.setMapTargets(_dev(cells), res, origin)
    bounds = _bounds(cells, res, origin)
    x = _states(rng, bounds)
    ut = warm_ut(rng, B, gpu.steps, MODEL_OMNI)
    gpu.set_ut(ut)
    metric = np.empty(B)
    u0 = gpu.control(None, x, metric=metric)
    phik, ext = gpu.get_phik_batch()
    for i in rng.choice(B, 16, replace=False):
        want = centre_phik(Oracle.entropy_grid(cells[i]), res[i], nb)
        assert_coeff_close(phik[i], want, f"phi_k[{i}]")
        o = make_oracle(MODEL_OMNI, nb=nb)
        o.set_phik(want, ext[i, 0], ext[i, 1])
        o.set_ut(ut[i])
        assert_abs_rel_close(u0[i], o.control(tuple(bounds[i]), x[i]), f"u0[{i}]")
        assert_abs_rel_close(metric[i], o.last()["metric"], f"metric[{i}]")


def test_errors_and_lifetime():
    from ergodic_exploration_b200 import capi

    lib = capi.load()
    rng = np.random.default_rng(14)
    B, nb = 4, 10
    cells, res, origin = _maps(rng, [(40, 30), (25, 60), (50, 50), (31, 17)])
    dev = _dev(cells)
    gpu = make_gpu(MODEL_OMNI, B, nb=nb)
    ptrs = (C.c_void_p * B)(*[c.data_ptr() for c in dev])
    xs = np.array([c.shape[1] for c in cells], dtype=np.uint32)
    ys = np.array([c.shape[0] for c in cells], dtype=np.uint32)
    org = np.ascontiguousarray(origin)

    def call(xs=xs, ys=ys, res=res, ptrs=ptrs, upd=None):
        res = np.ascontiguousarray(res, dtype=np.float64)
        return lib.eb_set_map_targets_batch_dev(gpu._h, C.addressof(ptrs), xs.ctypes.data, ys.ctypes.data,
                                                res.ctypes.data, org.ctypes.data,
                                                upd.ctypes.data if upd is not None else None)

    l0 = gpu.launch_count()
    bad = capi.EB_ERR_INVALID_ARGUMENT
    for k, v in ((xs, 0), (ys, 0)):
        z = k.copy()
        z[1] = v
        assert call(**({"xs": z} if k is xs else {"ys": z})) == bad
    for r in (0.0, -0.1, np.inf, np.nan):
        rr = res.copy()
        rr[2] = r
        assert call(res=rr) == bad
    big = xs.copy()
    big[0] = 65536
    yb = ys.copy()
    yb[0] = 32768
    assert call(xs=big, ys=yb) == bad  # 2^31 cells
    nul = (C.c_void_p * B)(*[c.data_ptr() for c in dev])
    nul[3] = None
    assert call(ptrs=nul) == bad
    assert gpu.launch_count() == l0, "refused calls launch nothing"
    upd = np.array([1, 1, 1, 0], dtype=np.int32)
    assert call(ptrs=nul, upd=upd) == capi.EB_OK  # the NULL map is not flagged
    assert gpu.launch_count() == l0 + 1
    assert call() == capi.EB_OK
    # shared target calls are refused afterwards, peer gather is unsupported
    ph = np.zeros(nb * nb)
    assert lib.eb_set_phik(gpu._h, ph.ctypes.data, 1.0, 1.0) == bad
    assert lib.eb_config_target(gpu._h, 0.0, 1.0, 0.0, 1.0, None) == bad
    assert lib.eb_get_phik(gpu._h, ph.ctypes.data, None, None) == bad
    assert lib.eb_control_dev_gather(gpu._h, C.c_void_p(1), 0.0, 10.0, 0.0, 10.0, None, None, None) == \
        capi.EB_ERR_UNSUPPORTED
    # clone carries the map-derived rows and frames: one step gives the same bits on both copies
    bounds = _bounds(cells, res, origin)
    x = _states(rng, bounds)
    gpu.set_ut(warm_ut(rng, B, gpu.steps, MODEL_OMNI))
    twin = gpu.clone()
    assert all(np.array_equal(a, b) for a, b in zip(gpu.get_phik_batch(), twin.get_phik_batch()))
    ua = gpu.control(None, x)
    ub = twin.control(bounds, x)
    assert np.array_equal(ua, ub)
    assert np.array_equal(gpu.get_ut(), twin.get_ut()) and np.array_equal(gpu.get_ck(), twin.get_ck())
    with pytest.raises(ValueError):
        gpu.setMapTargets([cells[0]] + [c.astype(np.int16) for c in cells[1:]], res, origin)
