"""-m gpu: per-instance targets and map frames (eb_*_batch calls): every instance owns its Gaussians, phi_k and
Fourier frame, as B reference ErgodicControl objects driven with their own maps.  One oracle object per instance;
tolerances from tests/helpers.py."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import (MODEL_OMNI, MODEL_SIMPLE_CART, assert_abs_rel_close, assert_coeff_close, make_gpu, make_oracle,
                     warm_ut)

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _instances(rng, B):
    """per-instance bounds (origins incl. maze-like offsets, extents 6..25 m) and 1..4 Gaussians inside each map"""
    bounds = np.empty((B, 4))
    mus, sgs = [], []
    for i in range(B):
        x0 = rng.choice([0.0, -8.350015, rng.uniform(-20, 20)])
        y0 = rng.choice([0.0, -13.950030, rng.uniform(-20, 20)])
        lx, ly = np.round(rng.uniform(6, 25, 2), 1)
        bounds[i] = (x0, x0 + lx, y0, y0 + ly)
        n = rng.integers(1, 5)
        mus.append(np.column_stack([x0 + rng.uniform(1, lx - 1, n), y0 + rng.uniform(1, ly - 1, n)]))
        sgs.append(rng.uniform(0.8, 2.5, (n, 2)))
    return bounds, mus, sgs


def _targets(mus, sgs):
    import ergodic_exploration_b200 as eb

    return [[eb.Gaussian(m, s) for m, s in zip(mu, sg)] for mu, sg in zip(mus, sgs)]


def _states(rng, bounds):
    x = np.empty((len(bounds), 3))
    for i, (x0, x1, y0, y1) in enumerate(bounds):
        x[i] = rng.uniform(x0 + 0.5, x1 - 0.5), rng.uniform(y0 + 0.5, y1 - 0.5), rng.uniform(-np.pi, np.pi)
    return x


def _per_inst_gpu(model, B, nb, mus, sgs, **kw):
    gpu = make_gpu(model, B, nb=nb, **kw)
    gpu.setTargets(_targets(mus, sgs))
    return gpu


def _compare(gpu, oracles, bounds, x, tag):
    metric = np.empty(gpu.batch)
    u0 = gpu.control(bounds, x, metric=metric)
    gck = gpu.get_ck()
    gut = gpu.get_ut()
    phik, ext = gpu.get_phik_batch()
    for i, o in enumerate(oracles):
        b = bounds[i]
        ou0 = o.control(tuple(b), x[i])
        last = o.last()
        assert_abs_rel_close(u0[i], ou0, f"{tag} u0[{i}]")
        assert_abs_rel_close(gut[i], o.get_ut(), f"{tag} ut[{i}]")
        assert_coeff_close(gck[i], last["ck"], f"{tag} c_k[{i}]")
        assert_abs_rel_close(metric[i], last["metric"], f"{tag} metric[{i}]")
        assert_coeff_close(phik[i], o.get_phik(), f"{tag} phi_k[{i}]")
    return u0


@pytest.mark.parametrize("model", [MODEL_SIMPLE_CART, MODEL_OMNI])
@pytest.mark.parametrize("nb", [7, 10, 16, 20, 32, 40])
def test_parity_distinct_frames_and_targets(model, nb):
    rng = np.random.default_rng(100 + nb + 7 * model)
    B = 37
    bounds, mus, sgs = _instances(rng, B)
    gpu = _per_inst_gpu(model, B, nb, mus, sgs)
    oracles = [make_oracle(model, nb=nb, mu=mus[i], sigma=sgs[i]) for i in range(B)]
    x = _states(rng, bounds)
    for step in range(2):  # teacher forced: both sides start every step from the same ut
        ut = warm_ut(rng, B, gpu.steps, model)
        gpu.set_ut(ut)
        for i, o in enumerate(oracles):
            o.set_ut(ut[i])
        _compare(gpu, oracles, bounds, x, f"nb={nb} step {step}")
    phik, ext = gpu.get_phik_batch()
    assert np.array_equal(ext, np.column_stack([bounds[:, 1] - bounds[:, 0], bounds[:, 3] - bounds[:, 2]]))
    # against the shared route (phi_k plan) on the same bounds and Gaussians: only the summation order differs
    for i in range(0, B, 6):
        one = make_gpu(model, 1, nb=nb, mu=mus[i], sigma=sgs[i])
        one.configTarget(tuple(bounds[i]))
        ph, _, _ = one.get_phik()
        assert_coeff_close(phik[i], ph, f"per-instance vs shared route, instance {i}", rtol=1e-12)


def _replay(rng, n, B, bounds):
    return [_states(rng, bounds) for _ in range(n)]


@pytest.mark.parametrize("nb", [10, 12, 16, 24, 40])
@pytest.mark.parametrize("stored", [0, 50, 150])
def test_replicated_frames_are_bit_identical_to_shared(nb, stored):
    import torch

    rng = np.random.default_rng(nb * 1000 + stored)
    B = 64
    bounds = (-8.350015, -8.350015 + 19.9, -13.950030, -13.950030 + 31.8)
    shared = make_gpu(MODEL_OMNI, B, nb=nb)
    per = make_gpu(MODEL_OMNI, B, nb=nb)
    shared.configTarget(bounds)
    ph, lx, ly = shared.get_phik()
    mems = _replay(rng, stored, B, np.tile(bounds, (B, 1)))
    for m in mems:
        shared.addStateMemory(m)
        per.addStateMemory(m)
    per.set_phik_batch(torch.from_numpy(np.tile(ph, (B, 1))).cuda(), torch.tensor([[lx, ly]] * B, dtype=torch.float64).cuda())
    bb = np.tile(bounds, (B, 1))
    x = _states(rng, bb)
    ut = warm_ut(rng, B, shared.steps, MODEL_OMNI)
    shared.set_ut(ut)
    per.set_ut(ut)
    idx = rng.integers(0, stored, size=(B, 100)).astype(np.int32) if stored > 100 else None
    for step in range(2):
        ms, mp = np.empty(B), np.empty(B)
        us = shared.control(bounds, x, mem_idx=idx, metric=ms)
        up = per.control(bb, x, mem_idx=idx, metric=mp)
        assert np.array_equal(us, up), f"u0 step {step}"
        assert np.array_equal(ms, mp), f"metric step {step}"
        assert np.array_equal(shared.get_ut(), per.get_ut()), f"ut step {step}"
        assert np.array_equal(shared.get_ck(), per.get_ck()), f"c_k step {step}"


def test_frame_moves_after_memory_is_stored():
    rng = np.random.default_rng(5)
    B, nb = 24, 10
    bounds, mus, sgs = _instances(rng, B)
    gpu = _per_inst_gpu(MODEL_OMNI, B, nb, mus, sgs, batch_size=20)
    oracles = [make_oracle(MODEL_OMNI, nb=nb, batch_size=20, mu=mus[i], sigma=sgs[i]) for i in range(B)]
    assert gpu.configTargets(bounds).all()
    for _ in range(12):  # stored <= batch_size: every state is used, in insertion order
        m = _states(rng, bounds)
        gpu.addStateMemory(m)
        for i, o in enumerate(oracles):
            o.add_state_memory(m[i])
    x = _states(rng, bounds)
    ut = warm_ut(rng, B, gpu.steps, MODEL_OMNI)
    gpu.set_ut(ut)
    for i, o in enumerate(oracles):
        o.set_ut(ut[i])
    _compare(gpu, oracles, bounds, x, "before the move")
    ph0, _ = gpu.get_phik_batch()
    moved = bounds.copy()
    grow = np.arange(B) % 3 == 0
    shift = np.arange(B) % 3 == 1
    moved[grow, 1] += 2.0  # the map grew: extent changes
    moved[grow, 3] += 1.0
    moved[shift] += np.array([1.5, 1.5, -2.0, -2.0])  # same extent, new origin
    rebuilt = gpu.configTargets(moved)
    assert np.array_equal(rebuilt, grow)
    ph1, ext = gpu.get_phik_batch()
    assert np.array_equal(ph1[~grow], ph0[~grow])
    _compare(gpu, oracles, moved, x, "after the move")  # the stored rows' cosines follow the moved frames


@pytest.mark.skipif(os.environ.get("EB_REPLAY_COS") == "0", reason="already the uncached run")
def test_frame_moves_without_replay_cosine_cache():
    env = dict(os.environ, EB_REPLAY_COS="0")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", os.path.abspath(__file__),
                        "-k", "test_frame_moves_after_memory_is_stored or (bit_identical and 150)"],
                       cwd=HERE, env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


def test_map_rows_through_map_target():
    import torch

    import ergodic_exploration_b200 as eb
    from oracle.pyoracle import Oracle
    from test_gpu_map_target import centre_phik

    rng = np.random.default_rng(21)
    nb, res = 10, 0.05
    shapes = [(120, 90), (200, 200), (96, 160)]
    B = len(shapes)
    gpu = make_gpu(MODEL_OMNI, B, nb=nb)
    rows = torch.empty((B, nb * nb), dtype=torch.float64, device="cuda")
    ext = torch.empty((B, 2), dtype=torch.float64, device="cuda")
    wants = []
    for i, (nx, ny) in enumerate(shapes):
        cells = rng.integers(-1, 101, size=(ny, nx)).astype(np.int8)
        mt = eb.MapTarget(nx, ny, res, nb)
        mt.execute(torch.from_numpy(cells).cuda(), phik=rows[i])
        ext[i, 0], ext[i, 1] = mt.lx, mt.ly
        wants.append((centre_phik(Oracle.entropy_grid(cells), res, nb), mt.lx, mt.ly))
    gpu.set_phik_batch(rows, ext)
    bounds = np.array([(0.0, lx, 0.0, ly) for _, lx, ly in wants])
    x = _states(rng, bounds)
    ut = warm_ut(rng, B, gpu.steps, MODEL_OMNI)
    gpu.set_ut(ut)
    u0 = gpu.control(bounds, x)
    for i, (want, lx, ly) in enumerate(wants):
        o = make_oracle(MODEL_OMNI, nb=nb)
        o.set_phik(want, lx, ly)
        o.set_ut(ut[i])
        assert_abs_rel_close(u0[i], o.control(tuple(bounds[i]), x[i]), f"u0[{i}] with a map-derived row")


def test_errors_and_lifetime():
    from ergodic_exploration_b200 import capi

    lib = capi.load()
    rng = np.random.default_rng(8)
    B, nb = 6, 10
    bounds, mus, sgs = _instances(rng, B)
    gpu = _per_inst_gpu(MODEL_OMNI, B, nb, mus, sgs)
    x = _states(rng, bounds)
    gpu.set_ut(warm_ut(rng, B, gpu.steps, MODEL_OMNI))
    gpu.control(bounds, x)
    # shared target calls on a per-instance controller
    ph = np.zeros(nb * nb)
    assert lib.eb_set_phik(gpu._h, ph.ctypes.data, 1.0, 1.0) == capi.EB_ERR_INVALID_ARGUMENT
    assert lib.eb_config_target(gpu._h, 0.0, 1.0, 0.0, 1.0, None) == capi.EB_ERR_INVALID_ARGUMENT
    assert lib.eb_get_phik(gpu._h, ph.ctypes.data, None, None) == capi.EB_ERR_INVALID_ARGUMENT
    assert lib.eb_set_target_gaussians(gpu._h, 0, None, None) == capi.EB_ERR_INVALID_ARGUMENT
    u0 = np.empty((B, 3))
    assert lib.eb_control_host(gpu._h, 0.0, 10.0, 0.0, 10.0, x.ctypes.data, None, u0.ctypes.data, None) == \
        capi.EB_ERR_INVALID_ARGUMENT
    assert lib.eb_control_dev_gather(gpu._h, C.c_void_p(1), 0.0, 10.0, 0.0, 10.0, None, None, None) == \
        capi.EB_ERR_UNSUPPORTED
    assert lib.eb_control_dev_gather_wait(gpu._h, C.c_void_p(1), 0.0, 10.0, 0.0, 10.0, None, None, None) == \
        capi.EB_ERR_UNSUPPORTED
    # clone + one step: the same bits on both copies; bounds None == unchanged bounds
    twin = gpu.clone()
    ua = gpu.control(bounds, x)
    ub = twin.control(None, x)
    assert np.array_equal(ua, ub)
    assert np.array_equal(gpu.get_ut(), twin.get_ut()) and np.array_equal(gpu.get_ck(), twin.get_ck())
    # an instance whose extent moved without Gaussians
    gpu.setTargets([[] if i == 2 else t for i, t in enumerate(_targets(mus, sgs))])
    moved = bounds.copy()
    moved[2, 1] += 1.0
    gpu.configTargets(moved)
    with pytest.raises(ValueError):
        gpu.check()
    gpu.check()  # reported once; the controller stays usable
    gpu.control(bounds, x)


def test_scale_4096_distinct_frames():
    rng = np.random.default_rng(4096)
    B, nb = 4096, 10
    bounds, mus, sgs = _instances(rng, B)
    gpu = _per_inst_gpu(MODEL_OMNI, B, nb, mus, sgs)
    x = _states(rng, bounds)
    ut = warm_ut(rng, B, gpu.steps, MODEL_OMNI)
    gpu.set_ut(ut)
    metric = np.empty(B)
    u0 = gpu.control(bounds, x, metric=metric)
    phik, _ = gpu.get_phik_batch()
    for i in rng.choice(B, 16, replace=False):
        o = make_oracle(MODEL_OMNI, nb=nb, mu=mus[i], sigma=sgs[i])
        o.set_ut(ut[i])
        assert_abs_rel_close(u0[i], o.control(tuple(bounds[i]), x[i]), f"u0[{i}]")
        assert_abs_rel_close(metric[i], o.last()["metric"], f"metric[{i}]")
        assert_coeff_close(phik[i], o.get_phik(), f"phi_k[{i}]")
