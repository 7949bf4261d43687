"""-m gpu: row-band map updates (GridMapBatch.set_rows / eb_grid_batch_set_rows_*) and entropy targets derived from
a grid batch with kept per-unit blocks (ErgodicControl.setMapTargets(grids, row_begin, row_count) /
eb_set_map_targets_from_grid_batch).  The arena is checked byte for byte against the expected maps, and every phi_k
row, extent, control() output and safe tick bit for bit against a controller given the whole cells through
setMapTargets(cells, resolution, origin)."""
import ctypes as C

import numpy as np
import pytest

from helpers import MODEL_OMNI, make_gpu, warm_ut
from test_gpu_map_targets import SHAPES, _maps

pytestmark = pytest.mark.gpu


def _bits(a):
    a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
    return np.ascontiguousarray(a).view(np.int64 if a.dtype == np.float64 else np.int32)


def _same(got, want, what):
    np.testing.assert_array_equal(_bits(got), _bits(want), what)


def _fresh(cells, res, origin, nb):
    """phik and extents of a new controller given the whole cells"""
    ref = make_gpu(MODEL_OMNI, len(cells), nb=nb)
    ref.setMapTargets(cells, res, origin)
    return ref.get_phik_batch()


def _check_targets(ctl, cells, res, origin, nb, what):
    ph, ext = ctl.get_phik_batch()
    wph, wext = _fresh(cells, res, origin, nb)
    _same(ph, wph, f"{what}: phi_k")
    _same(ext, wext, f"{what}: extent")


def _band(rng, ny):
    """(first row, rows): single rows, the last partial unit, whole maps, unaligned bands"""
    kind = rng.integers(0, 5)
    if kind == 0:
        return int(rng.integers(0, ny)), 1
    if kind == 1:
        return (ny - 1) // 64 * 64, ny - (ny - 1) // 64 * 64
    if kind == 2:
        return 0, ny
    r0 = int(rng.integers(0, ny))
    return r0, int(rng.integers(1, ny - r0 + 1))


def _step(rng, cells, p_flag=0.7):
    """random bands for a random subset; the expected maps are updated in place.  Returns (rows, rb, rc, update)"""
    B = len(cells)
    upd = rng.random(B) < p_flag
    rows, rb, rc = [None] * B, np.zeros(B, dtype=np.uint32), np.zeros(B, dtype=np.uint32)
    for i in range(B):
        ny, nx = cells[i].shape
        r0, n = _band(rng, ny)
        rb[i] = r0
        if rng.random() < 0.1:
            continue  # a flagged or unflagged instance with nothing to write
        band = rng.integers(-1, 101, size=(n, nx)).astype(np.int8)
        rows[i], rc[i] = band, n
        if upd[i]:
            cells[i][r0:r0 + n] = band
    return rows, rb, rc, upd


def _dev(a):
    import torch

    return [torch.from_numpy(np.ascontiguousarray(x)).cuda() if x is not None else None for x in a]


def _grids(cells, res, origin):
    import ergodic_exploration_b200 as eb

    gb = eb.GridMapBatch(len(cells))
    gb.set([c.copy() for c in cells], res, origin)
    return gb


@pytest.mark.parametrize("nb", [1, 10, 16, 32, 40, 64])
def test_row_sequences_arena_bytes_and_target_bits(nb):
    import torch

    rng = np.random.default_rng(900 + nb)
    shapes = list(SHAPES) + [tuple(int(v) for v in rng.integers(20, 300, 2)) for _ in range(6)]
    cells, res, origin = _maps(rng, shapes)
    B = len(cells)
    gb = _grids(cells, res, origin)
    ctl = make_gpu(MODEL_OMNI, B, nb=nb)
    ctl.setMapTargets(gb, np.zeros(B, dtype=np.uint32), np.ones(B, dtype=np.uint32))  # first call: whole maps
    _check_targets(ctl, cells, res, origin, nb, "first call")
    for step in range(6):
        rows, rb, rc, upd = _step(rng, cells)
        dev = step % 2 == 1
        gb.set_rows(_dev(rows) if dev else rows, rb, update=upd)
        if dev:
            torch.cuda.synchronize()
        for i in range(B):
            np.testing.assert_array_equal(gb.get_map(i), cells[i], f"step {step}: map {i} bytes")
        ctl.setMapTargets(gb, rb, np.where(upd, rc, 0).astype(np.uint32), update=upd)
        _check_targets(ctl, cells, res, origin, nb, f"nb {nb} step {step}")
    whole = make_gpu(MODEL_OMNI, B, nb=nb)
    whole.setMapTargets(gb)  # NULL ranges: the same bits
    _same(whole.get_phik_batch()[0], ctl.get_phik_batch()[0], "NULL ranges")


def test_whole_recompute_cases_match():
    rng = np.random.default_rng(11)
    nb = 16
    cells, res, origin = _maps(rng, [(120, 90), (64, 128), (333, 257), (17, 333), (40, 65)])
    B = len(cells)
    none = np.zeros(B, dtype=np.uint32)
    gb = _grids(cells, res, origin)
    ctl = make_gpu(MODEL_OMNI, B, nb=nb)
    ctl.setMapTargets(gb)
    # a grown map (more units than its kept slot: the kept blocks move), with empty declared ranges
    cells[1] = rng.integers(-1, 101, size=(700, 64)).astype(np.int8)
    cells[3] = rng.integers(-1, 101, size=(333, 18)).astype(np.int8)  # same rows, another xsize
    gb.set(cells, res, origin)
    ctl.setMapTargets(gb, none, none)
    _check_targets(ctl, cells, res, origin, nb, "grown map and new xsize")
    # a map replaced by set() with the same geometry
    cells[2] = rng.integers(-1, 101, size=cells[2].shape).astype(np.int8)
    upd = np.zeros(B, dtype=bool)
    upd[2] = True
    gb.set([c if f else None for c, f in zip(cells, upd)], res, origin, upd)
    ctl.setMapTargets(gb, none, none)
    _check_targets(ctl, cells, res, origin, nb, "replaced map")
    # a second grid batch with other cells in the same geometry
    other = [rng.integers(-1, 101, size=c.shape).astype(np.int8) for c in cells]
    gb2 = _grids(other, res, origin)
    ctl.setMapTargets(gb2, none, none)
    _check_targets(ctl, other, res, origin, nb, "second grid batch")
    ctl.setMapTargets(gb, none, none)
    _check_targets(ctl, cells, res, origin, nb, "back to the first grid batch")
    # a different resolution with the same shape
    res2 = res.copy()
    res2[0] *= 2
    gb.set(cells, res2, origin)
    ctl.setMapTargets(gb, none, none)
    _check_targets(ctl, cells, res2, origin, nb, "new resolution")


def test_replay_cosines_closed_loop_equals_pointer_flow():
    rng = np.random.default_rng(12)
    nb = 10
    cells, res, origin = _maps(rng, [(60, 45), (90, 130), (33, 71), (150, 100), (77, 77)])
    B = len(cells)
    a = make_gpu(MODEL_OMNI, B, nb=nb, batch_size=100)
    b = make_gpu(MODEL_OMNI, B, nb=nb, batch_size=100)
    a.setMapTargets(cells, res, origin)
    gb = _grids(cells, res, origin)
    b.setMapTargets(gb)
    lo = np.array([o for o in origin])
    for k in range(150):
        m = np.column_stack([lo[:, 0] + rng.uniform(0, 3, B), lo[:, 1] + rng.uniform(0, 3, B), rng.uniform(-3, 3, B)])
        a.addStateMemory(m)
        b.addStateMemory(m)
    for step in range(5):
        rows, rb, rc, upd = _step(rng, cells)
        if step == 3:  # map 0 moves: a new frame, its replay cosines re-derived
            upd[0], rows[0], rc[0] = True, None, 0
            origin[0] = origin[0] + 0.37
            gb.set([cells[0]] + [None] * (B - 1), res, origin, np.arange(B) == 0)
        a.setMapTargets(cells, res, origin)
        gb.set_rows(rows, rb, update=upd)
        b.setMapTargets(gb, rb, np.where(upd, rc, 0).astype(np.uint32), update=upd)
        x = np.column_stack([lo[:, 0] + rng.uniform(0, 3, B), lo[:, 1] + rng.uniform(0, 3, B), rng.uniform(-3, 3, B)])
        ut = warm_ut(rng, B, a.steps, MODEL_OMNI)
        a.set_ut(ut)
        b.set_ut(ut)
        ma, mb = np.empty(B), np.empty(B)
        _same(b.control(None, x, metric=mb), a.control(None, x, metric=ma), f"step {step} u0")
        _same(mb, ma, f"step {step} metric")
        _same(b.get_ut(), a.get_ut(), f"step {step} ut")


def test_update_masks_and_launch_counts():
    rng = np.random.default_rng(13)
    nb = 10
    cells, res, origin = _maps(rng, [(50, 200), (70, 64), (31, 129), (90, 1)])
    B = len(cells)
    gb = _grids(cells, res, origin)
    ctl = make_gpu(MODEL_OMNI, B, nb=nb)
    g0, c0 = gb.launch_count(), ctl.launch_count()
    ctl.setMapTargets(gb)
    assert ctl.launch_count() == c0 + 1
    ph0, ext0 = ctl.get_phik_batch()
    none = np.zeros(B, dtype=bool)
    # nothing flagged, or nothing to write / recompute: no launch
    zero, one = np.zeros(B, dtype=int), np.ones(B, dtype=int)
    gb.set_rows([np.zeros((1, c.shape[1]), np.int8) for c in cells], zero, update=none)
    gb.set_rows([None] * B, zero)
    ctl.setMapTargets(gb, zero, one, update=none)
    ctl.setMapTargets(gb, zero, zero)
    assert gb.launch_count() == g0 and ctl.launch_count() == c0 + 1
    _same(ctl.get_phik_batch()[0], ph0, "no work")
    # map 1 gets a band but only map 2's target is derived: map 1's target and the other maps stay as they were
    upd = np.array([False, True, True, False])
    band1 = rng.integers(-1, 101, size=(5, 70)).astype(np.int8)
    band2 = rng.integers(-1, 101, size=(2, 31)).astype(np.int8)
    rows = [np.full((3, 50), 100, np.int8), band1, band2, np.full((1, 90), 100, np.int8)]
    rb = np.array([10, 58, 127, 0])
    gb.set_rows(rows, rb, update=upd)
    assert gb.launch_count() == g0 + 1
    cells[1][58:63] = band1
    cells[2][127:129] = band2
    for i in range(B):
        np.testing.assert_array_equal(gb.get_map(i), cells[i], f"map {i}")
    ctl.setMapTargets(gb, rb, np.array([0, 5, 2, 0]), update=np.array([False, False, True, False]))
    assert ctl.launch_count() == c0 + 2
    ph, ext = ctl.get_phik_batch()
    want, _ = _fresh(cells, res, origin, nb)
    for i in (0, 1, 3):
        _same(ph[i], ph0[i], f"unflagged instance {i}")
    _same(ph[2], want[2], "flagged instance 2")
    _same(ext, ext0, "extents")
    # the rows of map 1 that changed are declared now: instance 1 catches up
    ctl.setMapTargets(gb, rb, np.array([0, 5, 0, 0]), update=np.array([False, True, False, False]))
    assert ctl.launch_count() == c0 + 3
    _same(ctl.get_phik_batch()[0], want, "after instance 1")


def test_safe_tick_after_both_flows():
    import torch

    import ergodic_exploration_b200 as eb
    from test_dwa_cpu import COL, DWA_OMNI
    from test_gpu_grid_batch import mixed_maps, robots
    from test_gpu_safe_control import _obstacles, safe

    rng = np.random.default_rng(14)
    geoms = [(120, 160, 0.05, -1.0, 2.0), (80, 90, 0.1, 0.0, 0.0), (60, 60, 0.1, 3.0, -2.0)] * 3
    maps = mixed_maps(rng, copies=1, geoms=geoms)
    B = len(maps)
    x0, vb = robots(rng, maps)
    maps = _obstacles(maps, x0)
    cells = [m[0].copy() for m in maps]
    res, origin = [m[1] for m in maps], [(m[2], m[3]) for m in maps]
    ut = warm_ut(rng, B, make_gpu(MODEL_OMNI, 1).steps, MODEL_OMNI)
    a, b = make_gpu(MODEL_OMNI, B), make_gpu(MODEL_OMNI, B)
    for c in (a, b):
        c.set_ut(ut)
    gba, gbb = _grids(cells, res, origin), _grids(cells, res, origin)
    b.setMapTargets(gbb)
    dwa = eb.DynamicWindow(eb.Collision(*COL), *DWA_OMNI, 3, 8, 5)
    x, v = torch.from_numpy(x0).cuda(), torch.from_numpy(vb).cuda()
    for tick in range(3):
        rows, rb, rc, upd = _step(rng, cells, p_flag=0.5)
        gba.set(cells, res, origin)  # (a) whole maps to both calls
        a.setMapTargets(cells, res, origin)
        gbb.set_rows(rows, rb, update=upd)  # (b) the bands, and only their units
        b.setMapTargets(gbb, rb, np.where(upd, rc, 0).astype(np.uint32), update=upd)
        ua, ba, ma = safe(a, gba, dwa, x, v)
        ub, bb, mb = safe(b, gbb, dwa, x, v)
        for name, g, w in (("u", ub, ua), ("branch", bb, ba), ("metric", mb, ma)):
            _same(g, w, f"tick {tick} {name}")
        x = eb.integrate_twist(x, ua, 0.1)
        v = ua


def test_side_stream_without_host_synchronisation():
    import torch

    import ergodic_exploration_b200 as eb

    rng = np.random.default_rng(15)
    nb = 16
    cells, res, origin = _maps(rng, [(200, 300), (64, 64), (99, 513), (7, 3)])
    B = len(cells)
    steps = [_step(rng, [c.copy() for c in cells]) for _ in range(4)]
    ctl = make_gpu(MODEL_OMNI, B, nb=nb)
    side = torch.cuda.Stream()
    keep, want = [], [c.copy() for c in cells]
    with torch.cuda.stream(side):
        gb = eb.GridMapBatch(B)
        first = [torch.from_numpy(c).cuda() for c in cells]
        gb.set(first, res, origin)
        ctl.setMapTargets(gb)
        for rows, rb, rc, upd in steps:
            d = _dev(rows)
            keep.append(d)
            gb.set_rows(d, rb, update=upd)
            ctl.setMapTargets(gb, rb, np.where(upd, rc, 0).astype(np.uint32), update=upd)
            for i in range(B):
                if upd[i] and rows[i] is not None:
                    want[i][rb[i]:rb[i] + rc[i]] = rows[i]
    side.synchronize()
    for i in range(B):
        np.testing.assert_array_equal(gb.get_map(i), want[i], f"map {i}")
    _check_targets(ctl, want, res, origin, nb, "side stream")
    del first, keep


def test_scale_4096_maps():
    import torch

    rng = np.random.default_rng(16)
    B, nb = 4096, 10
    sides = rng.integers(160, 641, size=(B, 2))
    dev = [torch.randint(-1, 101, (int(ny), int(nx)), dtype=torch.int8, device="cuda") for nx, ny in sides]
    res = np.full(B, 0.05)
    origin = rng.uniform(-20, 20, (B, 2))
    import ergodic_exploration_b200 as eb

    gb = eb.GridMapBatch(B)
    gb.set(dev, res, origin)
    ctl = make_gpu(MODEL_OMNI, B, nb=nb)
    ctl.setMapTargets(gb)
    upd = rng.random(B) < 0.1
    rb = np.array([int(rng.integers(0, ny - 64 + 1)) for _, ny in sides], dtype=np.uint32)
    rows = [torch.randint(-1, 101, (64, int(nx)), dtype=torch.int8, device="cuda") if f else None
            for (nx, _), f in zip(sides, upd)]
    gb.set_rows(rows, rb, update=upd)
    ctl.setMapTargets(gb, rb, np.where(upd, 64, 0).astype(np.uint32), update=upd)
    for i in np.flatnonzero(upd):
        dev[i][int(rb[i]):int(rb[i]) + 64] = rows[i]
    ref = make_gpu(MODEL_OMNI, B, nb=nb)
    ref.setMapTargets(dev, res, origin)
    _same(ctl.get_phik_batch()[0], ref.get_phik_batch()[0], "4096 maps")
    for i in np.flatnonzero(upd)[:8]:
        np.testing.assert_array_equal(gb.get_map(int(i)), dev[i].cpu().numpy(), f"map {i}")


def test_errors_leave_everything_unchanged():
    import ergodic_exploration_b200 as eb
    from ergodic_exploration_b200 import capi

    rng = np.random.default_rng(17)
    nb = 10
    cells, res, origin = _maps(rng, [(50, 130), (70, 64), (31, 200)])
    B = len(cells)
    gb = _grids(cells, res, origin)
    ctl = make_gpu(MODEL_OMNI, B, nb=nb)
    ctl.setMapTargets(gb)
    lib = capi.load()
    # a pending change of map 0 rows 100..109, written but not yet declared to the controller
    band = rng.integers(-1, 101, size=(10, 50)).astype(np.int8)
    gb.set_rows([band, None, None], np.array([100, 0, 0]))
    cells[0][100:110] = band
    state = lambda: ([gb.get_map(i) for i in range(B)], ctl.get_phik_batch(), gb.launch_count(), ctl.launch_count())
    before = state()
    rb3 = lambda *v: (C.c_uint * B)(*v)
    ptrs = (C.c_void_p * B)(None, None, None)
    bad = capi.EB_ERR_INVALID_ARGUMENT
    with pytest.raises(ValueError, match="pass its"):
        gb.set_rows([np.zeros((10, 50), np.int8), None, None], np.array([121, 0, 0]))
    assert lib.eb_grid_batch_set_rows_host(gb._h, C.addressof(ptrs), rb3(0, 0, 0), rb3(1, 0, 0), None) == bad  # NULL band
    assert lib.eb_grid_batch_set_rows_host(gb._h, C.addressof(ptrs), rb3(0xFFFFFFFF, 0, 0), rb3(2, 0, 0), None) == bad
    assert lib.eb_grid_batch_set_rows_dev(gb._h, None, rb3(0, 0, 0), rb3(0, 0, 0), None) == bad
    assert lib.eb_grid_batch_get_map_host(gb._h, 3, (C.c_byte * 16)()) == bad
    with pytest.raises(ValueError, match="pass its"):
        ctl.setMapTargets(gb, np.array([0, 0, 190]), np.array([0, 0, 11]))
    assert lib.eb_set_map_targets_from_grid_batch(ctl._h, gb._h, rb3(0, 0, 0), None, None) == bad
    with pytest.raises(ValueError, match="4 maps for 3"):
        ctl.setMapTargets(eb.GridMapBatch(4))
    four = _grids(cells + [cells[0]], np.append(res, res[0]), np.vstack([origin, origin[:1]]))
    assert lib.eb_set_map_targets_from_grid_batch(ctl._h, four._h, None, None, None) == bad
    empty = eb.GridMapBatch(B)
    with pytest.raises(ValueError, match="no map"):
        ctl.setMapTargets(empty)
    assert lib.eb_set_map_targets_from_grid_batch(ctl._h, empty._h, None, None, None) == bad
    part = eb.GridMapBatch(B)
    part.set([cells[0], None, None], res, origin, np.array([True, False, False]))
    assert lib.eb_grid_batch_set_rows_host(part._h, C.addressof(ptrs), rb3(0, 0, 0), rb3(0, 0, 0), None) == bad
    after = state()
    for i in range(B):
        np.testing.assert_array_equal(after[0][i], before[0][i], f"map {i}")
    _same(after[1][0], before[1][0], "phi_k")
    assert after[2:] == before[2:]
    # the kept blocks are intact: declaring the pending rows gives the whole-map bits
    ctl.setMapTargets(gb, np.array([100, 0, 0]), np.array([10, 0, 0]))
    _check_targets(ctl, cells, res, origin, nb, "after the refusals")
