"""CPU: the per-instance occupancy maps (eb_grid_batch_*) validate their arguments without a device, the Python
GridMapBatch checks shapes before it calls the library, and without a device there is no grid batch (no CPU
fallback)."""
import ctypes as C
import os

import numpy as np
import pytest


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g

    from ergodic_exploration_b200 import capi

    if not os.path.exists(capi.LIB_PATH):
        g.build()
    return capi.load()


def test_null_arguments_need_no_device(lib):
    from ergodic_exploration_b200 import capi

    bad = capi.EB_ERR_INVALID_ARGUMENT
    ptrs = (C.c_void_p * 2)(1, 1)
    xs = (C.c_uint * 2)(4, 4)
    d = (C.c_double * 4)(0.1, 0.1, 0.0, 0.0)
    for fn in (lib.eb_grid_batch_set_maps_dev, lib.eb_grid_batch_set_maps_host):
        assert fn(None, C.addressof(ptrs), xs, xs, d, d, None) == bad
        assert b"eb_grid_batch_set_maps" in lib.eb_last_error()
    col = capi.EbCollision(0.2, 1.0, 0.05, 0.65)
    dwa = capi.EbDwa()
    assert lib.eb_collision_check_batch_host(None, C.byref(col), None, 1, None) == bad
    assert lib.eb_validate_control_batch_dev(None, C.byref(col), None, None, 1, 0.1, 1.0, None) == bad
    assert lib.eb_dwa_control_twist_batch_dev(None, C.byref(col), C.byref(dwa), None, None, None, None, None, None) == bad
    assert lib.eb_dwa_control_traj_batch_host(None, C.byref(col), C.byref(dwa), None, None, None, 1, 0, 0.1, None, None,
                                              None) == bad
    h = C.c_void_p()
    assert lib.eb_grid_batch_create(0, 0, C.byref(h)) == bad  # batch < 1
    assert lib.eb_grid_batch_create(0, 4, None) == bad
    assert lib.eb_grid_batch_launch_count(None) == 0


class _Fake:
    """GridMapBatch's argument checks, without a device handle behind them"""

    def __new__(cls, batch):
        import ergodic_exploration_b200 as eb

        from ergodic_exploration_b200 import capi

        o = object.__new__(eb.GridMapBatch)
        o._lib, o._h, o.batch, o.device = capi.load(), None, batch, 0
        return o


def test_set_shape_checks_raise(lib):
    gb = _Fake(3)
    cells = [np.zeros((4, 5), dtype=np.int8)] * 3
    with pytest.raises(ValueError, match="needs 3 maps"):
        gb.set(cells[:2], 0.1, np.zeros((3, 2)))
    with pytest.raises(ValueError):
        gb.set(cells, [0.1, 0.1], np.zeros((3, 2)))  # resolution (2,) for B = 3
    with pytest.raises(ValueError):
        gb.set(cells, 0.1, np.zeros((3, 3)))  # origin must be (B, 2)
    with pytest.raises(ValueError, match="update"):
        gb.set(cells, 0.1, np.zeros((3, 2)), update=[True, False])
    with pytest.raises(ValueError, match="int8"):
        gb.set([c.astype(np.int16) for c in cells], 0.1, np.zeros((3, 2)))
    with pytest.raises(ValueError, match="2-D"):
        gb.set([np.zeros(5, dtype=np.int8)] * 3, 0.1, np.zeros((3, 2)))


def test_check_shape_checks_raise(lib):
    import ergodic_exploration_b200 as eb

    gb = _Fake(3)
    col = eb.Collision(0.2, 1.0, 0.05, 0.65)
    dwa = eb.DynamicWindow(col, 0.1, 2.0, 0.2, 1.0, 1.0, 2.0, 1.0, -1.0, 1.0, -1.0, 2.0, -2.0, 3, 8, 5)
    with pytest.raises(ValueError, match="poses"):
        col.collisionCheck(gb, np.zeros((4, 3)))  # B = 3
    with pytest.raises(ValueError, match="poses"):
        col.collisionCheck(gb, np.zeros((3, 2, 2)))
    with pytest.raises(ValueError, match="same shape"):
        eb.validate_control(col, gb, np.zeros((3, 2, 3)), np.zeros((3, 3)), 0.1, 1.0)
    with pytest.raises(ValueError, match="x0"):
        dwa.control(gb, np.zeros((3, 2, 3)), np.zeros((3, 3)), vref=np.zeros((3, 3)))  # one robot per map
    with pytest.raises(ValueError, match="vref"):
        dwa.control(gb, np.zeros((3, 3)), np.zeros((3, 3)), vref=np.zeros((2, 3)))
    with pytest.raises(ValueError, match="xt_ref"):
        dwa.control(gb, np.zeros((3, 3)), np.zeros((3, 3)), xt_ref=np.zeros((2, 10, 3)), dt_ref=0.1)
    with pytest.raises(ValueError, match="min_cost"):
        dwa.control(gb, np.zeros((3, 3)), np.zeros((3, 3)), vref=np.zeros((3, 3)), min_cost=np.zeros(2))


def test_no_device_means_no_grid_batch(lib):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import ergodic_exploration_b200 as eb

    with pytest.raises(eb.ErgodicB200Error) as e:
        eb.GridMapBatch(3)
    assert e.value.status == eb.EB_ERR_NO_DEVICE


def test_cpp_grid_batch_demo_compiles_warning_free():
    import shutil
    import subprocess

    cxx = shutil.which("g++")
    if cxx is None:
        pytest.skip("no C++ compiler")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([cxx, "-std=c++20", "-Wall", "-Wextra", "-Wno-unused-parameter", "-fsyntax-only",
                        "-I", os.path.join(root, "include"), "-I", os.path.join(root, "oracle", "shim"),
                        os.path.join(root, "tests", "cpp", "grid_batch_demo.cpp")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "warning" not in r.stderr, r.stderr[-3000:]
