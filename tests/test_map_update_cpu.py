"""CPU: the row-band map update calls (eb_grid_batch_set_rows_*, eb_grid_batch_get_map_host,
eb_set_map_targets_from_grid_batch) refuse NULL handles and arrays without a device, and the Python wrappers check
their arguments before they call the library."""
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
    rb = (C.c_uint * 2)(0, 0)
    rc = (C.c_uint * 2)(1, 1)
    cells = (C.c_byte * 16)()
    for fn, name in ((lib.eb_grid_batch_set_rows_dev, b"eb_grid_batch_set_rows_dev"),
                     (lib.eb_grid_batch_set_rows_host, b"eb_grid_batch_set_rows_host")):
        assert fn(None, C.addressof(ptrs), rb, rc, None) == bad
        assert name in lib.eb_last_error()
    assert lib.eb_grid_batch_get_map_host(None, 0, cells) == bad
    assert b"eb_grid_batch_get_map_host" in lib.eb_last_error()
    assert lib.eb_set_map_targets_from_grid_batch(None, None, None, None, None) == bad
    assert lib.eb_set_map_targets_from_grid_batch(None, None, rb, rc, None) == bad
    assert b"eb_set_map_targets_from_grid_batch" in lib.eb_last_error()


def _fake_grids(batch, shapes):
    import ergodic_exploration_b200 as eb

    from ergodic_exploration_b200 import capi

    o = object.__new__(eb.GridMapBatch)
    o._lib, o._h, o.batch, o.device, o._shape = capi.load(), None, batch, 0, list(shapes)
    return o


def test_set_rows_and_get_map_checks_raise(lib):
    gb = _fake_grids(2, [(6, 5), None])
    band = np.zeros((2, 5), dtype=np.int8)
    with pytest.raises(ValueError, match="2 bands"):
        gb.set_rows([band], [0, 0])
    with pytest.raises(ValueError, match="row_begin"):
        gb.set_rows([band, None], [0])
    with pytest.raises(ValueError, match="row_begin"):
        gb.set_rows([band, None], [-1, 0])
    with pytest.raises(ValueError, match="update"):
        gb.set_rows([band, None], [0, 0], update=[1])
    with pytest.raises(ValueError, match=r"\(n, 5\)"):
        gb.set_rows([np.zeros((2, 4), dtype=np.int8), None], [0, 0])
    with pytest.raises(ValueError, match="int8"):
        gb.set_rows([np.zeros((2, 5), dtype=np.int16), None], [0, 0])
    with pytest.raises(ValueError, match="no map"):
        gb.set_rows([None, band], [0, 0])
    with pytest.raises(ValueError, match="no map"):
        gb.get_map(1)
    with pytest.raises(ValueError, match="no map"):
        gb.get_map(2)


def test_set_map_targets_from_grids_checks_raise(lib):
    import ergodic_exploration_b200 as eb

    from ergodic_exploration_b200 import capi

    ctl = object.__new__(eb.ErgodicControl)
    ctl._lib, ctl._h, ctl.batch, ctl.device = capi.load(), None, 2, 0
    with pytest.raises(ValueError, match="holds 3 maps for 2"):
        ctl.setMapTargets(_fake_grids(3, [None] * 3))
    gb = _fake_grids(2, [None, None])
    with pytest.raises(ValueError, match="both"):
        ctl.setMapTargets(gb, row_begin=[0, 0])
    with pytest.raises(ValueError, match="row_count"):
        ctl.setMapTargets(gb, [0, 0], [1, 2, 3])
    with pytest.raises(TypeError, match="twice"):
        ctl.setMapTargets(gb, [0, 0], [1, 1], row_begin=[0, 0])
    with pytest.raises(TypeError, match="resolution and origin"):
        ctl.setMapTargets([np.zeros((2, 2), dtype=np.int8)] * 2)
