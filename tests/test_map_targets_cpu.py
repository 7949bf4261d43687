"""CPU: the per-instance map-target entry points (eb_set_map_targets_batch_*) validate their arguments without a
device, the Python wrapper checks shapes before it calls the library, and without a device there is no controller to
take map targets (no CPU fallback)."""
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
    for fn in (lib.eb_set_map_targets_batch_dev, lib.eb_set_map_targets_batch_host):
        assert fn(None, C.addressof(ptrs), xs, xs, d, d, None) == bad
        assert b"eb_set_map_targets_batch" in lib.eb_last_error()
        assert fn(None, None, xs, xs, d, d, None) == bad


class _Fake:
    """ErgodicControl's argument checks, without a controller behind them"""

    def __new__(cls, batch):
        import ergodic_exploration_b200 as eb

        from ergodic_exploration_b200 import capi

        o = object.__new__(eb.ErgodicControl)
        o._lib, o._h, o.batch, o.device = capi.load(), None, batch, 0
        return o


def test_wrapper_shape_checks_raise(lib):
    ec = _Fake(3)
    cells = [np.zeros((4, 5), dtype=np.int8)] * 3
    with pytest.raises(ValueError, match="needs 3 maps"):
        ec.setMapTargets(cells[:2], 0.1, np.zeros((3, 2)))
    with pytest.raises(ValueError):
        ec.setMapTargets(cells, [0.1, 0.1], np.zeros((3, 2)))  # resolution (2,) for B = 3
    with pytest.raises(ValueError):
        ec.setMapTargets(cells, 0.1, np.zeros((3, 3)))  # origin must be (B, 2)
    with pytest.raises(ValueError, match="update"):
        ec.setMapTargets(cells, 0.1, np.zeros((3, 2)), update=[True, False])
    with pytest.raises(ValueError, match="int8"):
        ec.setMapTargets([c.astype(np.int16) for c in cells], 0.1, np.zeros((3, 2)))
    with pytest.raises(ValueError, match="2-D"):
        ec.setMapTargets([np.zeros(5, dtype=np.int8)] * 3, 0.1, np.zeros((3, 2)))
    ec._h = None  # keep __del__ from reaching the library


def test_no_device_means_no_map_targets(lib):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import ergodic_exploration_b200 as eb

    with pytest.raises(eb.ErgodicB200Error) as e:
        eb.ErgodicControl(eb.Omni(), 0.1, 5.0, 0.1, 1.0, 10, 1000, 100, np.eye(3), [-1] * 3, [1] * 3, batch=3)
    assert e.value.status == eb.EB_ERR_NO_DEVICE


def test_cpp_map_targets_demo_compiles_warning_free():
    import shutil
    import subprocess

    cxx = shutil.which("g++")
    if cxx is None:
        pytest.skip("no C++ compiler")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([cxx, "-std=c++20", "-Wall", "-Wextra", "-Wno-unused-parameter", "-fsyntax-only",
                        "-I", os.path.join(root, "include"), "-I", os.path.join(root, "oracle", "shim"),
                        os.path.join(root, "tests", "cpp", "map_targets_demo.cpp")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "warning" not in r.stderr, r.stderr[-3000:]
