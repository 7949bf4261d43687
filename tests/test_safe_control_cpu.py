"""CPU: the safe control tick (eb_control_safe_batch_*) refuses NULL handles without a device, ErgodicControl.control_safe
checks shapes and paths before it calls the library, and the C++ demo of b200::controlSafe compiles warning-free."""
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


def test_null_handles_need_no_device(lib):
    from ergodic_exploration_b200 import capi

    col = capi.EbCollision(0.2, 1.0, 0.05, 0.65)
    dwa = capi.EbDwa()
    x = np.zeros((2, 3))
    u, b = np.empty((2, 3)), np.empty(2, dtype=np.int32)
    for fn, name in ((lib.eb_control_safe_batch_dev, b"eb_control_safe_batch_dev"),
                     (lib.eb_control_safe_batch_host, b"eb_control_safe_batch_host")):
        assert fn(None, None, C.byref(col), C.byref(dwa), 0.1, 1.0, None, x.ctypes.data, None, x.ctypes.data,
                  u.ctypes.data, b.ctypes.data, None) == capi.EB_ERR_INVALID_ARGUMENT
        assert name in lib.eb_last_error()


class _Fakes:
    """an ErgodicControl and a GridMapBatch without device handles behind them: their argument checks only"""

    def __init__(self, batch, grid_batch=None):
        import ergodic_exploration_b200 as eb

        from ergodic_exploration_b200 import capi

        self.ctl = object.__new__(eb.ErgodicControl)
        self.ctl._lib, self.ctl._h, self.ctl.batch, self.ctl.device = capi.load(), None, batch, 0
        self.gb = object.__new__(eb.GridMapBatch)
        self.gb._lib, self.gb._h, self.gb.batch, self.gb.device = capi.load(), None, grid_batch or batch, 0
        col = eb.Collision(0.2, 1.0, 0.05, 0.65)
        self.dwa = eb.DynamicWindow(col, 0.1, 2.0, 0.2, 1.0, 1.0, 2.0, 1.0, -1.0, 1.0, -1.0, 2.0, -2.0, 3, 8, 5)


def test_control_safe_argument_checks_raise(lib):
    f = _Fakes(3)
    z = np.zeros((3, 3))
    with pytest.raises(ValueError, match="x"):
        f.ctl.control_safe(f.gb, f.dwa, np.zeros((4, 3)), z, 0.1, 1.0)
    with pytest.raises(ValueError, match="x"):
        f.ctl.control_safe(f.gb, f.dwa, np.zeros((3, 2, 3)), z, 0.1, 1.0)  # one pose per robot
    with pytest.raises(ValueError, match="vb"):
        f.ctl.control_safe(f.gb, f.dwa, z, np.zeros((3, 2)), 0.1, 1.0)
    with pytest.raises(ValueError):
        f.ctl.control_safe(f.gb, f.dwa, z, z, 0.1, 1.0, bounds=np.zeros((3, 3)))
    with pytest.raises(ValueError, match="metric"):
        f.ctl.control_safe(f.gb, f.dwa, z, z, 0.1, 1.0, metric=np.zeros(2))
    with pytest.raises(ValueError, match="metric"):
        f.ctl.control_safe(f.gb, f.dwa, z, z, 0.1, 1.0, metric=np.zeros(3, dtype=np.float32))
    g = _Fakes(3, grid_batch=4)
    with pytest.raises(ValueError, match="4 maps for 3 instances"):
        g.ctl.control_safe(g.gb, g.dwa, z, z, 0.1, 1.0)


def test_cpp_safe_control_demo_compiles_warning_free():
    import shutil
    import subprocess

    cxx = shutil.which("g++")
    if cxx is None:
        pytest.skip("no C++ compiler")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([cxx, "-std=c++20", "-Wall", "-Wextra", "-Wno-unused-parameter", "-fsyntax-only",
                        "-I", os.path.join(root, "include"), "-I", os.path.join(root, "oracle", "shim"),
                        os.path.join(root, "tests", "cpp", "safe_control_demo.cpp")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "warning" not in r.stderr, r.stderr[-3000:]
