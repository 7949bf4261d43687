"""-m gpu: the C++ adapter's safe tick (b200::controlSafe next to BatchedErgodicControl::setMapTargets and
DeviceGridBatch::update) in a closed loop with a growing map, replayed through the composed Python calls --
control(None, x), validate_control, optTraj() and DynamicWindow.control on the grid batch -- with identical twists and
branches."""
import os
import subprocess

import numpy as np
import pytest

from test_cpp_grid_batch import cell_values
from test_dwa_cpu import COL, DWA_OMNI

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_cpp_safe_control_closed_loop_matches_composed_calls(tmp_path):
    import __graft_entry__ as g
    import ergodic_exploration_b200 as eb
    from ergodic_exploration_b200 import capi

    if not os.path.exists(capi.LIB_PATH):
        g.build()
    exe = str(tmp_path / "safe_control_demo")
    libdir = os.path.join(ROOT, "ergodic_exploration_b200")
    r = subprocess.run(["g++", "-std=c++20", "-O1", "-Wall", "-Wextra", "-Wno-unused-parameter",
                        "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle", "shim"),
                        os.path.join(ROOT, "tests", "cpp", "safe_control_demo.cpp"), "-o", exe, "-L" + libdir,
                        "-lergodic_b200", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert r.returncode == 0 and "warning" not in r.stderr, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout + r.stderr
    recs = {}
    for line in r.stdout.splitlines():
        t = line.split()
        if len(t) > 2:
            recs.setdefault(t[0], {}).setdefault(int(t[1]), []).append(np.array([float(v) for v in t[2:]]))
    B = 3
    ticks = len(recs["u"][0])
    R = np.diag([1.0, 1.0, 2.0])
    ctl = eb.ErgodicControl(eb.Omni(), 0.1, 5.0, 0.1, 1.0, 10, 1000, 100, R, [-1.0, -1.0, -2.0], [1.0, 1.0, 2.0],
                            batch=B)
    gb = eb.GridMapBatch(B)
    col = eb.Collision(*COL)
    dwa = eb.DynamicWindow(col, *DWA_OMNI, 3, 8, 5)
    last, grown, branches = [None] * B, False, set()
    for step in range(ticks):
        geo = [recs["grid"][i][step] for i in range(B)]
        upd = np.array([last[i] != (int(gr[0]), int(gr[1]), int(gr[5])) for i, gr in enumerate(geo)])
        grown |= step > 0 and bool(upd.any())
        cells = [cell_values(int(gr[0]), int(gr[1]), i, int(gr[5])) for i, gr in enumerate(geo)]
        res, org = [gr[2] for gr in geo], [(gr[3], gr[4]) for gr in geo]
        ctl.setMapTargets(cells, res, org, upd)
        gb.set(cells, res, org, upd)
        last = [(int(gr[0]), int(gr[1]), int(gr[5])) for gr in geo]
        x = np.array([recs["x"][i][step] for i in range(B)])
        vb = np.array([recs["vb"][i][step] for i in range(B)])
        ctl.addStateMemory(x)
        u0 = ctl.control(None, x)
        ok = eb.validate_control(col, gb, x, u0, 0.1, 1.0)
        found, ud = dwa.control(gb, x, vb, xt_ref=ctl.optTraj(), dt_ref=0.1)
        for i in range(B):
            want_b = 0 if ok[i] else (1 if found[i] else 2)
            want_u = u0[i] if ok[i] else (ud[i] if found[i] else np.zeros(3))
            assert int(recs["branch"][i][step][0]) == want_b, f"robot {i} tick {step} branch"
            np.testing.assert_array_equal(recs["u"][i][step], want_u, err_msg=f"robot {i} tick {step} u")
            branches.add(want_b)
    assert grown, "robot 1's map grew"
    assert len(branches) >= 2, branches
