"""-m gpu: the C++ adapter's per-instance maps (DeviceGridBatch next to BatchedErgodicControl::setMapTargets, then
DynamicWindow::controlBatch and validate_control on each robot's own map) in a closed loop with a growing map,
replayed per robot on the oracle with that robot's map at that tick."""
import os
import subprocess

import numpy as np
import pytest

from test_dwa_cpu import COL, DWA_OMNI

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def cell_values(xs, ys, robot, gen):
    """cell_value of tests/cpp/grid_batch_demo.cpp"""
    i = np.arange(ys, dtype=np.int64)[:, None]
    j = np.arange(xs, dtype=np.int64)[None, :]
    h = i * 31 + j * 17 + robot * 7 + gen * 13 + (i * j) % 5
    return np.where(h % 41 == 0, 100, np.where(h % 23 == 0, -1, 0)).astype(np.int8)


@pytest.mark.gpu
def test_cpp_grid_batch_closed_loop_matches_oracle(tmp_path):
    import __graft_entry__ as g
    from ergodic_exploration_b200 import capi
    from oracle.pyoracle import Oracle

    if not os.path.exists(capi.LIB_PATH):
        g.build()
    exe = str(tmp_path / "grid_batch_demo")
    libdir = os.path.join(ROOT, "ergodic_exploration_b200")
    r = subprocess.run(["g++", "-std=c++20", "-O1", "-Wall", "-Wextra", "-Wno-unused-parameter",
                        "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle", "shim"),
                        os.path.join(ROOT, "tests", "cpp", "grid_batch_demo.cpp"), "-o", exe, "-L" + libdir,
                        "-lergodic_b200", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert r.returncode == 0 and "warning" not in r.stderr, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout + r.stderr
    recs = {}
    for line in r.stdout.splitlines():
        t = line.split()
        if len(t) > 2:
            recs.setdefault((t[0], int(t[1])), []).append(np.array([float(v) for v in t[2:]]))
    grown, found_any = False, 0
    for i in range(3):
        last = None
        for step, (gr, x, vb, u0, xt, dw, va) in enumerate(zip(*(recs[(k, i)] for k in (
                "grid", "x", "vb", "u0", "xt", "dwa", "valid")))):
            xs, ys, res, x0, y0, gen = int(gr[0]), int(gr[1]), gr[2], gr[3], gr[4], int(gr[5])
            grown |= last is not None and (xs, ys, gen) != last
            last = (xs, ys, gen)
            cells = cell_values(xs, ys, i, gen)
            fo, uo, _ = Oracle.dwa_control(cells, res, x0, y0, COL, DWA_OMNI, (3, 8, 5), x[None], vb[None],
                                           xt_ref=xt.reshape(-1, 3), dt_ref=0.1)
            assert int(dw[0]) == fo[0], f"robot {i} step {step} found"
            np.testing.assert_array_equal(dw[1:], uo[0], err_msg=f"robot {i} step {step} u_opt")
            vo = Oracle.validate_control(cells, res, x0, y0, COL, x[None], u0[None], 0.1, 1.0)
            assert int(va[0]) == vo[0], f"robot {i} step {step} validate"
            found_any += fo[0]
    assert grown, "robot 1's map grew"
    assert found_any > 0
