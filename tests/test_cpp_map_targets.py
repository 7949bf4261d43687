"""-m gpu: the C++ adapter's map-derived targets (BatchedErgodicControl::setMapTargets over GridMap-like maps, then
control(grids, x)) in a closed loop with a growing map, replayed on one oracle object per robot."""
import os
import subprocess

import numpy as np
import pytest

from helpers import MODEL_OMNI, assert_abs_rel_close, make_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def cell_values(xs, ys, robot, gen):
    """cell_value of tests/cpp/map_targets_demo.cpp"""
    i = np.arange(ys, dtype=np.int64)[:, None]
    j = np.arange(xs, dtype=np.int64)[None, :]
    return (((i * 31 + j * 17 + robot * 7 + gen * 13 + (i * j) % 5) % 102) - 1).astype(np.int8)


@pytest.mark.gpu
def test_cpp_map_targets_closed_loop_matches_oracle(tmp_path):
    import __graft_entry__ as g
    from ergodic_exploration_b200 import capi
    from oracle.pyoracle import Oracle
    from test_gpu_map_target import centre_phik

    if not os.path.exists(capi.LIB_PATH):
        g.build()
    exe = str(tmp_path / "map_targets_demo")
    libdir = os.path.join(ROOT, "ergodic_exploration_b200")
    r = subprocess.run(["g++", "-std=c++20", "-O1", "-Wall", "-Wextra", "-Wno-unused-parameter",
                        "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle", "shim"),
                        os.path.join(ROOT, "tests", "cpp", "map_targets_demo.cpp"), "-o", exe, "-L" + libdir,
                        "-lergodic_b200", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert r.returncode == 0 and "warning" not in r.stderr, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout + r.stderr
    recs = {}
    for line in r.stdout.splitlines():
        t = line.split()
        if len(t) > 2:
            recs.setdefault((t[0], int(t[1])), []).append(np.array([float(v) for v in t[2:]]))
    grown = False
    for i in range(3):
        o = make_oracle(MODEL_OMNI, batch_size=100, buffer_size=1000)
        last = None
        for step, (gr, x, u0, m) in enumerate(zip(recs[("grid", i)], recs[("x", i)], recs[("u0", i)],
                                                  recs[("metric", i)])):
            xs, ys, res, x0, y0, gen = int(gr[0]), int(gr[1]), gr[2], gr[3], gr[4], int(gr[5])
            if (xs, ys, gen) != last:
                cells = cell_values(xs, ys, i, gen)
                o.set_phik(centre_phik(Oracle.entropy_grid(cells), res, 10), xs * res, ys * res)
                grown |= last is not None
                last = (xs, ys, gen)
            o.add_state_memory(x)
            assert_abs_rel_close(u0, o.control((x0, x0 + xs * res, y0, y0 + ys * res), x), f"robot {i} step {step} u0")
            assert_abs_rel_close(m[0], o.last()["metric"], f"robot {i} step {step} metric")
    assert grown, "robot 1's map grew"
