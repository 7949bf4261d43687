"""-m gpu: the C++ adapter's per-instance face (BatchedErgodicControl::setTargets and control over one map per
robot) in a closed loop, replayed on one oracle object per robot."""
import os
import subprocess

import numpy as np
import pytest

from helpers import MODEL_OMNI, assert_abs_rel_close, make_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TARGETS = [
    ([[2.5, 2.5], [8.5, 2.5]], [[1.5, 1.5], [1.5, 1.5]]),
    ([[0.0, 5.0]], [[2.0, 1.0]]),
    ([[6.0, 1.0], [12.0, 4.0], [9.0, 0.0]], [[1.0, 1.0], [1.5, 0.8], [1.2, 1.2]]),
]


@pytest.mark.gpu
def test_cpp_per_instance_closed_loop_matches_oracle(tmp_path):
    import __graft_entry__ as g
    from ergodic_exploration_b200 import capi

    if not os.path.exists(capi.LIB_PATH):
        g.build()
    exe = str(tmp_path / "per_instance_demo")
    libdir = os.path.join(ROOT, "ergodic_exploration_b200")
    r = subprocess.run(["g++", "-std=c++20", "-O1", "-Wall", "-Wextra", "-Wno-unused-parameter",
                        "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle", "shim"),
                        os.path.join(ROOT, "tests", "cpp", "per_instance_demo.cpp"), "-o", exe, "-L" + libdir,
                        "-lergodic_b200", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert r.returncode == 0 and "warning" not in r.stderr, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout + r.stderr
    recs = {}
    for line in r.stdout.splitlines():
        t = line.split()
        if len(t) > 2:
            recs.setdefault((t[0], int(t[1])), []).append(np.array([float(v) for v in t[2:]]))
    for i, (mu, sg) in enumerate(TARGETS):
        o = make_oracle(MODEL_OMNI, batch_size=100, buffer_size=1000, mu=np.array(mu), sigma=np.array(sg))
        for step, (b, x, u0, m) in enumerate(zip(recs[("bounds", i)], recs[("x", i)], recs[("u0", i)],
                                                recs[("metric", i)])):
            o.add_state_memory(x)
            assert_abs_rel_close(u0, o.control(tuple(b), x), f"robot {i} step {step} u0")
            assert_abs_rel_close(m[0], o.last()["metric"], f"robot {i} step {step} metric")
