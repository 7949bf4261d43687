"""-m gpu: the C++ adapter's row-band map update (b200::DeviceGridBatch::updateRows and b200::setMapTargets) gives,
after every step, the phi_k rows and extents that BatchedErgodicControl::setMapTargets of the whole maps gives, bit
for bit."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_cpp_map_update_matches_whole_maps(tmp_path):
    import __graft_entry__ as g
    from ergodic_exploration_b200 import capi

    if not os.path.exists(capi.LIB_PATH):
        g.build()
    exe = str(tmp_path / "map_update_demo")
    libdir = os.path.join(ROOT, "ergodic_exploration_b200")
    r = subprocess.run(["g++", "-std=c++20", "-O1", "-Wall", "-Wextra", "-Wno-unused-parameter",
                        "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle", "shim"),
                        os.path.join(ROOT, "tests", "cpp", "map_update_demo.cpp"), "-o", exe, "-L" + libdir,
                        "-lergodic_b200", "-Wl,-rpath," + libdir], capture_output=True, text=True)
    assert r.returncode == 0 and "warning" not in r.stderr, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout + r.stderr
    assert r.stdout.count("equal") == 4, r.stdout
