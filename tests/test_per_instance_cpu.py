"""CPU: the per-instance target entry points (eb_*_batch) validate their arguments without a device, and without a
device there is no controller to hold per-instance targets (no CPU fallback)."""
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


def test_null_and_invalid_arguments_need_no_device(lib):
    from ergodic_exploration_b200 import capi

    bad = capi.EB_ERR_INVALID_ARGUMENT
    counts = (C.c_int * 4)(1, 1, 1, 1)
    mu = (C.c_double * 8)()
    assert lib.eb_set_target_gaussians_batch(None, 1, counts, mu, mu) == bad
    assert b"eb_set_target_gaussians_batch" in lib.eb_last_error()
    assert lib.eb_set_phik_batch_dev(None, mu, mu) == bad
    assert lib.eb_get_phik_batch(None, mu, mu) == bad
    assert lib.eb_config_target_batch_dev(None, mu, None) == bad
    assert lib.eb_control_batch_dev(None, None, mu, None, mu, None) == bad
    assert lib.eb_control_batch_host(None, mu, mu, None, mu, None) == bad


def test_no_device_means_no_per_instance_controller(lib):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import ergodic_exploration_b200 as eb

    with pytest.raises(eb.ErgodicB200Error) as e:
        eb.ErgodicControl(eb.Omni(), 0.1, 5.0, 0.1, 1.0, 10, 1000, 100, np.eye(3), [-1] * 3, [1] * 3, batch=4)
    assert e.value.status == eb.EB_ERR_NO_DEVICE


def test_cpp_per_instance_demo_compiles_warning_free(tmp_path):
    import shutil
    import subprocess

    cxx = shutil.which("g++")
    if cxx is None:
        pytest.skip("no C++ compiler")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([cxx, "-std=c++20", "-Wall", "-Wextra", "-Wno-unused-parameter", "-fsyntax-only",
                        "-I", os.path.join(root, "include"), "-I", os.path.join(root, "oracle", "shim"),
                        os.path.join(root, "tests", "cpp", "per_instance_demo.cpp")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "warning" not in r.stderr, r.stderr[-3000:]
