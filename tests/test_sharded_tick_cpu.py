"""CPU: the multi-GPU per-instance calls (eb_control_batch_dev_gather[_wait], eb_control_safe_batch_dev_gather[_wait])
refuse NULL handles without a device, and PeerGather's new methods are typed in the binding."""
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


def test_plain_gathers_refuse_null_handles(lib):
    from ergodic_exploration_b200 import capi

    x = np.zeros((2, 3))
    bounds = np.zeros((2, 4))
    for name in ("eb_control_batch_dev_gather", "eb_control_batch_dev_gather_wait"):
        fn = getattr(lib, name)
        assert fn(None, None, bounds.ctypes.data, x.ctypes.data, None, None) == capi.EB_ERR_INVALID_ARGUMENT
        assert name.encode() in lib.eb_last_error()


def test_safe_gathers_refuse_null_handles(lib):
    from ergodic_exploration_b200 import capi

    col = capi.EbCollision(0.2, 1.0, 0.05, 0.65)
    dwa = capi.EbDwa()
    x = np.zeros((2, 3))
    b = np.empty(2, dtype=np.int32)
    for name in ("eb_control_safe_batch_dev_gather", "eb_control_safe_batch_dev_gather_wait"):
        fn = getattr(lib, name)
        assert fn(None, None, None, C.byref(col), C.byref(dwa), 0.1, 1.0, None, x.ctypes.data, None, x.ctypes.data,
                  b.ctypes.data, None) == capi.EB_ERR_INVALID_ARGUMENT
        assert name.encode() in lib.eb_last_error()


def test_peer_gather_has_the_per_instance_steps():
    from ergodic_exploration_b200.sharding import PeerGather

    for name in ("control_batch", "control_batch_wait", "control_safe", "control_safe_wait"):
        assert callable(getattr(PeerGather, name))
