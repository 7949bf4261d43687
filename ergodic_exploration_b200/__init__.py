"""ergodic_exploration_b200 -- B200-native (sm_100a) hot path of
bostoncleek/ergodic_exploration: the receding-horizon ergodic controller step
ErgodicControl::control() and the phi_k target-coefficient contraction.

The arithmetic lives in hand-written CUDA behind a C ABI
(include/ergodic_b200.h -> libergodic_b200.so).  This package is the thin
Python host mirror used by the tests and the benchmark; the C++ drop-in
adapter is include/ergodic_exploration_b200/.  No CPU fallback exists.
"""
from .capi import (EB_ERR_CUDA, EB_ERR_INVALID_ARGUMENT, EB_ERR_NO_DEVICE, EB_OK, MODEL_CART, MODEL_MECANUM, MODEL_OMNI,
                   MODEL_SIMPLE_CART, ErgodicB200Error)
from .collision import Collision, DynamicWindow, GridMap, GridMapBatch, integrate_twist, validate_control
from .controller import (Cart, ErgodicControl, Gaussian, GridBounds, MapTarget, Mecanum, Omni, PhikPlan, RungeKutta,
                         SimpleCart, Target, fp64_peak, l2_gather_peak)

__all__ = [
    "Cart", "Mecanum", "RungeKutta", "MapTarget", "l2_gather_peak", "MODEL_CART", "MODEL_MECANUM",
    "Collision", "DynamicWindow", "GridMap", "GridMapBatch", "integrate_twist", "validate_control", "ErgodicControl", "Gaussian", "GridBounds", "Omni", "PhikPlan", "SimpleCart", "Target", "fp64_peak",
    "ErgodicB200Error", "MODEL_OMNI", "MODEL_SIMPLE_CART", "EB_OK", "EB_ERR_CUDA",
    "EB_ERR_INVALID_ARGUMENT", "EB_ERR_NO_DEVICE",
]
