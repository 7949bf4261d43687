"""ctypes binding of the C ABI declared in include/ergodic_b200.h.

The shared library is built in-tree (ergodic_exploration_b200/libergodic_b200.so)
by ``__graft_entry__.build()`` / ``make -C ergodic_exploration_b200/csrc``.
There is no CPU fallback: if the library is missing, loading fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("EB_LIB_PATH") or os.path.join(_HERE, "libergodic_b200.so")  # override: debug builds

EB_OK = 0
EB_ERR_INVALID_ARGUMENT = 1
EB_ERR_OUT_OF_RANGE = 2
EB_ERR_CUDA = 3
EB_ERR_NO_DEVICE = 4
EB_ERR_UNSUPPORTED = 5

MODEL_SIMPLE_CART = 0
MODEL_OMNI = 1
MODEL_CART = 2
MODEL_MECANUM = 3


class EbConfig(C.Structure):
    """struct eb_config (include/ergodic_b200.h)"""

    _fields_ = [
        ("model", C.c_int),
        ("batch", C.c_int),
        ("device", C.c_int),
        ("dt", C.c_double),
        ("horizon", C.c_double),
        ("resolution", C.c_double),
        ("expl_weight", C.c_double),
        ("num_basis", C.c_uint),
        ("buffer_size", C.c_uint),
        ("batch_size", C.c_uint),
        ("Rinv", C.c_double * 9),
        ("umin", C.c_double * 3),
        ("umax", C.c_double * 3),
        ("barrier_weight", C.c_double),
        ("barrier_eps", C.c_double),
        ("seed", C.c_ulonglong),
    ]


class EbCollision(C.Structure):
    """struct eb_collision (include/ergodic_b200.h)"""

    _fields_ = [("boundary_radius", C.c_double), ("search_radius", C.c_double),
                ("obstacle_threshold", C.c_double), ("occupied_threshold", C.c_double)]


class EbDwa(C.Structure):
    """struct eb_dwa (include/ergodic_b200.h)"""

    _fields_ = [(n, C.c_double) for n in ("dt", "horizon", "acc_dt", "acc_lim_x", "acc_lim_y", "acc_lim_th",
                                          "max_vel_x", "min_vel_x", "max_vel_y", "min_vel_y", "max_rot_vel",
                                          "min_rot_vel")] + [(n, C.c_uint) for n in ("vx_samples", "vy_samples",
                                                                                     "vth_samples")]


class ErgodicB200Error(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"[eb_status {status}] {message}")
        self.status = status
        self.message = message


_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_vp = C.c_void_p

# every symbol include/ergodic_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "eb_config_defaults": (None, [C.POINTER(EbConfig), C.c_int]),
    "eb_abi_version": (C.c_int, []),
    "eb_last_error": (C.c_char_p, []),
    "eb_device_count": (C.c_int, []),
    "eb_create": (C.c_int, [C.POINTER(EbConfig), C.POINTER(_vp)]),
    "eb_clone": (C.c_int, [_vp, C.POINTER(_vp)]),
    "eb_destroy": (None, [_vp]),
    "eb_set_stream": (C.c_int, [_vp, _vp]),
    "eb_steps": (C.c_int, [_vp]),
    "eb_num_coeff": (C.c_int, [_vp]),
    "eb_batch": (C.c_int, [_vp]),
    "eb_time_step": (C.c_double, [_vp]),
    "eb_memory_size": (C.c_longlong, [_vp]),
    "eb_set_target_gaussians": (C.c_int, [_vp, C.c_int, _vp, _vp]),
    "eb_config_target": (C.c_int, [_vp, C.c_double, C.c_double, C.c_double, C.c_double, _ip]),
    "eb_set_phik": (C.c_int, [_vp, _vp, C.c_double, C.c_double]),
    "eb_get_phik": (C.c_int, [_vp, _vp, _dp, _dp]),
    "eb_reserve_state_memory": (C.c_int, [_vp, C.c_longlong]),
    "eb_add_state_memory_host": (C.c_int, [_vp, _vp]),
    "eb_add_state_memory_dev": (C.c_int, [_vp, _vp]),
    "eb_control_host": (C.c_int, [_vp, C.c_double, C.c_double, C.c_double, C.c_double, _vp, _vp, _vp, _vp]),
    "eb_control_dev": (C.c_int, [_vp, C.c_double, C.c_double, C.c_double, C.c_double, _vp, _vp, _vp, _vp]),
    "eb_check_status": (C.c_int, [_vp]),
    "eb_opt_traj_host": (C.c_int, [_vp, _vp]),
    "eb_opt_traj_dev": (C.c_int, [_vp, _vp]),
    "eb_get_ut": (C.c_int, [_vp, _vp]),
    "eb_set_ut": (C.c_int, [_vp, _vp]),
    "eb_get_ck": (C.c_int, [_vp, _vp]),
    "eb_get_last_mem_idx": (C.c_int, [_vp, _vp, _ip]),
    "eb_ut_dev": (_vp, [_vp]),
    "eb_ck_dev": (_vp, [_vp]),
    "eb_set_keep_ck": (C.c_int, [_vp, C.c_int]),
    "eb_launch_count": (C.c_longlong, [_vp]),
    "eb_phik_plan_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int,
                                      C.POINTER(_vp)]),
    "eb_phik_plan_create_rows": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double,
                                           C.c_double, C.c_int, C.POINTER(_vp)]),
    "eb_phik_plan_destroy": (None, [_vp]),
    "eb_phik_plan_set_stream": (C.c_int, [_vp, _vp]),
    "eb_phik_plan_set_algo": (C.c_int, [_vp, C.c_int]),
    "eb_phik_plan_fold": (C.c_int, [_vp, _ip, _dp]),
    "eb_phik_execute_dev": (C.c_int, [_vp, _vp, _vp, _vp]),
    "eb_phik_execute_host": (C.c_int, [_vp, _vp, _vp, _vp]),
    "eb_phik_execute_raw_dev": (C.c_int, [_vp, _vp, _vp]),
    "eb_phik_from_grid_host": (C.c_int, [C.c_int, _vp, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double,
                                         C.c_int, _vp, _vp]),
    "eb_phik_launch_count": (C.c_longlong, [_vp]),
    "eb_basis_traj_coeff_host": (C.c_int, [C.c_int, C.c_double, C.c_double, C.c_int, _vp, C.c_int, C.c_int, _vp]),
    "eb_basis_grad_host": (C.c_int, [C.c_int, C.c_double, C.c_double, C.c_int, _vp, _vp]),
    "eb_basis_spatial_coeff_host": (C.c_int, [C.c_int, C.c_double, C.c_double, C.c_int, _vp, _vp, C.c_longlong, _vp]),
    "eb_target_fill_host": (C.c_int, [C.c_int, C.c_int, _vp, _vp, _vp, _vp, C.c_longlong, _vp]),
    "eb_fp64_peak": (C.c_int, [C.c_int, _dp, _dp]),
    "eb_integrate_twist_dev": (C.c_int, [C.c_int, _vp, _vp, C.c_double, C.c_int, _vp, _vp]),
    "eb_dwa_control_twist_host": (C.c_int, [_vp, C.POINTER(EbCollision), C.POINTER(EbDwa), _vp, _vp, _vp, C.c_int, _vp, _vp, _vp]),
    "eb_dwa_control_twist_dev": (C.c_int, [_vp, C.POINTER(EbCollision), C.POINTER(EbDwa), _vp, _vp, _vp, C.c_int, _vp, _vp, _vp]),
    "eb_dwa_control_traj_host": (C.c_int, [_vp, C.POINTER(EbCollision), C.POINTER(EbDwa), _vp, _vp, _vp, C.c_int, C.c_int,
                                           C.c_double, C.c_int, _vp, _vp, _vp]),
    "eb_dwa_control_traj_dev": (C.c_int, [_vp, C.POINTER(EbCollision), C.POINTER(EbDwa), _vp, _vp, _vp, C.c_int, C.c_int,
                                          C.c_double, C.c_int, _vp, _vp, _vp]),
    "eb_peer_blob_bytes": (C.c_int, []),
    "eb_peer_group_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_longlong, C.POINTER(_vp)]),
    "eb_peer_group_export": (C.c_int, [_vp, _vp]),
    "eb_peer_group_connect": (C.c_int, [_vp, _vp]),
    "eb_peer_group_destroy": (None, [_vp]),
    "eb_control_dev_gather": (C.c_int, [_vp, _vp, C.c_double, C.c_double, C.c_double, C.c_double, _vp, _vp, _vp]),
    "eb_peer_group_wait": (C.c_int, [_vp, _vp, C.c_ulonglong]),
    "eb_control_dev_gather_wait": (C.c_int, [_vp, _vp, C.c_double, C.c_double, C.c_double, C.c_double, _vp, _vp, _vp]),
    "eb_peer_gathered_dev": (_vp, [_vp, C.c_ulonglong]),
    "eb_peer_group_steps": (C.c_ulonglong, [_vp]),
    "eb_peer_group_fused": (C.c_int, [_vp, C.c_int]),
    "eb_gather_fuse_min_batch": (C.c_int, []),
    "eb_phik_plan_create_ex": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double,
                                         C.c_double, C.c_int, C.c_double, C.c_double, C.POINTER(_vp)]),
    "eb_phik_peer_blob_bytes": (C.c_int, []),
    "eb_phik_peer_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    "eb_phik_peer_export": (C.c_int, [_vp, _vp]),
    "eb_phik_peer_connect": (C.c_int, [_vp, _vp]),
    "eb_phik_peer_destroy": (None, [_vp]),
    "eb_phik_execute_allreduce_dev": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "eb_map_target_create": (C.c_int, [C.c_int, C.c_uint, C.c_uint, C.c_double, C.c_int, C.POINTER(_vp)]),
    "eb_map_target_destroy": (None, [_vp]),
    "eb_map_target_set_stream": (C.c_int, [_vp, _vp]),
    "eb_map_target_execute_dev": (C.c_int, [_vp, _vp, _vp, _vp]),
    "eb_map_target_execute_host": (C.c_int, [_vp, _vp, _vp, _vp]),
    "eb_map_target_density_dev": (_vp, [_vp]),
    "eb_map_target_extent": (C.c_int, [_vp, _dp, _dp]),
    "eb_map_target_launch_count": (C.c_longlong, [_vp]),
    "eb_set_phik_dev": (C.c_int, [_vp, _vp, C.c_double, C.c_double]),
    "eb_set_target_gaussians_batch": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp]),
    "eb_set_phik_batch_dev": (C.c_int, [_vp, _vp, _vp]),
    "eb_get_phik_batch": (C.c_int, [_vp, _vp, _vp]),
    "eb_config_target_batch_dev": (C.c_int, [_vp, _vp, _vp]),
    "eb_control_batch_dev": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "eb_control_batch_host": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "eb_set_map_targets_batch_dev": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "eb_set_map_targets_batch_host": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "eb_set_map_targets_from_grid_batch": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "eb_model_controls": (C.c_int, [C.c_int]),
    "eb_rk4_solve_host": (C.c_int, [C.c_int, C.c_int, _vp, C.c_double, C.c_double, _vp, _vp, C.c_int, C.c_int, _vp]),
    "eb_rk4_solve_dev": (C.c_int, [C.c_int, C.c_int, _vp, C.c_double, C.c_double, _vp, _vp, C.c_int, C.c_int, _vp, _vp, _vp]),
    "eb_model_eval_host": (C.c_int, [C.c_int, C.c_int, _vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp]),
    "eb_l2_gather_peak": (C.c_int, [C.c_int, _dp]),
    "eb_grid_create": (C.c_int, [C.c_int, _vp, C.c_uint, C.c_uint, C.c_double, C.c_double, C.c_double, C.POINTER(_vp)]),
    "eb_grid_update": (C.c_int, [_vp, _vp]),
    "eb_grid_destroy": (None, [_vp]),
    "eb_grid_set_stream": (C.c_int, [_vp, _vp]),
    "eb_grid_launch_count": (C.c_longlong, [_vp]),
    "eb_grid_set_dilation": (C.c_int, [_vp, C.c_int]),
    "eb_collision_check_host": (C.c_int, [_vp, C.POINTER(EbCollision), _vp, C.c_int, _vp]),
    "eb_collision_check_dev": (C.c_int, [_vp, C.POINTER(EbCollision), _vp, C.c_int, _vp]),
    "eb_validate_control_host": (C.c_int, [_vp, C.POINTER(EbCollision), _vp, _vp, C.c_int, C.c_double, C.c_double, _vp]),
    "eb_validate_control_dev": (C.c_int, [_vp, C.POINTER(EbCollision), _vp, _vp, C.c_int, C.c_double, C.c_double, _vp]),
    "eb_grid_batch_create": (C.c_int, [C.c_int, C.c_int, C.POINTER(_vp)]),
    "eb_grid_batch_destroy": (None, [_vp]),
    "eb_grid_batch_set_stream": (C.c_int, [_vp, _vp]),
    "eb_grid_batch_launch_count": (C.c_longlong, [_vp]),
    "eb_grid_batch_set_maps_dev": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "eb_grid_batch_set_maps_host": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "eb_grid_batch_set_rows_dev": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "eb_grid_batch_set_rows_host": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "eb_grid_batch_get_map_host": (C.c_int, [_vp, C.c_int, _vp]),
    "eb_collision_check_batch_host": (C.c_int, [_vp, C.POINTER(EbCollision), _vp, C.c_int, _vp]),
    "eb_collision_check_batch_dev": (C.c_int, [_vp, C.POINTER(EbCollision), _vp, C.c_int, _vp]),
    "eb_validate_control_batch_host": (C.c_int, [_vp, C.POINTER(EbCollision), _vp, _vp, C.c_int, C.c_double, C.c_double,
                                                 _vp]),
    "eb_validate_control_batch_dev": (C.c_int, [_vp, C.POINTER(EbCollision), _vp, _vp, C.c_int, C.c_double, C.c_double,
                                                _vp]),
    "eb_dwa_control_twist_batch_host": (C.c_int, [_vp, C.POINTER(EbCollision), C.POINTER(EbDwa), _vp, _vp, _vp, _vp, _vp,
                                                  _vp]),
    "eb_dwa_control_twist_batch_dev": (C.c_int, [_vp, C.POINTER(EbCollision), C.POINTER(EbDwa), _vp, _vp, _vp, _vp, _vp,
                                                 _vp]),
    "eb_dwa_control_traj_batch_host": (C.c_int, [_vp, C.POINTER(EbCollision), C.POINTER(EbDwa), _vp, _vp, _vp, C.c_int,
                                                 C.c_int, C.c_double, _vp, _vp, _vp]),
    "eb_dwa_control_traj_batch_dev": (C.c_int, [_vp, C.POINTER(EbCollision), C.POINTER(EbDwa), _vp, _vp, _vp, C.c_int,
                                                C.c_int, C.c_double, _vp, _vp, _vp]),
    "eb_control_safe_batch_dev": (C.c_int, [_vp, _vp, C.POINTER(EbCollision), C.POINTER(EbDwa), C.c_double, C.c_double,
                                            _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "eb_control_safe_batch_host": (C.c_int, [_vp, _vp, C.POINTER(EbCollision), C.POINTER(EbDwa), C.c_double, C.c_double,
                                             _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "eb_control_batch_dev_gather": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "eb_control_batch_dev_gather_wait": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "eb_control_safe_batch_dev_gather": (C.c_int, [_vp, _vp, _vp, C.POINTER(EbCollision), C.POINTER(EbDwa), C.c_double,
                                                   C.c_double, _vp, _vp, _vp, _vp, _vp, _vp]),
    "eb_control_safe_batch_dev_gather_wait": (C.c_int, [_vp, _vp, _vp, C.POINTER(EbCollision), C.POINTER(EbDwa),
                                                        C.c_double, C.c_double, _vp, _vp, _vp, _vp, _vp, _vp]),
}

_lib = None


def load():
    """Load libergodic_b200.so and type every entry point.  Raises if the
    extension has not been built -- the product has no other code path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  ergodic_exploration_b200 has no CPU fallback."
            )
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(status):
    if status != EB_OK:
        raise ErgodicB200Error(status, load().eb_last_error().decode(errors="replace"))
