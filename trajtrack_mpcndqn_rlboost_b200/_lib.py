"""ctypes binding of the product C-ABI (include/ttmpc.h).

The library is the sm_100a CUDA build ``libttmpc.so`` that lives next to this
file (built by ``make`` / ``__graft_entry__.build()``).  There is NO fallback:
if the library is missing, importing a compute entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TTMPC_LIB", os.path.join(_HERE, "libttmpc.so"))  # TTMPC_LIB: diagnostic builds


class TtmpcConfig(C.Structure):
    """struct ttmpc_config (include/ttmpc.h)."""
    _fields_ = [
        ("N_hor", C.c_int), ("nu", C.c_int), ("ns", C.c_int), ("nq", C.c_int),
        ("Nother", C.c_int), ("Nstcobs", C.c_int), ("nstcobs", C.c_int),
        ("Ndynobs", C.c_int), ("ndynobs", C.c_int), ("_pad0", C.c_int),
        ("ts", C.c_double), ("vehicle_width", C.c_double), ("social_margin", C.c_double),
        ("lin_vel_min", C.c_double), ("lin_vel_max", C.c_double), ("ang_vel_max", C.c_double),
        ("lin_acc_min", C.c_double), ("lin_acc_max", C.c_double), ("ang_acc_max", C.c_double),
        ("tolerance", C.c_double), ("initial_tolerance", C.c_double),
        ("delta_tolerance", C.c_double), ("initial_penalty", C.c_double),
        ("penalty_update_factor", C.c_double), ("inner_tolerance_update_factor", C.c_double),
        ("sufficient_decrease_coeff", C.c_double),
        ("lbfgs_memory", C.c_int), ("max_inner_iterations", C.c_int),
        ("max_outer_iterations", C.c_int), ("max_duration_ms", C.c_int),
    ]


class TtmpcResult(C.Structure):
    """struct ttmpc_result: raw addresses (host or device, depending on the call)."""
    _fields_ = [
        ("u", C.c_void_p), ("cost", C.c_void_p), ("exit_status", C.c_void_p),
        ("outer_iters", C.c_void_p), ("inner_iters", C.c_void_p), ("last_fpr", C.c_void_p),
        ("f1_infeas", C.c_void_p), ("f2_norm", C.c_void_p), ("penalty", C.c_void_p),
        ("y", C.c_void_p), ("pred_states", C.c_void_p), ("evals", C.c_void_p),
    ]


class TtdqnLayout(C.Structure):
    _fields_ = [
        ("num_segments", C.c_int), ("max_poly", C.c_int), ("max_vert", C.c_int),
        ("n_internal", C.c_int), ("use_memory", C.c_int), ("_pad", C.c_int),
        ("ray_length", C.c_double), ("max_distance", C.c_double),
    ]


class TtdqnQnet(C.Structure):
    _fields_ = [
        ("n_in", C.c_int), ("n_h1", C.c_int), ("n_h2", C.c_int), ("n_out", C.c_int),
        ("w0", C.c_void_p), ("b0", C.c_void_p), ("w1", C.c_void_p), ("b1", C.c_void_p),
        ("w2", C.c_void_p), ("b2", C.c_void_p),
    ]


class TtdqnMoving(C.Structure):
    """struct ttdqn_moving: moving solid rings of ttdqn_observe_act_moving_device (device addresses)."""
    _fields_ = [
        ("n_live", C.c_int), ("max_pv", C.c_int), ("shape_shared", C.c_int), ("_pad", C.c_int),
        ("centre", C.c_void_p), ("shape_xy", C.c_void_p), ("shape_nv", C.c_void_p),
    ]


FLEET_WARM_START, FLEET_SKIP_STOPPED = 1, 2  # ttmpc_fleet.options bits


class TtmpcFleet(C.Structure):
    """struct ttmpc_fleet: raw addresses (device for the product calls, host for the oracle)."""
    _fields_ = [
        ("n", C.c_int), ("ref_stride", C.c_int),
        ("state", C.c_void_p), ("goal", C.c_void_p), ("last_u", C.c_void_p),
        ("idx_ref", C.c_void_p), ("status", C.c_void_p), ("ref_traj", C.c_void_p),
        ("ref_len", C.c_void_p), ("stc", C.c_void_p),
        ("stc_shared", C.c_int), ("n_dyn_live", C.c_int), ("action_steps", C.c_int), ("options", C.c_int),
        ("other", C.c_void_p), ("dyn", C.c_void_p), ("dyn_cur", C.c_void_p),
        ("dyn_last", C.c_void_p), ("dyn_disp", C.c_void_p),
        ("dyn_size", C.c_double), ("tuning", C.c_double * 10),
        ("base_speed", C.c_double), ("low_speed", C.c_double),
        ("stc_weight", C.c_double), ("dyn_weight", C.c_double),
        ("hint", C.c_void_p), ("use_hint", C.c_void_p),
        ("sw_state", C.c_void_p), ("sw_poly_xy", C.c_void_p), ("sw_poly_nv", C.c_void_p),
        ("sw_max_poly", C.c_int), ("sw_max_pv", C.c_int), ("sw_poly_shared", C.c_int), ("sw_detach_steps", C.c_int),
        ("sw_switch_distance", C.c_double), ("sw_detach_distance", C.c_double), ("sw_dyn_radius", C.c_double),
    ]


class TtmpcFleetTasks(C.Structure):
    """struct ttmpc_fleet_tasks: per-robot task queues of ttmpc_fleet_step_tasks_device (device addresses)."""
    _fields_ = [
        ("max_tasks", C.c_int), ("max_nodes", C.c_int),
        ("count", C.c_void_p), ("next", C.c_void_p), ("goal", C.c_void_p), ("path_xy", C.c_void_p),
        ("path_n", C.c_void_p), ("path_out", C.c_void_p), ("path_out_n", C.c_void_p),
    ]


class TtmpcFleetMonitor(C.Structure):
    """struct ttmpc_fleet_monitor: obstacle-contact and tracking monitor of ttmpc_fleet_monitor_device
    (device addresses)."""
    _fields_ = [
        ("poly_xy", C.c_void_p), ("poly_nv", C.c_void_p),
        ("max_poly", C.c_int), ("max_pv", C.c_int), ("poly_shared", C.c_int), ("stop_on_contact", C.c_int),
        ("robot_radius", C.c_double), ("moving_radius", C.c_double),
        ("step", C.c_int), ("_pad", C.c_int),
        ("prev_xy", C.c_void_p), ("clearance", C.c_void_p), ("min_clearance", C.c_void_p),
        ("contact_steps", C.c_void_p), ("first_contact", C.c_void_p), ("deviation_max", C.c_void_p),
        ("deviation_sum", C.c_void_p), ("moved_steps", C.c_void_p),
    ]


class TtmpcFleetWorld(C.Structure):
    """struct ttmpc_fleet_world: shared obstacle map and its grid for ttmpc_fleet_world_select_device
    (device addresses)."""
    _fields_ = [
        ("M", C.c_int), ("max_pv", C.c_int),
        ("poly_xy", C.c_void_p), ("poly_nv", C.c_void_p), ("rows", C.c_void_p), ("bbox", C.c_void_p),
        ("reach", C.c_double), ("origin_x", C.c_double), ("origin_y", C.c_double), ("cell", C.c_double),
        ("nx", C.c_int), ("ny", C.c_int),
        ("cell_start", C.c_void_p), ("cell_items", C.c_void_p),
    ]


# every symbol include/ttmpc.h declares, with its signature
_VP, _I, _D = C.c_void_p, C.c_int, C.c_double
_CFG, _RES = C.POINTER(TtmpcConfig), C.POINTER(TtmpcResult)
_LAY, _QN, _MOV = C.POINTER(TtdqnLayout), C.POINTER(TtdqnQnet), C.POINTER(TtdqnMoving)
_FLT = C.POINTER(TtmpcFleet)
_TSK = C.POINTER(TtmpcFleetTasks)
_MON = C.POINTER(TtmpcFleetMonitor)
_WLD = C.POINTER(TtmpcFleetWorld)
SYMBOLS = {
    "ttmpc_default_config": (None, [_CFG]),
    "ttmpc_num_params": (_I, [_CFG]),
    "ttmpc_num_decision": (_I, [_CFG]),
    "ttmpc_num_alm": (_I, [_CFG]),
    "ttmpc_num_penalty": (_I, [_CFG]),
    "ttmpc_last_error": (C.c_char_p, []),
    "ttmpc_exit_status_name": (C.c_char_p, [_I]),
    "ttmpc_version": (_I, []),
    "ttmpc_set_device": (_I, [_I]),
    "ttmpc_get_device": (_I, [C.POINTER(C.c_int)]),
    "ttmpc_solve_batch_device": (_I, [_CFG, _I, _VP, _I, _I, _VP, _RES, _VP]),
    "ttmpc_solve_batch_host": (_I, [_CFG, _I, _VP, _I, _I, _VP, _RES]),
    "ttmpc_eval_batch_device": (_I, [_CFG, _I] + [_VP] * 10),
    "ttmpc_eval_batch_host": (_I, [_CFG, _I] + [_VP] * 9),
    "ttmpc_fleet_pack_device": (_I, [_CFG, _FLT, _VP, _VP]),
    "ttmpc_fleet_advance_device": (_I, [_CFG, _FLT, _VP, _VP, _VP]),
    "ttmpc_fleet_step_device": (_I, [_CFG, _FLT, _VP, _I, _RES, _VP]),
    "ttmpc_fleet_step_tasks_device": (_I, [_CFG, _FLT, _TSK, _VP, _I, _RES, _VP]),
    "ttmpc_fleet_monitor_device": (_I, [_CFG, _FLT, _MON, _VP]),
    "ttmpc_fleet_world_select_device": (_I, [_CFG, _FLT, _WLD, _VP, _VP, _VP, _VP]),
    "ttmpc_read_stats": (_I, [C.POINTER(C.c_ulonglong), _I]),
    "ttmpc_launch_info": (_I, [_CFG, _I] + [C.POINTER(C.c_int)] * 5),
    "ttmpc_measure_fp64_peak": (_I, [C.POINTER(_D), _VP]),
    "ttdqn_last_error": (C.c_char_p, []),
    "ttdqn_default_layout": (None, [_LAY]),
    "ttdqn_observe_act_device": (_I, [_LAY, _QN, _I] + [_VP] * 12 + [_VP]),
    "ttdqn_observe_act_moving_device": (_I, [_LAY, _QN, _I] + [_VP] * 5 + [_MOV] + [_VP] * 7 + [_VP]),
    "ttdqn_observe_act_host": (_I, [_LAY, _QN, _I] + [_VP] * 12),
    "ttdqn_internal_obs_device": (_I, [_I, _I, _I, _D, _D, _VP, _VP, _VP, _VP, _VP, _VP]),
    "ttdqn_rl_ref_device": (_I, [_I, _I, _D, _D, _VP, _VP, _VP, _VP]),
}

_lib = None


class TtmpcError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load libttmpc.so; raise loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TtmpcError(
            f"{LIB_PATH} not found: the CUDA extension is not built. Run `make` at the repo "
            "root (or __graft_entry__.build()). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        lib = load()
        msg = lib.ttmpc_last_error().decode()
        raise TtmpcError(f"{what} failed (code {rc}): {msg}")


def default_config() -> TtmpcConfig:
    cfg = TtmpcConfig()
    load().ttmpc_default_config(C.byref(cfg))
    return cfg
