"""ctypes binding of libmpcb200.so (C ABI declared in include/mpcb200.h).

There is no fallback: if the shared library is missing or a CUDA call fails, an exception is raised.
"""
import ctypes as C
import os

from . import _build

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)
c_u64_p = C.POINTER(C.c_ulonglong)


class MpcbError(RuntimeError):
    pass


class Params(C.Structure):
    """struct mpcb_params (include/mpcb200.h); mirrors TrajectoryTracker.__init__, trajectory_tracking.py:12-47."""
    _fields_ = [
        ("dt", C.c_double), ("N", C.c_int),
        ("u_min", C.c_double * 2), ("u_max", C.c_double * 2),
        ("vehicle_radius", C.c_double),
        ("w_d", C.c_double), ("w_o", C.c_double), ("w_v", C.c_double), ("w_u1", C.c_double), ("w_u2", C.c_double),
        ("obstacle_safety_distance", C.c_double), ("max_time_2_obs", C.c_double), ("wheelbase", C.c_double),
        ("lane_width", C.c_double), ("safe_lane_margin", C.c_double),
        ("brake_lookahead", C.c_double), ("brake_guess", C.c_double),
        ("max_rounds", C.c_int), ("max_segments", C.c_int), ("segment_iters", C.c_int),
        ("rho_lo", C.c_double), ("rho_hi", C.c_double), ("rho_init", C.c_double),
        ("alpha", C.c_double),
        ("eps_prim", C.c_double), ("eps_dual", C.c_double), ("eps_infeas", C.c_double),
        ("step_tol", C.c_double), ("feas_tol", C.c_double),
        ("fast_pass", C.c_int), ("fast_rho_off", C.c_double), ("fast_rho_on", C.c_double),
        ("fast_max_rounds", C.c_int), ("fast_max_segments", C.c_int), ("fast_segment_iters", C.c_int),
        ("coop_pass2", C.c_int), ("coop_max_batch", C.c_int),
        ("thread_max_rounds", C.c_int), ("thread_max_segments", C.c_int), ("thread_fail_rounds", C.c_int),
    ]


class PlannerParams(C.Structure):
    """struct mpcb_planner_params (include/mpcb200.h); mirrors TrajectoryOptimizer.__init__,
    trajectory_planning.py:14-48."""
    _fields_ = [
        ("dt", C.c_double),
        ("w_y", C.c_double), ("w_s", C.c_double), ("w_u", C.c_double), ("w_slack", C.c_double),
        ("u_min", C.c_double * 2), ("u_max", C.c_double * 2),
        ("k_min", C.c_double), ("k_max", C.c_double), ("a_max", C.c_double),
        ("simpson_sign", C.c_int),
        ("v_min", C.c_double), ("v_max", C.c_double),
        ("s_total", C.c_double),
    ]


class Scenario(C.Structure):
    """struct mpcb_scenario (include/mpcb200.h); mirrors ObstaclesFSM.__init__, trajectory_tracking.py:285-308."""
    _fields_ = [
        ("dynamic_obstacle", C.c_int), ("traffic_light", C.c_int),
        ("obs_trigger_s", C.c_double), ("obs_start_s", C.c_double), ("obs_v", C.c_double), ("obs_end_s", C.c_double),
        ("tl_pos", C.c_double), ("tl_trigger_s", C.c_double), ("tl_stop_duration", C.c_double),
    ]


# every symbol include/mpcb200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "mpcb_default_params": (C.c_int, [C.POINTER(Params)]),
    "mpcb_table_create": (C.c_int, [C.POINTER(C.c_void_p), c_double_p, C.c_int, c_double_p, C.c_int]),
    "mpcb_table_destroy": (C.c_int, [C.c_void_p]),
    "mpcb_table_save": (C.c_int, [C.c_void_p, C.c_char_p]),
    "mpcb_table_load": (C.c_int, [C.POINTER(C.c_void_p), C.c_char_p]),
    "mpcb_table_raw": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpcb_table_control_knots": (C.c_int, [C.c_void_p]),
    "mpcb_table_get_state": (C.c_int, [C.c_void_p, C.c_double, c_double_p]),
    "mpcb_table_get_control": (C.c_int, [C.c_void_p, C.c_double, c_double_p]),
    "mpcb_table_s_max": (C.c_double, [C.c_void_p]),
    "mpcb_table_knots": (C.c_int, [C.c_void_p]),
    "mpcb_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(Params), C.c_void_p, C.c_int]),
    "mpcb_destroy": (C.c_int, [C.c_void_p]),
    "mpcb_create_routes": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(Params), C.POINTER(C.c_void_p), C.c_int, C.c_int]),
    "mpcb_n_routes": (C.c_int, [C.c_void_p]),
    "mpcb_solve_batch_routes": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 11 + [C.c_void_p]),
    "mpcb_solve_batch": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 10 + [C.c_void_p]),
    "mpcb_solve_batch_host": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 10),
    "mpcb_solve_batch_host_u0": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 6),
    "mpcb_solve_batch_host_async": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 11),
    "mpcb_wait": (C.c_int, [C.c_void_p]),
    "mpcb_eval_batch": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 9 + [C.c_void_p]),
    "mpcb_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_ulonglong]),
    "mpcb_host_free": (C.c_int, [C.c_void_p]),
    "mpcb_device_alloc": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_ulonglong]),
    "mpcb_device_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mpcb_memcpy_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_ulonglong]),
    "mpcb_memcpy_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_ulonglong]),
    "mpcb_last_kernel_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "mpcb_last_pass_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "mpcb_last_first_pass_shape": (C.c_int, [C.c_void_p]),
    "mpcb_launch_count": (C.c_ulonglong, [C.c_void_p]),
    "mpcb_measure_fp64_peak": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_float)]),
    "mpcb_planner_default_params": (C.c_int, [C.POINTER(PlannerParams)]),
    "mpcb_hs_eval": (C.c_int, [C.c_void_p, C.POINTER(PlannerParams), C.c_int, C.c_int] + [C.c_void_p] * 5 + [C.c_void_p]),
    "mpcb_hs_nodes": (C.c_int, [C.c_void_p, C.POINTER(PlannerParams), C.c_int, C.c_int] + [C.c_void_p] * 9 + [C.c_void_p]),
    "mpcb_scenario_default": (C.c_int, [C.POINTER(Scenario), C.c_int]),
    "mpcb_sim_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.c_int, C.POINTER(Scenario), C.c_int, C.c_void_p, C.c_int]),
    "mpcb_sim_create_routes": (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.c_int, C.POINTER(Scenario), C.c_int, C.c_void_p,
                                         C.c_void_p, C.c_int]),
    "mpcb_sim_destroy": (C.c_int, [C.c_void_p]),
    "mpcb_sim_step": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "mpcb_sim_set_hot_start": (C.c_int, [C.c_void_p, C.c_int]),
    "mpcb_sim_set_follow": (C.c_int, [C.c_void_p, C.c_int, C.c_double]),
    "mpcb_sim_follow_history": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpcb_sim_follow_check": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpcb_sim_set_noise": (C.c_int, [C.c_void_p, C.c_ulonglong, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpcb_sim_noise_history": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.c_void_p, C.c_void_p]),
    "mpcb_sim_alive":(C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.c_void_p]),
    "mpcb_sim_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpcb_sim_check": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpcb_sim_running_check": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpcb_sim_branch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpcb_sim_set_worlds": (C.c_int, [C.c_void_p, C.c_int]),
    "mpcb_sim_running_follow_check": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpcb_sim_branch_worlds": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "mpcb_check_histories": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_double, C.POINTER(Scenario)] + [C.c_void_p] * 8),
    "mpcb_sim_history": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)] + [C.c_void_p] * 5 + [C.c_void_p]),
    "mpcb_strerror": (C.c_char_p, [C.c_int]),
    "mpcb_last_cuda_error": (C.c_char_p, []),
    "mpcb_abi_version": (C.c_int, []),
    "mpcb_sizeof_params": (C.c_ulonglong, []),
    "mpcb_sizeof_planner_params": (C.c_ulonglong, []),
}

_lib = None


def library_path():
    return _build.LIB


def load(build_if_missing=True):
    """Load libmpcb200.so (building it with nvcc when absent and a compiler is present)."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        if not build_if_missing:
            raise MpcbError(f"{path} is missing; run `python __graft_entry__.py` (build()) first")
        _build.build()
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)   # AttributeError if the ABI is incomplete: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.mpcb_sizeof_params() != C.sizeof(Params) or lib.mpcb_sizeof_planner_params() != C.sizeof(PlannerParams):
        raise MpcbError("libmpcb200.so and its ctypes mirror disagree on the parameter structs (stale build?)")
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        lib = load()
        msg = lib.mpcb_strerror(rc).decode()
        if rc == -2:
            msg += ": " + lib.mpcb_last_cuda_error().decode()
        raise MpcbError(f"{what or 'libmpcb200'} failed ({rc}): {msg}")
