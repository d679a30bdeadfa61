"""ctypes binding of libsocp_b200.so (include/socp_b200.h).  No fallback of any kind: if the
CUDA library is missing or no GPU is present, the calls raise."""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# SOCP_LIB selects another build of the same library (the -fmad=false parity build, socp_b200/build.py)
SO_PATH = os.environ.get("SOCP_LIB") or os.path.join(HERE, "libsocp_b200.so")

MAX_NODES, MAX_DIM = 64, 7
HOST, DEVICE = 0, 1


class SocpError(RuntimeError):
    pass


class Shape(ctypes.Structure):
    _fields_ = [("model_id", ctypes.c_int), ("num_multi", ctypes.c_int), ("step_nbr", ctypes.c_int),
                ("mode_t", ctypes.c_int * MAX_NODES), ("mode_X", (ctypes.c_int * MAX_DIM) * MAX_NODES),
                ("integrator", ctypes.c_int), ("ode_tol", ctypes.c_double)]


class Stats(ctypes.Structure):
    _fields_ = [("rk4_steps", ctypes.c_double), ("kernel_launches", ctypes.c_double),
                ("solver_rounds", ctypes.c_double), ("device_bytes", ctypes.c_double),
                ("integrate_ms", ctypes.c_double), ("integrate_launches", ctypes.c_double),
                ("advance_ms", ctypes.c_double), ("advance_launches", ctypes.c_double),
                ("assemble_ms", ctypes.c_double), ("jac_ms", ctypes.c_double),
                ("iterations", ctypes.c_double), ("jac_evals", ctypes.c_double), ("dopri_steps", ctypes.c_double),
                ("qpass_ms", ctypes.c_double), ("res_evals", ctypes.c_double)]


_LIB = None
# every symbol include/socp_b200.h declares
SYMBOLS = ["socp_create", "socp_destroy", "socp_last_error", "socp_set_stream", "socp_sync",
           "socp_get_stats", "socp_reset_stats", "socp_set_profiling", "socp_timer_start", "socp_timer_stop",
           "socp_model_dim", "socp_model_nparams", "socp_model_default_steps",
           "socp_model_default_params", "socp_num_param", "socp_jac_band", "socp_set_obstacles", "socp_traj_batch", "socp_traj_adaptive_batch",
           "socp_trace_width", "socp_trace_max_rows", "socp_trace_batch", "socp_point_batch", "socp_residual_batch", "socp_fdjac_batch", "socp_solve_batch",
           "socp_traj_var_batch", "socp_jacobian_batch", "socp_solve_hybrj_batch",
           "socp_continuation_param_batch", "socp_continuation_boundary_batch",
           "socp_move_batch", "socp_solution_batch", "socp_solution_trace_batch", "socp_init_shooting_batch",
           "socp_measure_fp64_peak"]


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(SO_PATH):
        raise SocpError("%s is missing: run `python -m socp_b200.build` (nvcc, sm_100a). "
                        "There is no CPU fallback." % SO_PATH)
    L = ctypes.CDLL(SO_PATH)
    vp, ci, cl, cd = ctypes.c_void_p, ctypes.c_int, ctypes.c_long, ctypes.c_double
    P = ctypes.POINTER
    sp = P(Shape)
    L.socp_create.argtypes = [ci, P(vp)]
    L.socp_destroy.argtypes = [vp]
    L.socp_destroy.restype = None
    L.socp_last_error.argtypes = [vp]
    L.socp_last_error.restype = ctypes.c_char_p
    L.socp_set_stream.argtypes = [vp, vp]
    L.socp_sync.argtypes = [vp]
    L.socp_get_stats.argtypes = [vp, P(Stats)]
    L.socp_reset_stats.argtypes = [vp]
    L.socp_set_profiling.argtypes = [vp, ci]
    L.socp_timer_start.argtypes = [vp]
    L.socp_timer_stop.argtypes = [vp, P(ctypes.c_float)]
    L.socp_model_dim.argtypes = [ci]
    L.socp_model_nparams.argtypes = [ci]
    L.socp_model_default_steps.argtypes = [ci]
    L.socp_model_default_params.argtypes = [ci, vp]
    L.socp_num_param.argtypes = [sp]
    L.socp_jac_band.argtypes = [sp, vp, vp]
    L.socp_set_obstacles.argtypes = [vp, ci, vp, vp, vp]
    L.socp_traj_batch.argtypes = [vp, ci, ci, cl, vp, vp, vp, vp, vp, vp, ci]
    L.socp_traj_adaptive_batch.argtypes = [vp, ci, ci, cl, vp, vp, vp, vp, vp, cd, vp, vp, ci]
    L.socp_trace_width.argtypes = [ci]
    L.socp_trace_max_rows.argtypes = [ci, ci]
    L.socp_trace_batch.argtypes = [vp, ci, ci, cl, vp, vp, vp, vp, vp, vp, vp, vp, ci]
    L.socp_point_batch.argtypes = [vp, ci, cl, vp, vp, vp, vp, vp, vp, vp, vp, ci]
    L.socp_residual_batch.argtypes = [vp, sp, cl, vp, vp, vp, vp, vp, ci]
    L.socp_fdjac_batch.argtypes = [vp, sp, cl, vp, vp, vp, vp, cd, vp, ci]
    L.socp_solve_batch.argtypes = [vp, sp, cl, vp, vp, vp, vp, cd, ci, vp, vp, vp, ci]
    L.socp_traj_var_batch.argtypes = [vp, ci, ci, cl, vp, vp, vp, vp, vp, ci]
    L.socp_jacobian_batch.argtypes = [vp, sp, cl, vp, vp, vp, vp, vp, ci]
    L.socp_solve_hybrj_batch.argtypes = [vp, sp, cl, vp, vp, vp, vp, cd, ci, vp, vp, vp, vp, ci]
    L.socp_continuation_param_batch.argtypes = [vp, sp, cl, vp, vp, vp, vp, cd, ci, cd, ci, vp, cd, vp, vp, ci]
    L.socp_continuation_boundary_batch.argtypes = [vp, sp, cl, vp, vp, vp, vp, vp, vp, cd, ci, cd, cd, vp, vp, ci]
    L.socp_move_batch.argtypes = [vp, sp, cl, vp, vp, vp, ci, vp, vp, ci]
    L.socp_solution_batch.argtypes = [vp, sp, cl, vp, vp, vp, vp, vp, ci]
    L.socp_solution_trace_batch.argtypes = [vp, sp, cl, vp, vp, vp, vp, vp, ci]
    L.socp_init_shooting_batch.argtypes = [vp, sp, cl, vp, vp, vp, vp, vp, vp, vp, vp, vp, ci]
    L.socp_measure_fp64_peak.argtypes = [vp, P(cd), P(cd)]
    for name in SYMBOLS:
        f = getattr(L, name)
        if f.restype is ctypes.c_int or name not in ("socp_destroy", "socp_last_error"):
            if name not in ("socp_destroy", "socp_last_error"):
                f.restype = ci
    _LIB = L
    return L
