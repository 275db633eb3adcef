"""ctypes binding of libqmb200.so (C ABI: include/qmb200.h).  Fails loudly when the library is missing."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
LIB_PATH = os.environ.get("QMB200_LIB", os.path.join(HERE, "libqmb200.so"))   # override only selects another build of the same library
ASSETS = os.path.join(ROOT, "assets")

NX, NU, RBD, CMD, TARGET, EMAX, KMAX = 30, 30, 55, 54, 37, 32, 4

dp = C.POINTER(C.c_double)
ip = C.POINTER(C.c_int32)


class QmbError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [("task_file", C.c_char_p), ("urdf_file", C.c_char_p), ("reference_file", C.c_char_p), ("wbc_gains_file", C.c_char_p),
                ("batch", C.c_int32), ("device", C.c_int32), ("time_horizon", C.c_double), ("dt", C.c_double), ("max_nodes", C.c_int32), ("wbc_variant", C.c_int32)]


class WbcGains(C.Structure):
    """qmb200_wbc_gains (WbcBase::dynamicCallback, qm_wbc/cfg/wbcWigeht.cfg:7-47)."""
    _fields_ = [(n, C.c_double) for n in ("kp_swing", "kd_swing", "base_height_kp", "base_height_kd", "kp_base_linear", "kd_base_linear", "kp_base_angular", "kd_base_angular")] + \
               [("kp_arm_joint", C.c_double * 6), ("kd_arm_joint", C.c_double * 6), ("kp_ee_linear", C.c_double * 3), ("kd_ee_linear", C.c_double * 3), ("kp_ee_angular", C.c_double * 3), ("kd_ee_angular", C.c_double * 3)]


# every symbol include/qmb200.h declares (checked by the CPU test-suite)
SYMBOLS = ["qmb200_create", "qmb200_destroy", "qmb200_last_error", "qmb200_get_dims", "qmb200_get_model_info", "qmb200_get_joint_name",
           "qmb200_wbc_update", "qmb200_wbc_update_dev", "qmb200_wbc_set_input_last", "qmb200_wbc_get_input_last", "qmb200_wbc_get_gains", "qmb200_wbc_set_gains", "qmb200_wbc_get_diagnostics", "qmb200_wbc_set_iteration_caps",
           "qmb200_mpc_solve", "qmb200_mpc_solve_dev", "qmb200_mpc_set_iterations", "qmb200_mpc_set_solver", "qmb200_mpc_get_solver", "qmb200_mpc_reset", "qmb200_mpc_set_solution", "qmb200_mpc_get_solution",
           "qmb200_policy_eval", "qmb200_policy_eval_dev", "qmb200_tick", "qmb200_tick_dev", "qmb200_centroidal_state_from_rbd",
           "qmb200_gait_schedule", "qmb200_launch_count", "qmb200_stream", "qmb200_debug_get_step",
           "qmb200_gait_create", "qmb200_gait_destroy", "qmb200_gait_insert_template", "qmb200_gait_get_mode_schedule",
           "qmb200_observation_update", "qmb200_observation_update_dev", "qmb200_target_trajectories", "qmb200_target_trajectories_dev", "qmb200_initial_ee_target",
           "qmb200_control_law", "qmb200_control_law_dev", "qmb200_set_arm_gains", "qmb200_hw_write", "qmb200_hw_write_dev", "qmb200_hw_set_delay", "qmb200_update", "qmb200_update_dev",
           "qmb200_debug_model_blob", "qmb200_comm_get_unique_id", "qmb200_comm_init", "qmb200_comm_destroy", "qmb200_comm_info", "qmb200_allgather_torque", "qmb200_gait_bin_permutation", "qmb200_set_pipeline", "qmb200_set_profiling", "qmb200_collect_kernel_times", "qmb200_get_kernel_times", "qmb200_get_flow_kernel_time", "qmb200_measure_fp64_peak",
           "qmb200_mpc_set_feedback_policy", "qmb200_mpc_get_feedback_policy", "qmb200_policy_eval_state", "qmb200_policy_eval_state_dev", "qmb200_mpc_get_controller", "qmb200_mpc_get_controller_dev",
           "qmb200_mpc_set_value_function", "qmb200_mpc_get_value_function", "qmb200_value_function", "qmb200_value_function_dev"]

_lib = None


def load_library():
    """Load libqmb200.so; raise (never fall back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise QmbError("libqmb200.so not built (%s): run `python -c 'import __graft_entry__ as g; g.build()'` — there is no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.qmb200_last_error.restype = C.c_char_p
    lib.qmb200_last_error.argtypes = [C.c_void_p]
    lib.qmb200_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_void_p)]
    lib.qmb200_destroy.argtypes = [C.c_void_p]
    lib.qmb200_destroy.restype = None
    lib.qmb200_debug_model_blob.restype = C.c_int64
    lib.qmb200_debug_model_blob.argtypes = [C.POINTER(Config), C.c_void_p, C.c_int64]
    lib.qmb200_launch_count.restype = C.c_int64
    lib.qmb200_launch_count.argtypes = [C.c_void_p]
    lib.qmb200_stream.restype = C.c_void_p
    lib.qmb200_stream.argtypes = [C.c_void_p]
    lib.qmb200_set_arm_gains.argtypes = [C.c_void_p, C.c_double, C.c_double]
    lib.qmb200_hw_set_delay.argtypes = [C.c_void_p, C.c_double]
    lib.qmb200_mpc_set_iterations.argtypes = [C.c_void_p, C.c_int32, C.c_double]
    lib.qmb200_initial_ee_target.restype = None
    lib.qmb200_gait_destroy.restype = None
    lib.qmb200_gait_destroy.argtypes = [C.c_void_p]
    lib.qmb200_gait_insert_template.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_double, C.c_double]
    lib.qmb200_gait_get_mode_schedule.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_void_p]
    for name in SYMBOLS:
        getattr(lib, name)
    _lib = lib
    return lib


def asset(name):
    return os.path.join(ASSETS, name)
