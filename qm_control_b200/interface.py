"""Python mirror of qm::QMInterface (qm_interface/include/qm_interface/QMInterface.h:31-54) and the solver handle.

QMInterface only records the three files the reference constructor takes and raises the same way on missing files
(QMInterface.cpp:45,53,61); ``Solver`` owns one ``qmb200_handle`` (one per GPU) and exposes the C-ABI calls on numpy
(host) or torch-cuda (device) buffers.
"""
import ctypes as C
import os

import numpy as np

from . import _lib
from ._lib import NX, NU, RBD, CMD, TARGET, EMAX, KMAX, Config, QmbError, dp, ip


class QMInterface:
    def __init__(self, taskFile=None, urdfFile=None, referenceFile=None, wbcGainsFile=None):
        self.taskFile = taskFile or _lib.asset("qm_task.info")
        self.urdfFile = urdfFile or _lib.asset("qm_robot.urdf")
        self.referenceFile = referenceFile or _lib.asset("qm_reference.info")
        self.gaitFile = _lib.asset("qm_gait.info")
        self.wbcGainsFile = wbcGainsFile
        for what, path in (("Task file", self.taskFile), ("URDF file", self.urdfFile), ("targetCommand file", self.referenceFile)):
            if not os.path.exists(path):
                raise ValueError("[QMInterface] %s not found: %s" % (what, path))


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None and tuple(a.shape) != tuple(shape):
        raise ValueError("expected shape %s, got %s" % (shape, a.shape))
    return a


def _i32(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.int32)
    if shape is not None and tuple(a.shape) != tuple(shape):
        raise ValueError("expected shape %s, got %s" % (shape, a.shape))
    return a


def _p(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return C.c_void_p(a.ctypes.data)
    return C.c_void_p(a.data_ptr())   # torch tensor (device pointer)


class Solver:
    """One qmb200_handle: batched MPC + WBC for `batch` robots on CUDA device `device`."""

    def __init__(self, interface=None, batch=1, device=0, time_horizon=0.0, dt=0.0, max_nodes=0, wbc_variant=0):
        self.lib = _lib.load_library()
        self.interface = interface or QMInterface()
        cfg = Config(self.interface.taskFile.encode(), self.interface.urdfFile.encode(), self.interface.referenceFile.encode(),
                     self.interface.wbcGainsFile.encode() if self.interface.wbcGainsFile else None, batch, device, time_horizon, dt, max_nodes, wbc_variant)
        self._cfg = cfg
        h = C.c_void_p()
        rc = self.lib.qmb200_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise QmbError("qmb200_create failed (%d): %s" % (rc, self.lib.qmb200_last_error(None).decode()))
        self.h = h
        b, n, e, k = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
        self.lib.qmb200_get_dims(self.h, C.byref(b), C.byref(n), C.byref(e), C.byref(k))
        self.batch, self.nmax, self.emax, self.kmax = b.value, n.value, e.value, k.value
        mass, hor, dtt = C.c_double(), C.c_double(), C.c_double()
        self.initial_state = np.zeros(NX); self.default_joint_state = np.zeros(18)
        self.lib.qmb200_get_model_info(self.h, C.byref(mass), _p(self.initial_state), _p(self.default_joint_state), C.byref(hor), C.byref(dtt))
        self.robot_mass, self.time_horizon, self.dt = mass.value, hor.value, dtt.value

    def close(self):
        if getattr(self, "h", None):
            self.lib.qmb200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc, what):
        if rc != 0:
            raise QmbError("%s failed (%d): %s" % (what, rc, self.lib.qmb200_last_error(self.h).decode()))

    @property
    def launch_count(self):
        return int(self.lib.qmb200_launch_count(self.h))

    @property
    def stream(self):
        return self.lib.qmb200_stream(self.h)

    def joint_names(self):
        out = []
        for j in range(18):
            buf = C.create_string_buffer(64); self.lib.qmb200_get_joint_name(self.h, j, buf, 64); out.append(buf.value.decode())
        return out

    # ---------------- WBC ----------------
    def wbc_update(self, x_des, u_des, rbd, mode, period, time):
        B = self.batch
        x_des = _f64(x_des, (B, NX)); u_des = _f64(u_des, (B, NU)); rbd = _f64(rbd, (B, RBD)); mode = _i32(mode, (B,)); period = _f64(period, (B,)); time = _f64(time, (B,))
        cmd = np.empty((B, CMD)); status = np.empty(B, dtype=np.int32)
        self._chk(self.lib.qmb200_wbc_update(self.h, _p(x_des), _p(u_des), _p(rbd), _p(mode), _p(period), _p(time), _p(cmd), _p(status)), "qmb200_wbc_update")
        return cmd, status

    def wbc_update_dev(self, x_des, u_des, rbd, mode, period, time, cmd, status, stream=None):
        self._chk(self.lib.qmb200_wbc_update_dev(self.h, _p(x_des), _p(u_des), _p(rbd), _p(mode), _p(period), _p(time), _p(cmd), _p(status), C.c_void_p(stream) if stream else None), "qmb200_wbc_update_dev")

    def wbc_get_gains(self):
        """→ dict of the task-formulator PD gains (WbcBase::dynamicCallback fields)."""
        g = _lib.WbcGains(); self._chk(self.lib.qmb200_wbc_get_gains(self.h, C.byref(g)), "qmb200_wbc_get_gains")
        return {n: (list(getattr(g, n)) if hasattr(getattr(g, n), "__len__") else getattr(g, n)) for n, _ in _lib.WbcGains._fields_}

    def wbc_set_gains(self, **gains):
        """Dynamic reconfigure of the WBC gains: keyword per field of qmb200_wbc_gains; unspecified fields keep their value."""
        g = _lib.WbcGains(); self._chk(self.lib.qmb200_wbc_get_gains(self.h, C.byref(g)), "qmb200_wbc_get_gains")
        for k, v in gains.items():
            cur = getattr(g, k)
            if hasattr(cur, "__len__"):
                for i, x in enumerate(v):
                    cur[i] = float(x)
            else:
                setattr(g, k, float(v))
        self._chk(self.lib.qmb200_wbc_set_gains(self.h, C.byref(g)), "qmb200_wbc_set_gains")

    def wbc_set_input_last(self, input_last=None):
        self._chk(self.lib.qmb200_wbc_set_input_last(self.h, _p(_f64(input_last, (self.batch, NU))) if input_last is not None else None), "qmb200_wbc_set_input_last")

    def wbc_get_diagnostics(self):
        """→ dict(level0_passes, level1_iterations, level2_iterations, working_set) of the last WBC update, per robot."""
        d = np.zeros(self.batch, dtype=np.int32); self._chk(self.lib.qmb200_wbc_get_diagnostics(self.h, _p(d)), "qmb200_wbc_get_diagnostics")
        return dict(level0_passes=d & 0xFF, level1_iterations=(d >> 8) & 0xFF, level2_iterations=(d >> 16) & 0xFF, working_set=(d >> 24) & 0xFF)

    def wbc_set_iteration_caps(self, level0_passes=0, active_set_iterations=0):
        self._chk(self.lib.qmb200_wbc_set_iteration_caps(self.h, int(level0_passes), int(active_set_iterations)), "qmb200_wbc_set_iteration_caps")

    def wbc_get_input_last(self):
        out = np.empty((self.batch, NU)); self._chk(self.lib.qmb200_wbc_get_input_last(self.h, _p(out)), "qmb200_wbc_get_input_last"); return out

    # ---------------- MPC ----------------
    def _prob(self, prob):
        B = self.batch
        return [_f64(prob["t0"], (B,)), _f64(prob["x0"], (B, NX)), _i32(prob["n_events"], (B,)), _f64(prob["event_times"], (B, EMAX)), _i32(prob["modes"], (B, EMAX + 1)),
                _i32(prob["n_target"], (B,)), _f64(prob["target_times"], (B, KMAX)), _f64(prob["target_states"], (B, KMAX, TARGET))]

    def mpc_solve(self, prob):
        B, N = self.batch, self.nmax; a = self._prob(prob)
        out = dict(n_nodes=np.zeros(B, dtype=np.int32), t=np.zeros((B, N)), event=np.zeros((B, N), dtype=np.int32), x=np.zeros((B, N, NX)), u=np.zeros((B, N, NU)),
                   status=np.zeros(B, dtype=np.int32), step_info=np.zeros((B, 4)))
        self._chk(self.lib.qmb200_mpc_solve(self.h, *[_p(v) for v in a], _p(out["n_nodes"]), _p(out["t"]), _p(out["event"]), _p(out["x"]), _p(out["u"]), _p(out["status"]), _p(out["step_info"])), "qmb200_mpc_solve")
        return out

    def mpc_solve_dev(self, prob_dev, stream=None):
        keys = ("t0", "x0", "n_events", "event_times", "modes", "n_target", "target_times", "target_states")
        self._chk(self.lib.qmb200_mpc_solve_dev(self.h, *[_p(prob_dev[k]) for k in keys], C.c_void_p(stream) if stream else None), "qmb200_mpc_solve_dev")

    SOLVERS = {"sqp": 0, "ipm": 1, "ddp": 2}

    def mpc_set_solver(self, solver):
        """'sqp' (SqpMpc, what QMController runs), 'ipm' (ipm{} block) or 'ddp' (ddp{} block, discrete-time form): include/qmb200.h."""
        self._chk(self.lib.qmb200_mpc_set_solver(self.h, self.SOLVERS[solver] if isinstance(solver, str) else int(solver)), "qmb200_mpc_set_solver")

    def mpc_get_solver(self):
        s, it = C.c_int32(), C.c_int32(); dt, gx, gn = C.c_double(), C.c_double(), C.c_double()
        self.lib.qmb200_mpc_get_solver(self.h, C.byref(s), C.byref(it), C.byref(dt), C.byref(gx), C.byref(gn))
        return dict(solver=s.value, iterations=it.value, delta_tol=dt.value, g_max=gx.value, g_min=gn.value)

    def mpc_set_iterations(self, sqp_iterations=0, cost_tol=0.0):
        """sqp.sqpIteration / costTol (SqpSolver::runImpl loop bound and checkConvergence tolerance)."""
        self._chk(self.lib.qmb200_mpc_set_iterations(self.h, int(sqp_iterations), float(cost_tol)), "qmb200_mpc_set_iterations")

    def mpc_reset(self):
        self._chk(self.lib.qmb200_mpc_reset(self.h), "qmb200_mpc_reset")

    def mpc_set_solution(self, sol):
        B, N = self.batch, self.nmax
        self._chk(self.lib.qmb200_mpc_set_solution(self.h, _p(_i32(sol["n_nodes"], (B,))), _p(_f64(sol["t"], (B, N))), _p(_i32(sol["event"], (B, N))), _p(_f64(sol["x"], (B, N, NX))), _p(_f64(sol["u"], (B, N, NU)))), "qmb200_mpc_set_solution")

    def mpc_get_solution(self):
        B, N = self.batch, self.nmax
        out = dict(n_nodes=np.zeros(B, dtype=np.int32), t=np.zeros((B, N)), event=np.zeros((B, N), dtype=np.int32), x=np.zeros((B, N, NX)), u=np.zeros((B, N, NU)),
                   status=np.zeros(B, dtype=np.int32), step_info=np.zeros((B, 4)))
        self._chk(self.lib.qmb200_mpc_get_solution(self.h, _p(out["n_nodes"]), _p(out["t"]), _p(out["event"]), _p(out["x"]), _p(out["u"]), _p(out["status"]), _p(out["step_info"])), "qmb200_mpc_get_solution")
        return out

    def policy_eval(self, t):
        B = self.batch; t = _f64(t, (B,)); xd = np.empty((B, NX)); ud = np.empty((B, NU)); mode = np.empty(B, dtype=np.int32)
        self._chk(self.lib.qmb200_policy_eval(self.h, _p(t), _p(xd), _p(ud), _p(mode)), "qmb200_policy_eval")
        return xd, ud, mode

    def mpc_set_feedback_policy(self, on=True):
        """useFeedbackPolicy: evaluate the LinearController u = uff(t) + K(t) x of the last solve instead of the feed-forward policy (include/qmb200.h)."""
        self._chk(self.lib.qmb200_mpc_set_feedback_policy(self.h, 1 if on else 0), "qmb200_mpc_set_feedback_policy")

    def mpc_get_feedback_policy(self):
        v = C.c_int32(); self._chk(self.lib.qmb200_mpc_get_feedback_policy(self.h, C.byref(v)), "qmb200_mpc_get_feedback_policy"); return bool(v.value)

    def policy_eval_state(self, t, x):
        """MPC_MRT_Interface::evaluatePolicy(t, x) → (x_des, u_des, mode); with the switch off identical to policy_eval(t)."""
        B = self.batch; t = _f64(t, (B,)); x = _f64(x, (B, NX)); xd = np.empty((B, NX)); ud = np.empty((B, NU)); mode = np.empty(B, dtype=np.int32)
        self._chk(self.lib.qmb200_policy_eval_state(self.h, _p(t), _p(x), _p(xd), _p(ud), _p(mode)), "qmb200_policy_eval_state")
        return xd, ud, mode

    def policy_eval_state_dev(self, t, x, x_des, u_des, mode, stream=None):
        self._chk(self.lib.qmb200_policy_eval_state_dev(self.h, _p(t), _p(x), _p(x_des), _p(u_des), _p(mode), C.c_void_p(stream) if stream else None), "qmb200_policy_eval_state_dev")

    def mpc_get_controller(self, b0=0, count=None):
        """LinearController of robots [b0, b0 + count) → dict(bias[count, NMAX, 30], gain[count, NMAX, 30, 30] (row = input), feedback[count])."""
        count = self.batch - b0 if count is None else int(count); N = self.nmax
        out = dict(bias=np.zeros((count, N, NU)), gain=np.zeros((count, N, NU, NX)), feedback=np.zeros(count, dtype=np.int32))
        self._chk(self.lib.qmb200_mpc_get_controller(self.h, int(b0), count, _p(out["bias"]), _p(out["gain"]), _p(out["feedback"])), "qmb200_mpc_get_controller")
        return out

    def mpc_get_controller_dev(self, b0, count, bias, gain, feedback, stream=None):
        self._chk(self.lib.qmb200_mpc_get_controller_dev(self.h, int(b0), int(count), _p(bias), _p(gain), _p(feedback), C.c_void_p(stream) if stream else None), "qmb200_mpc_get_controller_dev")

    def mpc_set_value_function(self, on=True):
        """createValueFunction: the solve keeps the Riccati cost-to-go of its last QP for value_function (include/qmb200.h).  Refused with the DDP solver."""
        self._chk(self.lib.qmb200_mpc_set_value_function(self.h, 1 if on else 0), "qmb200_mpc_set_value_function")

    def mpc_get_value_function(self):
        v = C.c_int32(); self._chk(self.lib.qmb200_mpc_get_value_function(self.h, C.byref(v)), "qmb200_mpc_get_value_function"); return bool(v.value)

    def value_function(self, t, x):
        """getValueFunction(t, x) of every robot → dict(dfdx[B, 30], dfdxx[B, 30, 30], valid[B]); f is 0.  Zero where valid is 0."""
        B = self.batch; t = _f64(t, (B,)); x = _f64(x, (B, NX))
        out = dict(dfdx=np.empty((B, NX)), dfdxx=np.empty((B, NX, NX)), valid=np.empty(B, dtype=np.int32))
        self._chk(self.lib.qmb200_value_function(self.h, _p(t), _p(x), _p(out["dfdx"]), _p(out["dfdxx"]), _p(out["valid"])), "qmb200_value_function")
        return out

    def value_function_dev(self, t, x, dfdx, dfdxx, valid, stream=None):
        self._chk(self.lib.qmb200_value_function_dev(self.h, _p(t), _p(x), _p(dfdx), _p(dfdxx), _p(valid), C.c_void_p(stream) if stream else None), "qmb200_value_function_dev")

    def tick(self, prob, t_eval, rbd, period):
        B = self.batch; a = self._prob(prob); t_eval = _f64(t_eval, (B,)); rbd = _f64(rbd, (B, RBD)); period = _f64(period, (B,))
        cmd = np.empty((B, CMD)); status = np.empty(B, dtype=np.int32)
        self._chk(self.lib.qmb200_tick(self.h, *[_p(v) for v in a], _p(t_eval), _p(rbd), _p(period), _p(cmd), _p(status)), "qmb200_tick")
        return cmd, status

    def tick_dev(self, prob_dev, t_eval, rbd, period, cmd, status, stream=None):
        keys = ("t0", "x0", "n_events", "event_times", "modes", "n_target", "target_times", "target_states")
        self._chk(self.lib.qmb200_tick_dev(self.h, *[_p(prob_dev[k]) for k in keys], _p(t_eval), _p(rbd), _p(period), _p(cmd), _p(status), C.c_void_p(stream) if stream else None), "qmb200_tick_dev")

    # ---------------- multi-GPU (include/qmb200.h: one NCCL all-gather of the torque rows per tick, driven from the C++ host) ----------------
    def comm_unique_id(self):
        """rank 0: the 128-byte ncclUniqueId to ship to the other ranks."""
        buf = C.create_string_buffer(128)
        if self.lib.qmb200_comm_get_unique_id(buf) != 0:
            raise QmbError("qmb200_comm_get_unique_id: %s" % self.lib.qmb200_last_error(None).decode())
        return buf.raw

    def comm_init(self, nranks, rank, unique_id):
        self._chk(self.lib.qmb200_comm_init(self.h, int(nranks), int(rank), C.c_char_p(bytes(unique_id))), "qmb200_comm_init")

    def comm_info(self):
        n, r, v = C.c_int32(), C.c_int32(), C.c_int32(); self.lib.qmb200_comm_info(self.h, C.byref(n), C.byref(r), C.byref(v)); return n.value, r.value, v.value

    def allgather_torque(self, cmd_dev, torque_all_dev, perm_dev=None, stream=None):
        """torque_all[r * B + i] = cmd[i, 36:54] of rank r (original robot order when perm_dev is given); device tensors."""
        self._chk(self.lib.qmb200_allgather_torque(self.h, None, _p(cmd_dev), _p(perm_dev), _p(torque_all_dev), C.c_void_p(stream) if stream else None), "qmb200_allgather_torque")

    def gait_bin_permutation(self, prob):
        """Host: perm[p] = original index of the robot at position p after sorting by contact phase (qmb200_gait_bin_permutation)."""
        n = len(prob["t0"]); perm = np.zeros(n, dtype=np.int32)
        rc = self.lib.qmb200_gait_bin_permutation(n, _p(_f64(prob["t0"])), _p(_i32(prob["n_events"])), _p(_f64(prob["event_times"])), _p(_i32(prob["modes"])), _p(perm))
        if rc != 0:
            raise QmbError("qmb200_gait_bin_permutation failed")
        return perm

    def set_pipeline(self, chunks):
        """Number of robot ranges the tick runs as concurrent stream chains (include/qmb200.h: qmb200_set_pipeline)."""
        self._chk(self.lib.qmb200_set_pipeline(self.h, int(chunks)), "qmb200_set_pipeline")

    def set_profiling(self, on=True):
        self._chk(self.lib.qmb200_set_profiling(self.h, 1 if on else 0), "qmb200_set_profiling")

    def collect_kernel_times(self):
        self.lib.qmb200_collect_kernel_times(self.h)

    def kernel_times(self):
        ms = np.zeros(6); self._chk(self.lib.qmb200_get_kernel_times(self.h, _p(ms)), "qmb200_get_kernel_times")
        d = dict(zip(("setup", "lq", "riccati", "linesearch", "policy_eval", "wbc"), ms.tolist()))
        v = C.c_double(); self._chk(self.lib.qmb200_get_flow_kernel_time(self.h, C.byref(v)), "qmb200_get_flow_kernel_time"); d["lq_flow"] = v.value   # part of "lq"
        return d

    def measure_fp64_peak(self):
        v = C.c_double(); self._chk(self.lib.qmb200_measure_fp64_peak(self.h, C.byref(v)), "qmb200_measure_fp64_peak"); return v.value

    def debug_get_step(self):
        B, N = self.batch, self.nmax; dx = np.zeros((B, N, NX)); du = np.zeros((B, N, NU)); robot = np.zeros((B, 8))
        self._chk(self.lib.qmb200_debug_get_step(self.h, _p(dx), _p(du), _p(robot)), "qmb200_debug_get_step"); return dx, du, robot

    # ---------------- controller side (SURVEY §8f): observation, targets, control law, plant law, QMController::update ----------------
    def observation_update(self, rbd, period, t_obs, x_obs):
        """QMController::updateStateEstimation tail (QMController.cpp:236-243) → (t_obs, x_obs) advanced."""
        B = self.batch; rbd = _f64(rbd, (B, RBD)); period = _f64(period, (B,)); t = _f64(t_obs, (B,)).copy(); x = _f64(x_obs, (B, NX)).copy()
        self._chk(self.lib.qmb200_observation_update(self.h, _p(rbd), _p(period), _p(t), _p(x)), "qmb200_observation_update"); return t, x

    def target_trajectories(self, kind, cmd, t_obs, x_obs, ee_state, last_ee_target):
        """QmTargetTrajectoriesPublisher_node.cpp:44-208 → (n_target, target_times, target_states, last_ee_target)."""
        B = self.batch; c = np.zeros((B, 7)); cmd = np.asarray(cmd, dtype=np.float64).reshape(B, -1); c[:, :cmd.shape[1]] = cmd
        t = _f64(t_obs, (B,)); x = _f64(x_obs, (B, NX)); ee = _f64(ee_state, (B, 7)); le = _f64(last_ee_target, (B, 7)).copy()
        nt = np.zeros(B, dtype=np.int32); tt = np.zeros((B, KMAX)); ts = np.zeros((B, KMAX, TARGET))
        self._chk(self.lib.qmb200_target_trajectories(self.h, int(kind), _p(c), _p(t), _p(x), _p(ee), _p(le), _p(nt), _p(tt), _p(ts)), "qmb200_target_trajectories"); return nt, tt, ts, le

    def initial_ee_target(self):
        v = np.zeros(7); self.lib.qmb200_initial_ee_target(_p(v)); return np.tile(v, (self.batch, 1))

    def set_arm_gains(self, kp, kd):
        self._chk(self.lib.qmb200_set_arm_gains(self.h, float(kp), float(kd)), "qmb200_set_arm_gains")

    def control_law(self, x_des, u_des, wbc_cmd, t_obs, x_obs, joint_cmd, arm_pos_cmd, last_time):
        """SafetyChecker + updateControlLaw (QMController.cpp:159-190 / 427-445) → (joint_cmd, arm_pos_cmd, last_time, status)."""
        B = self.batch; jc = _f64(joint_cmd, (B, 18, 5)).copy(); ap = _f64(arm_pos_cmd, (B, 6)).copy(); lt = _f64(last_time, (B,)).copy(); st = np.zeros(B, dtype=np.int32)
        self._chk(self.lib.qmb200_control_law(self.h, _p(_f64(x_des, (B, NX))), _p(_f64(u_des, (B, NU))), _p(_f64(wbc_cmd, (B, CMD))), _p(_f64(t_obs, (B,))), _p(_f64(x_obs, (B, NX))), _p(jc), _p(ap), _p(lt), _p(st)),
                  "qmb200_control_law"); return jc, ap, lt, st

    def hw_set_delay(self, delay):
        self._chk(self.lib.qmb200_hw_set_delay(self.h, float(delay)), "qmb200_hw_set_delay")

    def hw_write(self, time, period, joint_cmd, joint_pos, joint_vel):
        """QMHWSim::writeSim (QMHWSim.cpp:98-116) → (effort[B,18], status)."""
        B = self.batch; eff = np.zeros((B, 18)); st = np.zeros(B, dtype=np.int32)
        self._chk(self.lib.qmb200_hw_write(self.h, _p(_f64(time, (B,))), _p(_f64(period, (B,))), _p(_f64(joint_cmd, (B, 18, 5))), _p(_f64(joint_pos, (B, 18))), _p(_f64(joint_vel, (B, 18))), _p(eff), _p(st)), "qmb200_hw_write")
        return eff, st

    def update(self, rbd, period, t_obs, x_obs, joint_cmd, arm_pos_cmd, last_time):
        """QMController::update (QMController.cpp:128-175) on the stored policy → (t_obs, x_obs, joint_cmd, arm_pos_cmd, last_time, cmd[B,54], status)."""
        B = self.batch; t = _f64(t_obs, (B,)).copy(); x = _f64(x_obs, (B, NX)).copy(); jc = _f64(joint_cmd, (B, 18, 5)).copy(); ap = _f64(arm_pos_cmd, (B, 6)).copy(); lt = _f64(last_time, (B,)).copy()
        cmd = np.zeros((B, CMD)); st = np.zeros(B, dtype=np.int32)
        self._chk(self.lib.qmb200_update(self.h, _p(_f64(rbd, (B, RBD))), _p(_f64(period, (B,))), _p(t), _p(x), _p(jc), _p(ap), _p(lt), _p(cmd), _p(st)), "qmb200_update")
        return t, x, jc, ap, lt, cmd, st

    # ---------------- utilities ----------------
    def centroidal_state_from_rbd(self, rbd):
        rbd = _f64(rbd); n = rbd.shape[0]; x = np.empty((n, NX))
        self._chk(self.lib.qmb200_centroidal_state_from_rbd(self.h, n, _p(rbd), _p(x)), "qmb200_centroidal_state_from_rbd"); return x


def gait_schedule(gait_name, t_start, lo, hi, gait_file=None):
    """GaitSchedule tiling of a gait.info template → (event_times[EMAX], mode_sequence[EMAX+1], n_events)."""
    lib = _lib.load_library(); ev = np.zeros(EMAX); md = np.full(EMAX + 1, 15, dtype=np.int32)
    n = lib.qmb200_gait_schedule((gait_file or _lib.asset("qm_gait.info")).encode(), gait_name.encode(), C.c_double(t_start), C.c_double(lo), C.c_double(hi), _p(ev), _p(md))
    if n < 0:
        raise QmbError("qmb200_gait_schedule failed: " + lib.qmb200_last_error(None).decode())
    return ev, md, n


class GaitSchedule:
    """ocs2::legged_robot::GaitSchedule as QMInterface::loadGaitSchedule builds it (QMInterface.cpp:455-480): stateful host object, one per robot."""

    def __init__(self, interface=None):
        self.lib = _lib.load_library(); self.interface = interface or QMInterface(); g = C.c_void_p()
        if self.lib.qmb200_gait_create(self.interface.taskFile.encode(), self.interface.referenceFile.encode(), C.byref(g)) != 0:
            raise QmbError("qmb200_gait_create failed: " + self.lib.qmb200_last_error(None).decode())
        self.g = g

    def __del__(self):
        try:
            self.lib.qmb200_gait_destroy(self.g)
        except Exception:
            pass

    def insertModeSequenceTemplate(self, gait_name, startTime, finalTime, gait_file=None):
        if self.lib.qmb200_gait_insert_template(self.g, (gait_file or self.interface.gaitFile).encode(), gait_name.encode(), float(startTime), float(finalTime)) != 0:
            raise QmbError("qmb200_gait_insert_template failed: " + self.lib.qmb200_last_error(None).decode())

    def getModeSchedule(self, lowerBoundTime, upperBoundTime):
        ev = np.zeros(EMAX); md = np.full(EMAX + 1, 15, dtype=np.int32)
        n = self.lib.qmb200_gait_get_mode_schedule(self.g, float(lowerBoundTime), float(upperBoundTime), _p(ev), _p(md))
        if n < 0:
            raise QmbError("qmb200_gait_get_mode_schedule failed: " + self.lib.qmb200_last_error(None).decode())
        return ev, md, n
