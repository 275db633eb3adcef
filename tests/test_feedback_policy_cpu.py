"""Feedback policy (useFeedbackPolicy) on the CPU: the reference the GPU tests compare against (tests/_feedback_ref.py) and the public surface.

The gain reference is the sparse KKT system of the tail QP the oracle exports (orc_mpc_qp).  Here it is pinned against the oracle's own QP step (principle
of optimality) and against the structure every feedback gain of this OCP must have; the GPU file compares the CUDA controller with it."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from qm_control_b200 import synthetic
import _feedback_ref as fr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NMAX = 88


def _nodes(qp, event):
    """k = 0, the first post-event node, a mid-horizon node and N - 1 (all carry an input)."""
    N = qp["n_nodes"] - 1; post = int(np.nonzero(event[:N] == 2)[0][0])
    mid = N // 2
    while qp["is_event"][mid]:
        mid += 1
    return [0, post, mid, N - 1]


@pytest.mark.parametrize("robot", [1, 2])          # trot, flying trot
def test_dense_tail_kkt_reproduces_the_oracle_step_and_the_gain_structure(oracle, robot):
    oracle.mpc_set(dt=0.015, horizon=1.0); prob, _ = synthetic.make_batch(np.array([robot]), config=5)
    qp = oracle.mpc_qp(prob, NMAX); sol = oracle.mpc_solve_batch(prob, NMAX, nthreads=1); n = int(sol["n_nodes"][0]); event = sol["event"][0, :n]
    assert qp["n_nodes"] == n
    for k in _nodes(qp, event):
        assert not qp["is_event"][k]
        du = fr.tail_solution(qp, k, qp["dx"][k])                                           # tail QP from k at the full QP's dx_k
        np.testing.assert_allclose(du, qp["du"][k], rtol=0, atol=1e-8 * (1.0 + np.max(np.abs(qp["du"][k]))))
        K = fr.dense_gain(qp, k); ng = int(qp["ng"][k])
        assert np.max(np.abs(qp["C"][k, :ng] + qp["D"][k, :ng] @ K)) < 1e-8 * (1.0 + np.max(np.abs(qp["C"][k, :ng])))   # the equality rows hold for every dx_k
        # the affine part: du_k(dx_k) = du_k(0) + K dx_k
        np.testing.assert_allclose(fr.tail_solution(qp, k, np.zeros(30)) + K @ qp["dx"][k], qp["du"][k], rtol=0, atol=1e-8 * (1.0 + np.max(np.abs(qp["du"][k]))))
        mode = prob["modes"][0, int(np.searchsorted(prob["event_times"][0, :prob["n_events"][0]], sol["t"][0, k], side="right"))]
        for f in range(4):                                                                   # zero-force rows of swing legs (contact order LF, RF, LH, RH)
            if not (mode >> (3 - f)) & 1:
                assert np.all(np.abs(K[3 * f:3 * f + 3]) < 1e-12), (k, f)
        assert np.max(np.abs(K)) > 1e-3                                                      # not the trivial gain


def test_controller_copy_rules_and_evaluation(oracle):
    oracle.mpc_set(dt=0.015, horizon=1.0); prob, _ = synthetic.make_batch(np.array([2]), config=5)
    sol = oracle.mpc_solve_batch(prob, NMAX, nthreads=1); n = int(sol["n_nodes"][0]); t = sol["t"][0, :n]; ev = sol["event"][0, :n]; x = sol["x"][0, :n]; u = sol["u"][0, :n]
    u = u.copy(); u[n - 1] = u[n - 2]
    rng = np.random.default_rng(3); gains = {k: rng.normal(size=(30, 30)) for k in range(n - 1) if ev[k] != 1}
    bias, gain = fr.build_controller(ev, x, u, gains)
    pre = [k for k in range(1, n - 1) if ev[k] == 1]; assert pre
    for k in pre + [n - 1]:                                                                 # pre-event and last nodes copy the previous node's bias and gain
        s = k - 1 if ev[k - 1] != 1 else k - 2
        np.testing.assert_array_equal(gain[k], gain[s]); np.testing.assert_array_equal(bias[k], bias[s])
    ne = int(prob["n_events"][0]); et = prob["event_times"][0, :ne]; md = prob["modes"][0, :ne + 1]
    for k in [0, 5, n // 2]:                                                                 # at x*(t_k) of a regular node the policy returns u*_k
        if ev[k] != 0:
            continue
        _, ud, _ = fr.evaluate(oracle, t, ev, x, bias, gain, et, md, t[k], x[k])
        np.testing.assert_allclose(ud, u[k], rtol=0, atol=1e-9 * (1.0 + np.max(np.abs(u[k]))))
    zb, zg = fr.build_controller(ev, x, u, {k: np.zeros((30, 30)) for k in gains})           # zero gain: the feed-forward policy
    for tq in [t[0], t[3] + 0.004, t[n - 1] + 0.1]:
        xd, ud, mode = fr.evaluate(oracle, t, ev, x, zb, zg, et, md, tq, rng.normal(size=30))
        xd0, ud0, mode0 = oracle.evaluate_policy(t, ev, x, u, et, md, tq)
        np.testing.assert_allclose(ud, ud0, rtol=0, atol=1e-12); np.testing.assert_array_equal(xd, xd0); assert mode == mode0


def test_library_exports_the_feedback_entry_points():
    from qm_control_b200 import _lib
    lib = C.CDLL(_lib.LIB_PATH)
    for name in ("qmb200_mpc_set_feedback_policy", "qmb200_mpc_get_feedback_policy", "qmb200_policy_eval_state", "qmb200_policy_eval_state_dev",
                 "qmb200_mpc_get_controller", "qmb200_mpc_get_controller_dev"):
        getattr(lib, name)


def test_cpp_mirror_compiles_with_the_feedback_overloads(tmp_path):
    src = tmp_path / "fb.cpp"
    src.write_text('#include "qmb200.hpp"\n'
                   'void f(qm::SqpMpc& m) { qm::vector_t x(30), xs, us; size_t mode = 0; m.setFeedbackPolicy(true); m.evaluatePolicy(0.1, x, xs, us, mode);\n'
                   '  m.evaluatePolicy(0.1, xs, us, mode); qm::LinearController c = m.getLinearController(); (void)c.timeStamp; (void)c.biasArray; (void)c.gainArray; }\n'
                   'int main() { return 0; }\n')
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)])
