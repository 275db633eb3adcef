"""Feedback policy (useFeedbackPolicy) on the B200, through the C ABI.

The gains are compared with the sparse tail-QP KKT reference of tests/_feedback_ref.py (built on the QP the oracle exports, nothing shared with the CUDA
projection / Riccati code) and with central differences of the CUDA solve itself."""
import numpy as np
import pytest

import _feedback_ref as fr
from _parity import MPC_TOL, TICK_TOL, U_BLOCKS, assert_cmd, block_errors

pytestmark = pytest.mark.gpu

NMAX = 88


def _q():
    import qm_control_b200 as q
    from qm_control_b200 import synthetic
    return q, synthetic


def _regular(ev, n):
    return [k for k in range(n - 1) if ev[k] != 1]


def _assert_blocks(out, ref, tol, tag):
    lv = block_errors(out, ref, U_BLOCKS); bad = {k: v for k, v in lv.items() if not v < tol}
    assert not bad, "%s: per-block relative error above %.1e: %s" % (tag, tol, bad)


def test_switch_off_is_unchanged():
    q, synthetic = _q(); B = 8
    prob, wbc = synthetic.make_batch(np.arange(B), config=5)
    s = q.Solver(batch=B, dt=0.015); assert not s.mpc_get_feedback_policy()          # the shipped task.info says false
    s.mpc_solve(prob); rng = np.random.default_rng(0); tq = prob["t0"] + rng.uniform(0.0, 1.1, B); x = rng.normal(size=(B, 30))
    a = s.policy_eval(tq); b = s.policy_eval_state(tq, x)
    for u, v in zip(a, b):
        np.testing.assert_array_equal(u, v)
    never = q.Solver(batch=B, dt=0.015); toggled = q.Solver(batch=B, dt=0.015); toggled.mpc_set_feedback_policy(True); toggled.mpc_set_feedback_policy(False)
    t_eval = prob["t0"] + 0.002; c0 = never.tick(prob, t_eval, wbc["rbd"], wbc["period"]); c1 = toggled.tick(prob, t_eval, wbc["rbd"], wbc["period"])
    np.testing.assert_array_equal(c0[0], c1[0]); np.testing.assert_array_equal(c0[1], c1[1]); assert never.launch_count == toggled.launch_count
    on = q.Solver(batch=B, dt=0.015); on.mpc_set_feedback_policy(True); on.tick(prob, t_eval, wbc["rbd"], wbc["period"])
    assert on.launch_count == never.launch_count                                       # one policy launch either way


@pytest.mark.parametrize("robot,solver", [(0, "sqp"), (1, "sqp"), (2, "sqp"), (1, "ipm")])      # stance, trot, flying trot; IPM on the same path
def test_controller_matches_the_tail_qp_reference(oracle, robot, solver):
    q, synthetic = _q(); oracle.mpc_set(dt=0.015, horizon=1.0); oracle.mpc_set_solver(0, iterations=1)
    prob, _ = synthetic.make_batch(np.array([robot]), config=5)
    s = q.Solver(batch=1, dt=0.015, max_nodes=NMAX); s.mpc_set_solver(solver); s.mpc_set_feedback_policy(True)
    out = s.mpc_solve(prob); c = s.mpc_get_controller()                                 # right after the GPU's own solve
    assert c["feedback"][0] == 1 and out["status"][0] & ~16 == 0, out["status"]
    qp = oracle.mpc_qp(prob, NMAX); ref = oracle.mpc_solve_batch(prob, NMAX, nthreads=1); n = int(ref["n_nodes"][0]); ev = ref["event"][0, :n]
    assert int(out["n_nodes"][0]) == n
    regular = _regular(ev, n); post = [k for k in regular if ev[k] == 2]
    check = sorted(set([0, post[0], n // 2 if ev[n // 2] != 1 else n // 2 + 1, n - 2 if ev[n - 2] != 1 else n - 3]))
    gains = {k: fr.dense_gain(qp, k) for k in check}
    for k in check:
        gk = c["gain"][0, k]; rk = gains[k]
        for name, (lo, hi, floor) in U_BLOCKS.items():                                  # force rows, leg-joint rows, arm rows
            err = np.max(np.abs(gk[lo:hi] - rk[lo:hi])) / max(1.0, np.max(np.abs(rk[lo:hi])))
            assert err < MPC_TOL, (solver, robot, k, name, err)
        kx = rk @ ref["x"][0, k]; bias_ref = ref["u"][0, k] - kx                         # uff = u* - K x*: scaled by the larger of |u*| and |K x*| per block
        for name, (lo, hi, floor) in U_BLOCKS.items():
            err = np.max(np.abs(c["bias"][0, k, lo:hi] - bias_ref[lo:hi])) / max(floor, np.max(np.abs(ref["u"][0, k, lo:hi])), np.max(np.abs(kx[lo:hi])))
            assert err < MPC_TOL, (solver, robot, k, "bias " + name, err)
    pre = [k for k in range(1, n - 1) if ev[k] == 1]
    for k in pre + [n - 1]:                                                              # the copy rule on the GPU's own export
        src = fr.controller_node(ev, n, k)
        np.testing.assert_array_equal(c["gain"][0, k], c["gain"][0, src]); np.testing.assert_array_equal(c["bias"][0, k], c["bias"][0, src])
    assert np.all(c["gain"][0, n:] == 0.0) and np.all(c["bias"][0, n:] == 0.0)


def test_policy_evaluation_matches_the_reference(oracle):
    q, synthetic = _q(); oracle.mpc_set(dt=0.015, horizon=1.0); oracle.mpc_set_solver(0, iterations=1)
    prob, _ = synthetic.make_batch(np.array([2]), config=5)                             # flying trot: pre / post-event nodes, swing legs
    s = q.Solver(batch=1, dt=0.015, max_nodes=NMAX); s.mpc_set_feedback_policy(True); s.mpc_solve(prob)
    qp = oracle.mpc_qp(prob, NMAX); ref = oracle.mpc_solve_batch(prob, NMAX, nthreads=1); n = int(ref["n_nodes"][0])
    t = ref["t"][0, :n]; ev = ref["event"][0, :n]; x = ref["x"][0, :n]; u = ref["u"][0, :n]
    gains = {k: fr.dense_gain(qp, k) for k in _regular(ev, n)}; bias, gain = fr.build_controller(ev, x, u, gains)
    ne = int(prob["n_events"][0]); et = prob["event_times"][0, :ne]; md = prob["modes"][0, :ne + 1]
    rng = np.random.default_rng(1); pre = [k for k in range(1, n - 1) if ev[k] == 1]
    times = list(rng.uniform(t[0], t[-1], 12)) + [t[pre[0]], t[pre[0] + 1], t[-1], t[-1] + 0.05, t[3]]
    for tq in times:
        xq = x[min(int(np.searchsorted(t, tq)), n - 1)] + 0.01 * rng.normal(size=30)
        xd, ud, mode = s.policy_eval_state(np.array([tq]), xq[None])
        xr, ur, mr = fr.evaluate(oracle, t, ev, x, bias, gain, et, md, tq, xq)
        assert int(mode[0]) == mr
        _assert_blocks(ud[0], ur, MPC_TOL, "policy t=%.4f" % tq)


def test_solve_is_affine_in_the_measured_state_with_slope_K0():
    """Warm start whose guess covers t0: the LQ model does not depend on x0, and with a full step u*_0 = u_guess_0 + du_0(x0) is affine in x0 with slope K_0.
    Robot 0 is the base point, robots 1 + 2i / 2 + 2i the central differences of component i - one batched solve."""
    q, synthetic = _q(); B = 61; h = 1e-3
    prob, _ = synthetic.make_batch(np.full(B, 1), config=5)                              # trot, the same robot B times
    s = q.Solver(batch=B, dt=0.015); s.mpc_set_feedback_policy(True); first = s.mpc_solve(prob)
    p2 = {k: v.copy() for k, v in prob.items()}; p2["t0"] = prob["t0"] + 0.005
    xq, _, _ = s.policy_eval(p2["t0"]); x0 = xq[0].copy()
    for i in range(30):
        p2["x0"][1 + 2 * i] = x0; p2["x0"][1 + 2 * i, i] += h; p2["x0"][2 + 2 * i] = x0; p2["x0"][2 + 2 * i, i] -= h
    p2["x0"][0] = x0
    out = s.mpc_solve(p2); c = s.mpc_get_controller(0, 1)
    assert np.all(out["step_info"][:, 0] == 1.0), out["step_info"][:, 0]
    K0 = c["gain"][0, 0]; fd = np.stack([(out["u"][1 + 2 * i, 0] - out["u"][2 + 2 * i, 0]) / (2 * h) for i in range(30)], axis=1)
    for name, (lo, hi, floor) in U_BLOCKS.items():
        err = np.max(np.abs(fd[lo:hi] - K0[lo:hi])) / max(1.0, np.max(np.abs(K0[lo:hi])))
        assert err < 1e-6, (name, err)
    assert first["n_nodes"][0] > 60


def test_tick_and_update_chains(oracle):
    q, synthetic = _q(); B = 4; oracle.mpc_set(dt=0.015, horizon=1.0); oracle.mpc_set_solver(0, iterations=1)
    prob, wbc = synthetic.make_batch(np.arange(B), config=4)
    s = q.Solver(batch=B, dt=0.015); s.mpc_set_feedback_policy(True); t_eval = prob["t0"] + 0.002
    cmd, status = s.tick(prob, t_eval, wbc["rbd"], wbc["period"]); assert np.all((status & 0xFF) == 0)
    ref = oracle.mpc_solve_batch(prob, s.nmax, nthreads=4); xd_r = np.zeros((B, 30)); ud_r = np.zeros((B, 30)); md_r = np.zeros(B, dtype=np.int32)
    for b in range(B):                                                                   # reference chain: controller at (t_eval, x0) -> WbcBase::update
        pb = {k: v[b:b + 1] for k, v in prob.items()}; qp = oracle.mpc_qp(pb, s.nmax); n = int(ref["n_nodes"][b])
        t = ref["t"][b, :n]; ev = ref["event"][b, :n]; x = ref["x"][b, :n]; u = ref["u"][b, :n]
        i = max(0, int(np.searchsorted(t, t_eval[b])) - 1); need = {fr.controller_node(ev, n, k) for k in range(max(0, i - 1), min(n, i + 3))} - {-1}
        bias, gain = fr.build_controller(ev, x, u, {k: (fr.dense_gain(qp, k) if k in need else np.zeros((30, 30))) for k in _regular(ev, n)})
        ne = int(prob["n_events"][b]); xd_r[b], ud_r[b], md_r[b] = fr.evaluate(oracle, t, ev, x, bias, gain, prob["event_times"][b, :ne], prob["modes"][b, :ne + 1], t_eval[b], prob["x0"][b])
    cmd_r, _ = oracle.wbc_update_batch(xd_r, ud_r, wbc["rbd"], md_r, wbc["period"], t_eval, np.zeros((B, 30)), nthreads=4)
    assert_cmd(cmd, cmd_r, TICK_TOL, tag="feedback tick")
    # three RT updates on the policy: observation -> evaluatePolicy(t_obs, x_obs) -> WBC -> control law, against the same chain through the separate entry points
    ctrl = q.Solver(batch=B, dt=0.015); ctrl.mpc_set_feedback_policy(True); ctrl.mpc_solve(prob); sep = q.Solver(batch=B, dt=0.015); sep.mpc_set_feedback_policy(True); sep.mpc_solve(prob)
    t_obs = prob["t0"].copy(); x_obs = prob["x0"].copy(); jc = np.zeros((B, 18, 5)); ap = np.zeros((B, 6)); lt = t_obs.copy(); st = (t_obs.copy(), x_obs.copy(), jc.copy(), ap.copy(), lt.copy())
    for _ in range(3):
        t_obs, x_obs, jc, ap, lt, cmd_u, _ = ctrl.update(wbc["rbd"], wbc["period"], t_obs, x_obs, jc, ap, lt)
        ts, xs = sep.observation_update(wbc["rbd"], wbc["period"], st[0], st[1]); xd, ud, md = sep.policy_eval_state(ts, xs)
        cw, _ = sep.wbc_update(xd, ud, wbc["rbd"], md, wbc["period"], ts); j2, a2, l2, _ = sep.control_law(xd, ud, cw, ts, xs, st[2], st[3], st[4]); st = (ts, xs, j2, a2, l2)
        np.testing.assert_array_equal(cmd_u, cw); np.testing.assert_array_equal(jc, j2)
    xf, uf, _ = ctrl.policy_eval(t_obs); xs_, us_, _ = ctrl.policy_eval_state(t_obs, x_obs + 0.01)
    assert np.max(np.abs(us_ - uf)) > 1e-6                                                # the policy does react to the state


def test_cpp_mirror_evaluates_the_feedback_policy(tmp_path):
    import os
    import subprocess
    q, synthetic = _q(); root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    prob, _ = synthetic.make_batch(np.array([1]), config=5)
    s = q.Solver(batch=1, dt=0.015); s.mpc_set_feedback_policy(True); s.mpc_solve(prob)
    xq = prob["x0"][0] + 0.01; tq = float(prob["t0"][0] + 0.02); _, ud, _ = s.policy_eval_state(np.array([tq]), xq[None])
    src = tmp_path / "m.cpp"; exe = tmp_path / "m"
    ev = ", ".join("%.17g" % v for v in prob["event_times"][0, :prob["n_events"][0]]); md = ", ".join(str(int(v)) for v in prob["modes"][0, :prob["n_events"][0] + 1])
    tt = ", ".join("%.17g" % v for v in prob["target_times"][0, :prob["n_target"][0]])
    ts = ", ".join("qm::vector_t{" + ", ".join("%.17g" % v for v in prob["target_states"][0, k]) + "}" for k in range(prob["n_target"][0]))
    src.write_text('#include <cstdio>\n#include "qmb200.hpp"\nint main() {\n'
                   '  qm::QMInterface itf("%s", "%s", "%s"); auto solver = std::make_shared<qm::Solver>(itf, 1, 0, QMB200_WBC_HIERARCHICAL, 0.0, 0.015);\n'
                   '  qm::SqpMpc mpc(solver); mpc.setFeedbackPolicy(true);\n'
                   '  qm::ModeSchedule ms{{%s}, {%s}}; qm::TargetTrajectories tt{{%s}, {%s}}; qm::vector_t x0{%s}, xq{%s};\n'
                   '  mpc.run(%.17g, x0, ms, tt); qm::vector_t xs, us; size_t mode = 0; mpc.evaluatePolicy(%.17g, xq, xs, us, mode);\n'
                   '  qm::LinearController c = mpc.getLinearController(); if (!c.feedback || c.gainArray.size() != c.timeStamp.size()) return 2;\n'
                   '  for (double v : us) std::printf("%%.17g\\n", v); return 0; }\n'
                   % (s.interface.taskFile, s.interface.urdfFile, s.interface.referenceFile, ev, md, tt, ts, ", ".join("%.17g" % v for v in prob["x0"][0]),
                      ", ".join("%.17g" % v for v in xq), prob["t0"][0], tq))
    lib = os.path.join(root, "qm_control_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(root, "include"), str(src), "-o", str(exe), "-L", lib, "-lqmb200", "-Wl,-rpath," + lib])
    got = np.array([float(v) for v in subprocess.check_output([str(exe)]).split()])
    np.testing.assert_array_equal(got, ud[0])


def test_fallbacks_to_the_feed_forward_policy():
    q, synthetic = _q(); B = 4
    prob, _ = synthetic.make_batch(np.arange(B), config=5); rng = np.random.default_rng(2)
    s = q.Solver(batch=B, dt=0.015); s.mpc_set_feedback_policy(True); sol = s.mpc_solve(prob)
    tq = prob["t0"] + 0.03; x = prob["x0"] + 0.01 * rng.normal(size=(B, 30))
    assert np.max(np.abs(s.policy_eval_state(tq, x)[1] - s.policy_eval(tq)[1])) > 1e-6
    s.mpc_set_solution(sol)                                                              # a loaded solution has no controller
    np.testing.assert_array_equal(s.policy_eval_state(tq, x)[1], s.policy_eval(tq)[1]); assert np.all(s.mpc_get_controller()["feedback"] == 0)
    s.mpc_solve(prob); assert np.all(s.mpc_get_controller()["feedback"] == 1)
    s.mpc_reset(); assert np.all(s.mpc_get_controller()["feedback"] == 0)
    # robot 1758 of the bench workload: NEG_DT | NOT_PD -> no gain; its policy is the feed-forward one bit for bit, its neighbour keeps the feedback
    ids = np.array([1758, 5]); s2 = q.Solver(batch=2, dt=0.01); s2.mpc_set_feedback_policy(True); p2, _ = synthetic.make_batch(ids, config=4, horizon=1.0)
    out = s2.mpc_solve(p2); assert out["status"][0] & 8 and out["status"][0] & 64
    c = s2.mpc_get_controller(); assert list(c["feedback"]) == [0, 1] and np.all(c["gain"][0] == 0.0)
    t2 = p2["t0"] + 0.013; x2 = p2["x0"] + 0.01; a = s2.policy_eval_state(t2, x2); b = s2.policy_eval(t2)
    np.testing.assert_array_equal(a[1][0], b[1][0]); assert np.max(np.abs(a[1][1] - b[1][1])) > 1e-6


def test_full_batch_and_pipeline_do_not_change_the_controller():
    q, synthetic = _q(); B = 8192
    prob, wbc = synthetic.make_batch(np.arange(B), config=4, horizon=1.0)
    big = q.Solver(batch=B, dt=0.01); big.mpc_set_feedback_policy(True); big.mpc_solve(prob)
    sel = np.sort(np.random.default_rng(5).choice(B, 64, replace=False)); sel[0] = 1758
    small = q.Solver(batch=len(sel), dt=0.01); small.mpc_set_feedback_policy(True); ps, _ = synthetic.make_batch(sel, config=4, horizon=1.0); small.mpc_solve(ps)
    cs = small.mpc_get_controller()
    for j, b in enumerate(sel[:16]):
        cb = big.mpc_get_controller(int(b), 1)
        np.testing.assert_array_equal(cb["gain"][0], cs["gain"][j]); np.testing.assert_array_equal(cb["bias"][0], cs["bias"][j]); assert cb["feedback"][0] == cs["feedback"][j]
    tq = prob["t0"] + 0.004; x = prob["x0"] + 0.005
    ub = big.policy_eval_state(tq, x)[1]; us = small.policy_eval_state(tq[sel], x[sel])[1]
    np.testing.assert_array_equal(ub[sel], us)
    # qmb200_set_pipeline(4): the same ticks, bit for bit
    B2 = 16; p3, w3 = synthetic.make_batch(np.arange(B2), config=4); t3 = p3["t0"] + 0.002
    one = q.Solver(batch=B2, dt=0.015); one.mpc_set_feedback_policy(True); four = q.Solver(batch=B2, dt=0.015); four.mpc_set_feedback_policy(True); four.set_pipeline(4)
    for _ in range(2):
        a = one.tick(p3, t3, w3["rbd"], w3["period"]); b = four.tick(p3, t3, w3["rbd"], w3["period"])
        np.testing.assert_array_equal(a[0], b[0]); np.testing.assert_array_equal(a[1], b[1])
