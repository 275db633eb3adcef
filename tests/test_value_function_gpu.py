"""Value function (createValueFunction) on the B200, through the C ABI.

dfdxx and dfdx are compared with the sparse tail-QP KKT reference of tests/_value_function_ref.py (built on the QP the oracle exports and the oracle's
linearization trajectory, nothing shared with the CUDA projection / Riccati code)."""
import numpy as np
import pytest

import _value_function_ref as vr
from _parity import MPC_TOL

pytestmark = pytest.mark.gpu

NMAX = 88


def _q():
    import qm_control_b200 as q
    from qm_control_b200 import synthetic
    return q, synthetic


def _assert_close(P, g, P_ref, g_ref, Pxbar_ref, tol, tag):
    err = vr.block_errors(P, g, P_ref, g_ref, Pxbar_ref); bad = {k: v for k, v in err.items() if not v < tol}
    assert not bad, "%s: per-block relative error above %.1e: %s" % (tag, tol, bad)


def _reference(oracle, prob, nodes, nmax=NMAX):
    """{k: (dfdxx, dfdx)} of robot 0 of prob at the oracle's last QP (the handle's iteration count), plus dict(xlin, n_nodes, iterations) of that QP."""
    qp = oracle.mpc_qp(prob, nmax); sol = oracle.mpc_solve_batch({k: v[:1] for k, v in prob.items()}, nmax, nthreads=1)
    v = dict(xlin=vr.linearization(qp, sol), n_nodes=qp["n_nodes"], iterations=int(sol["dbg"][0, 9]))
    return vr.value_function(qp, v["xlin"], nodes), v


def test_switch_off_is_unchanged():
    q, synthetic = _q(); B = 8
    prob, wbc = synthetic.make_batch(np.arange(B), config=5); t_eval = prob["t0"] + 0.002
    never = q.Solver(batch=B, dt=0.015); assert not never.mpc_get_value_function()          # OCS2's default; the shipped task.info does not set the key
    toggled = q.Solver(batch=B, dt=0.015); toggled.mpc_set_value_function(True); toggled.mpc_set_value_function(False); assert not toggled.mpc_get_value_function()
    for _ in range(2):
        c0 = never.tick(prob, t_eval, wbc["rbd"], wbc["period"]); c1 = toggled.tick(prob, t_eval, wbc["rbd"], wbc["period"])
        np.testing.assert_array_equal(c0[0], c1[0]); np.testing.assert_array_equal(c0[1], c1[1])
    assert never.launch_count == toggled.launch_count
    on = q.Solver(batch=B, dt=0.015); on.mpc_set_value_function(True)
    for _ in range(2):
        c2 = on.tick(prob, t_eval, wbc["rbd"], wbc["period"])
    np.testing.assert_array_equal(c0[0], c2[0]); np.testing.assert_array_equal(c0[1], c2[1]); assert on.launch_count == never.launch_count
    a = q.Solver(batch=B, dt=0.015).mpc_solve(prob); s_on = q.Solver(batch=B, dt=0.015); s_on.mpc_set_value_function(True); b = s_on.mpc_solve(prob)
    for k in a:                                                                                # storing does not perturb the solve
        np.testing.assert_array_equal(a[k], b[k])
    assert np.all(s_on.value_function(prob["t0"], prob["x0"])["valid"] == 1)
    v = never.value_function(prob["t0"], prob["x0"])
    assert np.all(v["valid"] == 0) and np.all(v["dfdx"] == 0.0) and np.all(v["dfdxx"] == 0.0)


@pytest.mark.parametrize("robot,solver", [(0, "sqp"), (1, "sqp"), (2, "sqp"), (1, "ipm")])      # stance, trot, flying trot; IPM on the same path
def test_node_values_match_the_tail_qp_reference(oracle, robot, solver):
    q, synthetic = _q(); oracle.mpc_set(dt=0.015, horizon=1.0); oracle.mpc_set_solver(0, iterations=1)
    prob, _ = synthetic.make_batch(np.array([robot]), config=5)
    s = q.Solver(batch=1, dt=0.015, max_nodes=NMAX); s.mpc_set_solver(solver); s.mpc_set_value_function(True)
    out = s.mpc_solve(prob); assert out["status"][0] & ~16 == 0, out["status"]
    n = int(out["n_nodes"][0]); t = out["t"][0, :n]; ev = out["event"][0, :n]
    pre = [k for k in range(1, n - 1) if ev[k] == 1]; mid = next(k for k in range(n // 2, n) if ev[k] == 0)
    # a post-event node shares its time with the pre-event node before it, and evaluation at that time lands on the pre-event node
    nodes = sorted(k for k in {0, mid, n - 2, n - 1} | ({pre[0], pre[0] - 1} if pre else set()) if ev[k] != 2)
    ref, v = _reference(oracle, prob, nodes); assert v["n_nodes"] == n
    for k in nodes:
        got = s.value_function(np.array([t[k]]), np.zeros((1, 30))); assert got["valid"][0] == 1
        P, g = ref[k]
        _assert_close(got["dfdxx"][0], got["dfdx"][0], P, g, P @ v["xlin"][k], MPC_TOL, "%s robot %d node %d" % (solver, robot, k))
        np.testing.assert_array_equal(got["dfdxx"][0], got["dfdxx"][0].T)


def test_evaluation_at_random_time_and_state(oracle):
    q, synthetic = _q(); oracle.mpc_set(dt=0.015, horizon=1.0); oracle.mpc_set_solver(0, iterations=1)
    prob, _ = synthetic.make_batch(np.array([2]), config=5)                                   # flying trot: pre / post-event nodes
    s = q.Solver(batch=1, dt=0.015, max_nodes=NMAX); s.mpc_set_value_function(True); out = s.mpc_solve(prob)
    n = int(out["n_nodes"][0]); t = out["t"][0, :n]; ev = out["event"][0, :n]; x = out["x"][0, :n]
    ref, _ = _reference(oracle, prob, range(n)); Ps = np.stack([ref[k][0] for k in range(n)]); gs = np.stack([ref[k][1] for k in range(n)])
    post = [k for k in range(1, n) if ev[k] == 2]; assert post
    rng = np.random.default_rng(4)
    times = list(rng.uniform(t[0], t[-1], 10)) + [t[post[0]] + 0.3 * (t[post[0] + 1] - t[post[0]]), t[post[-1]] + 0.7 * (t[post[-1] + 1] - t[post[-1]]),
                                                  t[post[0]], t[0] - 0.05, t[0], t[-1], t[-1] + 0.05]
    for tq in times:
        xq = x[min(int(np.searchsorted(t, tq)), n - 1)] + 0.01 * rng.normal(size=30)
        got = s.value_function(np.array([tq]), xq[None]); assert got["valid"][0] == 1
        P = vr.interpolate(t, Ps, tq); g = vr.interpolate(t, gs, tq) + P @ xq
        _assert_close(got["dfdxx"][0], got["dfdx"][0], P, g, P @ xq, MPC_TOL, "t=%.4f" % tq)


def test_lifecycle():
    q, synthetic = _q(); B = 4
    prob, _ = synthetic.make_batch(np.arange(B), config=5); tq = prob["t0"] + 0.03; x = prob["x0"]
    s = q.Solver(batch=B, dt=0.015); s.mpc_set_value_function(True); sol = s.mpc_solve(prob)
    assert np.all(s.value_function(tq, x)["valid"] == 1)
    s.mpc_set_solution(sol); v = s.value_function(tq, x); assert np.all(v["valid"] == 0) and np.all(v["dfdxx"] == 0.0) and np.all(v["dfdx"] == 0.0)
    s.mpc_solve(prob); assert np.all(s.value_function(tq, x)["valid"] == 1)
    s.mpc_reset(); assert np.all(s.value_function(tq, x)["valid"] == 0)
    s.mpc_solve(prob); s.mpc_set_value_function(False); s.mpc_solve(prob); assert np.all(s.value_function(tq, x)["valid"] == 0)   # the last solve ran without it
    # robot 1758 of the bench workload: NEG_DT | NOT_PD -> no value function; its neighbour has one
    ids = np.array([1758, 5]); s2 = q.Solver(batch=2, dt=0.01); s2.mpc_set_value_function(True); p2, _ = synthetic.make_batch(ids, config=4, horizon=1.0)
    out = s2.mpc_solve(p2); assert out["status"][0] & 8 and out["status"][0] & 64
    v2 = s2.value_function(p2["t0"] + 0.013, p2["x0"]); assert list(v2["valid"]) == [0, 1] and np.all(v2["dfdxx"][0] == 0.0) and np.max(np.abs(v2["dfdxx"][1])) > 0.0
    # DDP: selecting it turns the switch off, and it refuses the switch
    s.mpc_set_value_function(True); s.mpc_set_solver("ddp"); assert not s.mpc_get_value_function()
    with pytest.raises(q.QmbError):
        s.mpc_set_value_function(True)
    s.mpc_set_solver("sqp"); s.mpc_set_value_function(True); assert s.mpc_get_value_function()


def test_early_convergence_keeps_the_last_qp(oracle):
    """sqpIteration = 3: a robot whose loop ends early skips the later Riccati sweeps and keeps the value function of its last QP, re-centred on that QP's
    linearization: bit for bit what a solve stopped after that many iterations gives, and the reference built at that iterate."""
    q, synthetic = _q(); B = 9; oracle.mpc_set(dt=0.015, horizon=1.0)
    prob, _ = synthetic.make_batch(np.arange(B), config=5); tq = prob["t0"] + 0.1; x = prob["x0"] + 0.01
    s = q.Solver(batch=B, dt=0.015); s.mpc_set_value_function(True); s.mpc_set_iterations(3); out = s.mpc_solve(prob); v3 = s.value_function(tq, x)
    assert np.all(v3["valid"] == 1)
    runs = {}
    for j in (1, 2):
        sj = q.Solver(batch=B, dt=0.015); sj.mpc_set_value_function(True); sj.mpc_set_iterations(j); sj.mpc_solve(prob); runs[j] = sj.value_function(tq, x)
    early = np.nonzero(out["status"] & 32)[0]
    for b in early:                                                                            # equal to the run that stopped where it stopped
        assert any(np.array_equal(v3["dfdxx"][b], runs[j]["dfdxx"][b]) and np.array_equal(v3["dfdx"][b], runs[j]["dfdx"][b]) for j in (1, 2)), b
    try:
        oracle.mpc_set_solver(0, iterations=3)
        for b in list(early[:2]) + list(np.nonzero((out["status"] & 32) == 0)[0][:1]):
            pb = {k: v[b:b + 1] for k, v in prob.items()}; n = int(out["n_nodes"][b]); tb = out["t"][b, :n]
            i, a = vr.time_segment(tb, tq[b]); ref, v = _reference(oracle, pb, [i, i + 1])
            assert (v["iterations"] < 3) == (b in early), (b, v["iterations"])
            P = a * ref[i][0] + (1 - a) * ref[i + 1][0]; g = a * ref[i][1] + (1 - a) * ref[i + 1][1] + P @ x[b]
            _assert_close(v3["dfdxx"][b], v3["dfdx"][b], P, g, P @ x[b], 10 * MPC_TOL, "3 iterations robot %d (%d run)" % (b, v["iterations"]))
    finally:
        oracle.mpc_set_solver(0, iterations=1)


def test_full_batch_and_pipeline(oracle):
    q, synthetic = _q(); B = 8192
    prob, _ = synthetic.make_batch(np.arange(B), config=4, horizon=1.0)
    big = q.Solver(batch=B, dt=0.01); big.mpc_set_value_function(True); out = big.mpc_solve(prob)
    sel = np.sort(np.random.default_rng(5).choice(B, 64, replace=False)); sel[0] = 1758
    small = q.Solver(batch=len(sel), dt=0.01); small.mpc_set_value_function(True); ps, _ = synthetic.make_batch(sel, config=4, horizon=1.0); small.mpc_solve(ps)
    rng = np.random.default_rng(6); tq = prob["t0"] + rng.uniform(-0.02, 1.05, B); x = prob["x0"] + 0.01 * rng.normal(size=(B, 30))
    vb = big.value_function(tq, x); vs = small.value_function(tq[sel], x[sel])
    for k in vb:                                                                               # independent of the batch position
        np.testing.assert_array_equal(vb[k][sel], vs[k])
    np.testing.assert_array_equal(vb["valid"], ((out["status"] & (2 | 4 | 8 | 64)) == 0).astype(np.int32)); assert vb["valid"][1758] == 0
    oracle.mpc_set(dt=0.01, horizon=1.0); oracle.mpc_set_solver(0, iterations=1)
    try:
        for b in sel[1:4]:                                                                     # a seeded sub-sample against the reference
            pb = {k: v[b:b + 1] for k, v in prob.items()}; n = int(out["n_nodes"][b]); tb = out["t"][b, :n]
            i, a = vr.time_segment(tb, tq[b]); ref, _ = _reference(oracle, pb, [i, min(i + 1, n - 1)], nmax=big.nmax)
            P = a * ref[i][0] + (1 - a) * ref[min(i + 1, n - 1)][0]; g = a * ref[i][1] + (1 - a) * ref[min(i + 1, n - 1)][1] + P @ x[b]
            _assert_close(vb["dfdxx"][b], vb["dfdx"][b], P, g, P @ x[b], MPC_TOL, "batch robot %d" % b)
    finally:
        oracle.mpc_set(dt=0.015, horizon=1.0)
    # qmb200_set_pipeline(4): the same ticks, bit for bit
    B2 = 16; p3, w3 = synthetic.make_batch(np.arange(B2), config=4); t3 = p3["t0"] + 0.002
    one = q.Solver(batch=B2, dt=0.015); one.mpc_set_value_function(True); four = q.Solver(batch=B2, dt=0.015); four.mpc_set_value_function(True); four.set_pipeline(4)
    for _ in range(2):
        a = one.tick(p3, t3, w3["rbd"], w3["period"]); b = four.tick(p3, t3, w3["rbd"], w3["period"])
        np.testing.assert_array_equal(a[0], b[0])
        va = one.value_function(t3 + 0.01, p3["x0"]); vb4 = four.value_function(t3 + 0.01, p3["x0"])
        for k in va:
            np.testing.assert_array_equal(va[k], vb4[k])


def test_cpp_mirror_returns_the_c_abi_value_function(tmp_path):
    import os
    import subprocess
    q, synthetic = _q(); root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    prob, _ = synthetic.make_batch(np.array([1]), config=5)
    s = q.Solver(batch=1, dt=0.015); s.mpc_set_value_function(True); s.mpc_solve(prob)
    xq = prob["x0"][0] + 0.01; tq = float(prob["t0"][0] + 0.02); ref = s.value_function(np.array([tq]), xq[None])
    src = tmp_path / "vf.cpp"; exe = tmp_path / "vf"
    ev = ", ".join("%.17g" % v for v in prob["event_times"][0, :prob["n_events"][0]]); md = ", ".join(str(int(v)) for v in prob["modes"][0, :prob["n_events"][0] + 1])
    tt = ", ".join("%.17g" % v for v in prob["target_times"][0, :prob["n_target"][0]])
    ts = ", ".join("qm::vector_t{" + ", ".join("%.17g" % v for v in prob["target_states"][0, k]) + "}" for k in range(prob["n_target"][0]))
    src.write_text('#include <cstdio>\n#include <stdexcept>\n#include "qmb200.hpp"\nint main() {\n'
                   '  qm::QMInterface itf("%s", "%s", "%s"); auto solver = std::make_shared<qm::Solver>(itf, 1, 0, QMB200_WBC_HIERARCHICAL, 0.0, 0.015);\n'
                   '  qm::SqpMpc mpc(solver);\n'
                   '  try { mpc.getValueFunction(%.17g, qm::vector_t{%s}); return 2; } catch (const std::runtime_error&) {}\n'
                   '  mpc.setValueFunction(true);\n'
                   '  qm::ModeSchedule ms{{%s}, {%s}}; qm::TargetTrajectories tt{{%s}, {%s}}; qm::vector_t x0{%s}, xq{%s};\n'
                   '  mpc.run(%.17g, x0, ms, tt); qm::ValueFunction v = mpc.getValueFunction(%.17g, xq); if (v.f != 0.0) return 3;\n'
                   '  for (double e : v.dfdx) std::printf("%%.17g\\n", e); for (double e : v.dfdxx) std::printf("%%.17g\\n", e);\n'
                   '  mpc.reset(); try { mpc.getValueFunction(%.17g, xq); return 4; } catch (const std::runtime_error&) {}\n'
                   '  return 0; }\n'
                   % (s.interface.taskFile, s.interface.urdfFile, s.interface.referenceFile, tq, ", ".join("%.17g" % v for v in xq), ev, md, tt, ts,
                      ", ".join("%.17g" % v for v in prob["x0"][0]), ", ".join("%.17g" % v for v in xq), prob["t0"][0], tq, tq))
    lib = os.path.join(root, "qm_control_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(root, "include"), str(src), "-o", str(exe), "-L", lib, "-lqmb200", "-Wl,-rpath," + lib])
    got = np.array([float(v) for v in subprocess.check_output([str(exe)]).split()])
    np.testing.assert_array_equal(got[:30], ref["dfdx"][0]); np.testing.assert_array_equal(got[30:], ref["dfdxx"][0].ravel())
