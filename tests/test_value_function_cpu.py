"""Value function (createValueFunction) on the CPU: the reference the GPU tests compare against (tests/_value_function_ref.py).

The reference reads P_k, p_k off the sparse KKT system of the tail QP the oracle exports.  Here it is pinned twice: against central differences of that tail
QP's optimal cost (exact for a quadratic up to round-off) and against the oracle's own QP step (the model of node k at the step's dx_k is the step's cost from
node k on)."""
import numpy as np
import pytest

from qm_control_b200 import synthetic
import _value_function_ref as vr

NMAX = 88


def _qp(oracle, robot):
    oracle.mpc_set(dt=0.015, horizon=1.0); oracle.mpc_set_solver(0, iterations=1)
    prob, _ = synthetic.make_batch(np.array([robot]), config=5)
    return prob, oracle.mpc_qp(prob, NMAX)


def _nodes(qp):
    """0, the first post-event node, the first pre-event node, a middle node, N - 1 and N (the event nodes where the horizon has any)."""
    N = qp["n_nodes"] - 1; pre = [k for k in range(1, N) if qp["is_event"][k]]
    return sorted({0, N // 2, N - 1, N} | ({pre[0], pre[0] + 1} if pre else set()))


@pytest.mark.parametrize("robot", [1, 2])          # trot, flying trot
def test_reference_is_the_derivative_of_the_tail_qp_cost(oracle, robot):
    _, qp = _qp(oracle, robot); rng = np.random.default_rng(robot)
    nodes = _nodes(qp); assert any(qp["is_event"][k] for k in nodes)
    for k in nodes:
        P, p = vr.cost_to_go(qp, k); E = np.eye(30)
        pairs = [tuple(rng.choice(30, 2, replace=False)) for _ in range(24)]
        dxs = [np.zeros(30)] + [s * E[i] for i in range(30) for s in (1.0, -1.0)] + [si * E[i] + sj * E[j] for i, j in pairs for si in (1.0, -1.0) for sj in (1.0, -1.0)]
        J = vr.optimal_costs(qp, k, np.array(dxs)); J0 = J[0]; Jd = J[1:61].reshape(30, 2); Jp = J[61:].reshape(len(pairs), 2, 2)
        scale = max(1.0, abs(J0), np.max(np.abs(P)))
        np.testing.assert_allclose(0.5 * (Jd[:, 0] - Jd[:, 1]), p, rtol=0, atol=1e-9 * scale)                   # quadratic: h = 1 is exact but for round-off
        np.testing.assert_allclose(Jd[:, 0] + Jd[:, 1] - 2.0 * J0, np.diag(P), rtol=0, atol=1e-9 * scale)
        mixed = 0.25 * (Jp[:, 0, 0] - Jp[:, 0, 1] - Jp[:, 1, 0] + Jp[:, 1, 1])
        np.testing.assert_allclose(mixed, [P[i, j] for i, j in pairs], rtol=0, atol=1e-9 * scale)
        assert np.max(np.abs(P - P.T)) <= 1e-10 * np.max(np.abs(P))
        assert np.min(np.linalg.eigvalsh(0.5 * (P + P.T))) >= -1e-10 * np.max(np.abs(P)), k


@pytest.mark.parametrize("robot", [0, 1, 2])       # stance, trot, flying trot
def test_reference_reproduces_the_oracle_qp_step(oracle, robot):
    """The quadratic model of node k, evaluated at the oracle's own QP step dx_k, is the cost of that step from node k on (principle of optimality);
    and the linearization recovered from the oracle's step is its cold-start guess (every node at x0)."""
    prob, qp = _qp(oracle, robot); sol = oracle.mpc_solve_batch(prob, NMAX, nthreads=1); n = qp["n_nodes"]
    assert int(sol["n_nodes"][0]) == n and sol["dbg"][0, 9] == 1 and sol["dbg"][0, 0] > 0.0
    xlin = vr.linearization(qp, sol)
    np.testing.assert_allclose(xlin, np.broadcast_to(prob["x0"][0], xlin.shape), rtol=0, atol=1e-12 * (1.0 + np.max(np.abs(prob["x0"]))))
    for k in _nodes(qp):
        P, p = vr.cost_to_go(qp, k); dx = qp["dx"][k]; J0 = vr.optimal_costs(qp, k, np.zeros(30))[0]
        model = 0.5 * dx @ P @ dx + p @ dx + J0; c = vr.step_cost(qp, k)
        assert abs(model - c) <= 1e-9 * max(1.0, abs(c), abs(J0)), (robot, k, model, c)
        assert np.max(np.abs(P)) > 1e-3 and np.min(np.linalg.eigvalsh(0.5 * (P + P.T))) >= -1e-10 * np.max(np.abs(P))


def test_interpolation_follows_the_policy_time_segment():
    t = np.array([0.0, 0.1, 0.2, 0.2, 0.3]); v = np.arange(5.0)
    assert vr.interpolate(t, v, -1.0) == 0.0 and vr.interpolate(t, v, 0.0) == 0.0 and vr.interpolate(t, v, 0.4) == 4.0
    assert vr.interpolate(t, v, 0.05) == pytest.approx(0.5) and vr.interpolate(t, v, 0.25) == pytest.approx(3.5)
    assert vr.interpolate(t, v, 0.2) == 2.0                                         # lower bound lands on the first of the two nodes at 0.2
