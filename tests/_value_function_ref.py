"""Reference of the value function (createValueFunction) built independently of both solvers' projection and Riccati code.

The value function of node k is the optimal cost of the tail QP from node k as a function of the state step dx_k: 1/2 dx_k' P_k dx_k + p_k' dx_k + const.
The tail QP is the one tests/_feedback_ref.py builds from the QP the oracle exports (orc_mpc_qp), with the rows x_k = dx_k as the parameter.  With the
multiplier lam of those rows, dJ/d dx_k = -lam, so ONE sparse solve with 31 right-hand sides (dx_k = 0 and the 30 unit vectors of the parameter alone) gives
p_k = -lam(0) and P_k = -d lam / d dx_k.  No projection, no Riccati.  SqpSolver::extractValueFunction [upstream ocs2_sqp, recalled] then stores
dfdxx_k = P_k and dfdx_k = p_k - P_k xbar_k, where xbar is the linearization trajectory of that QP."""
import numpy as np
import scipy.sparse.linalg as spla

from _feedback_ref import _tail_kkt
from _parity import X_BLOCKS


def tail_system(qp, k):
    """KKT matrix of the tail QP from node k, its size nz, the right-hand side with dx_k = 0 and the row offset of the x_k = dx_k rows."""
    K, xi, ui, nz, m, eqs = _tail_kkt(qp, k); N = qp["n_nodes"] - 1
    rhs = np.zeros(nz + m); prow = None
    for j in range(k, N):
        rhs[xi[j]:xi[j] + 30] -= qp["q"][j]
        if j in ui:
            rhs[ui[j]:ui[j] + 30] -= qp["r"][j]
    rhs[xi[N]:xi[N] + 30] -= qp["qN"]
    for kind, j, r in eqs:
        if kind == "p":
            prow = nz + r
        elif kind == "b":
            rhs[nz + r:nz + r + 30] = qp["b"][j]
        else:
            ng = int(qp["ng"][j]); rhs[nz + r:nz + r + ng] = -qp["e"][j, :ng]
    return K, nz, rhs, prow


def cost_to_go(qp, k):
    """(P_k, p_k) of the tail QP from node k: minus the multiplier of the x_k = dx_k rows at dx_k = 0 and its sensitivity."""
    K, nz, rhs0, prow = tail_system(qp, k)
    rhs = np.zeros((len(rhs0), 31)); rhs[:, 0] = rhs0; rhs[prow:prow + 30, 1:] = np.eye(30)
    z = spla.splu(K).solve(rhs); lam = z[prow:prow + 30]
    return -lam[:, 1:], -lam[:, 0]


def optimal_costs(qp, k, dxs):
    """Optimal cost 1/2 z'Hz + g'z of the tail QP from node k for each row of dxs (the central-difference check of cost_to_go)."""
    K, nz, rhs0, prow = tail_system(qp, k); dxs = np.atleast_2d(dxs)
    rhs = np.repeat(rhs0[:, None], len(dxs), axis=1); rhs[prow:prow + 30] = dxs.T
    z = spla.splu(K).solve(rhs)[:nz]; H = K[:nz, :nz]; g = -rhs0[:nz]
    return 0.5 * np.einsum("ij,ij->j", z, H @ z) + g @ z


def value_function(qp, xlin, nodes):
    """{k: (dfdxx_k, dfdx_k)} for the given nodes: dfdxx = P_k, dfdx = p_k - P_k xbar_k."""
    out = {}
    for k in nodes:
        P, p = cost_to_go(qp, k); out[k] = (P, p - P @ xlin[k])
    return out


def time_segment(times, tq):
    """ocs2::LinearInterpolation::timeSegment: (index, alpha) with value = alpha v[index] + (1 - alpha) v[index + 1]; clamped outside the time stamps."""
    n = len(times)
    if n <= 1:
        return 0, 1.0
    part = int(np.searchsorted(times, tq, side="left")); idx = part - 1 if (part != 0 or tq != times[0]) else 0; last = n - 1
    if idx < 0:
        return 0, 1.0
    if idx >= last:
        return max(last - 1, 0), 0.0
    ln = times[idx + 1] - times[idx]; till = times[idx + 1] - tq
    return idx, (till / ln if ln > 2.0 * np.finfo(float).eps else (1.0 if till > 0.5 * ln else 0.0))


def interpolate(times, values, tq):
    """Per-node arrays interpolated on the node times as getValueFunction interpolates dfdxx and dfdx."""
    i, a = time_segment(times, tq)
    return a * values[i] + (1.0 - a) * values[min(i + 1, len(times) - 1)]


def block_errors(P, g, P_ref, g_ref, Pxbar_ref):
    """Worst relative error per block of like quantities: dfdxx per (row block, column block) of X_BLOCKS scaled by max(1, |block|); dfdx per block scaled
    by the larger of |p| and |P xbar| (the two terms it is the difference of) and the block's floor."""
    worst = {}
    for rn, (r0, r1, _) in X_BLOCKS.items():
        for cn, (c0, c1, _) in X_BLOCKS.items():
            ref = P_ref[r0:r1, c0:c1]
            worst["P " + rn + "/" + cn] = np.max(np.abs(P[r0:r1, c0:c1] - ref)) / max(1.0, np.max(np.abs(ref)))
        p_ref = g_ref[r0:r1] + Pxbar_ref[r0:r1]
        worst["dfdx " + rn] = np.max(np.abs(g[r0:r1] - g_ref[r0:r1])) / max(X_BLOCKS[rn][2], np.max(np.abs(p_ref)), np.max(np.abs(Pxbar_ref[r0:r1])))
    return worst


def linearization(qp, sol):
    """Linearization trajectory of the oracle's last QP for robot 0 of an mpc_solve_batch result: the solution before that QP's step,
    x = xbar + alpha dx (takeStep; alpha = 0 when no step was taken)."""
    n = qp["n_nodes"]
    return sol["x"][0, :n] - sol["dbg"][0, 0] * qp["dx"][:n]


def step_cost(qp, k):
    """Cost of the oracle's QP step (qp["dx"], qp["du"]) from node k on: the tail QP's objective at its optimum when dx_k is the step's dx_k."""
    N = qp["n_nodes"] - 1; dx = qp["dx"]; du = qp["du"]; c = 0.0
    for j in range(k, N):
        c += 0.5 * dx[j] @ qp["Q"][j] @ dx[j] + qp["q"][j] @ dx[j]
        if not qp["is_event"][j]:
            c += 0.5 * du[j] @ qp["R"][j] @ du[j] + du[j] @ qp["P"][j] @ dx[j] + qp["r"][j] @ du[j]
    return c + 0.5 * dx[N] @ qp["QN"] @ dx[N] + qp["qN"] @ dx[N]
