"""Reference of the feedback policy (useFeedbackPolicy) built independently of both solvers' projection and Riccati code.

The gain of node k is the derivative of the optimal input step du_k with respect to the state step dx_k in the QP the tick solves.  Here it is read off the
tail QP from node k - dynamics, state-input equality rows, stage and final costs exactly as the oracle exports them (orc_mpc_qp) - solved as ONE sparse
KKT system with dx_k as a parameter: 30 right-hand sides, no constraint projection, no Riccati recursion.  The controller then follows
multiple_shooting::toPrimalSolution with feedback [upstream ocs2_oc, recalled]: uff_k = u*_k - K_k x*_k, and a pre-event node and the last node repeat the
bias and gain of the node before them."""
import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla


def _tail_kkt(qp, k):
    """Sparse KKT matrix of the tail QP from node k and the index maps of its variables."""
    N = qp["n_nodes"] - 1; nodes = list(range(k, N + 1)); ev = qp["is_event"]
    xi = {j: 30 * i for i, j in enumerate(nodes)}; off = 30 * len(nodes); ui = {}
    for j in range(k, N):
        if not ev[j]:
            ui[j] = off; off += 30
    nz = off; H = sp.lil_matrix((nz, nz)); rows = []   # rows: list of (block of G, rhs key)
    for j in range(k, N):
        H[xi[j]:xi[j] + 30, xi[j]:xi[j] + 30] = qp["Q"][j]
        if j in ui:
            H[ui[j]:ui[j] + 30, ui[j]:ui[j] + 30] = qp["R"][j]; H[ui[j]:ui[j] + 30, xi[j]:xi[j] + 30] = qp["P"][j]; H[xi[j]:xi[j] + 30, ui[j]:ui[j] + 30] = qp["P"][j].T
    H[xi[N]:xi[N] + 30, xi[N]:xi[N] + 30] = qp["QN"]
    G = []; r = 0; eqs = []
    g0 = sp.lil_matrix((30, nz)); g0[:, xi[k]:xi[k] + 30] = np.eye(30); G.append(g0); eqs.append(("p", None, r)); r += 30
    for j in range(k, N):
        g = sp.lil_matrix((30, nz)); g[:, xi[j + 1]:xi[j + 1] + 30] = np.eye(30); g[:, xi[j]:xi[j] + 30] = -qp["A"][j]
        if j in ui:
            g[:, ui[j]:ui[j] + 30] = -qp["B"][j]
        G.append(g); eqs.append(("b", j, r)); r += 30
        if j in ui:
            ng = int(qp["ng"][j]); g = sp.lil_matrix((ng, nz)); g[:, xi[j]:xi[j] + 30] = qp["C"][j, :ng]; g[:, ui[j]:ui[j] + 30] = qp["D"][j, :ng]
            G.append(g); eqs.append(("e", j, r)); r += ng
    Gm = sp.vstack(G).tocsc(); K = sp.bmat([[H.tocsc(), Gm.T], [Gm, None]]).tocsc()
    return K, xi, ui, nz, r, eqs


def tail_solution(qp, k, dxk):
    """Affine tail QP from node k with dx_k = dxk: → du_k (the principle of optimality: equals the full QP's du_k when dxk is its dx_k)."""
    K, xi, ui, nz, m, eqs = _tail_kkt(qp, k); N = qp["n_nodes"] - 1
    rhs = np.zeros(nz + m)
    for j in range(k, N):
        rhs[xi[j]:xi[j] + 30] -= qp["q"][j]
        if j in ui:
            rhs[ui[j]:ui[j] + 30] -= qp["r"][j]
    rhs[xi[N]:xi[N] + 30] -= qp["qN"]
    for kind, j, r in eqs:
        if kind == "p":
            rhs[nz + r:nz + r + 30] = dxk
        elif kind == "b":
            rhs[nz + r:nz + r + 30] = qp["b"][j]
        else:
            ng = int(qp["ng"][j]); rhs[nz + r:nz + r + ng] = -qp["e"][j, :ng]
    z = spla.splu(K).solve(rhs)
    return z[ui[k]:ui[k] + 30]


def dense_gain(qp, k):
    """K_k = d du_k / d dx_k of the tail QP from node k (k must carry an input: not a pre-event interval)."""
    K, xi, ui, nz, m, eqs = _tail_kkt(qp, k)
    rhs = np.zeros((nz + m, 30)); rhs[nz:nz + 30] = np.eye(30)
    z = spla.splu(K).solve(rhs)
    return z[ui[k]:ui[k] + 30]


def controller_node(event, n, k):
    """Node whose bias and gain node k uses (pre-event and last nodes repeat the node before them), -1 when there is none."""
    s = k
    while s > 0 and (s == n - 1 or event[s] == 1):
        s -= 1
    return -1 if (s >= n - 1 or event[s] == 1) else s


def build_controller(event, x, u, gains):
    """Dense LinearController of one robot: event/x/u of its n nodes, gains {regular node: 30x30} → (bias[n, 30], gain[n, 30, 30])."""
    n = len(event); bias = np.zeros((n, 30)); gain = np.zeros((n, 30, 30))
    for k in range(n):
        s = controller_node(event, n, k)
        if s < 0:
            bias[k] = u[k]
        else:
            gain[k] = gains[s]; bias[k] = u[s] - gains[s] @ x[s]
    return bias, gain


def evaluate(oracle, t, event, x, bias, gain, event_times, modes, tq, xq):
    """evaluatePolicy(tq, xq) of the controller: the per-node inputs uff_k + K_k xq interpolated on the node times as the oracle's feed-forward policy does
    (bias and gain are interpolated with the same (index, alpha) pair, so interpolating the node values is the same map)."""
    v = bias + gain @ xq
    return oracle.evaluate_policy(t, event, x, v, event_times, modes, tq)
