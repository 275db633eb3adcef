"""Solver variants the reference's settings name besides the SqpMpc the controller runs (SURVEY 8f-3; include/qmb200.h: qmb200_mpc_set_solver).
IPM: ipm{} block (task.info:95-125) - on this OCP (no inequality terms) the Newton step of the SQP with the block's line-search thresholds.
DDP: ddp{} block (task.info:33-71) in its discrete-time form: nominal rollout, LQ along it, discrete Riccati, rollout line search on the penalty merit.
Both against the oracle's restatement of the same variant, per block at the tolerances of tests/_parity.py; plus solver-independent properties of the DDP step."""
import os
import re

import numpy as np
import pytest

from _parity import MPC_TOL, assert_traj

pytestmark = pytest.mark.gpu
REF_TASK = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_inputs", "task.info")


def _block(name):
    """numbers of one top-level block of the reference's task.info, read here independently of both parsers."""
    txt = open(REF_TASK).read(); m = re.search(r"(?m)^" + name + r"\s*\n\{(.*?)^\}", txt, re.S); body = m.group(1)
    return {k: float(v) for k, v in re.findall(r"(?m)^\s*(\w+)\s+([-+.\deE]+)\s*(?:;.*)?$", body)}


def _run(oracle, solver_name, config, B, dt=0.015, ticks=2):
    import qm_control_b200 as q
    from qm_control_b200 import synthetic
    s = q.Solver(batch=B, dt=dt); s.mpc_set_solver(solver_name); oracle.mpc_set(dt=dt, horizon=1.0)
    prob, _ = synthetic.make_batch(np.arange(B), config=config); prev = None; res = []
    for tick in range(ticks):
        if tick > 0:
            prob = dict(prob); prob["t0"] = prob["t0"] + 0.01; x0 = np.zeros((B, 30))
            for b in range(B):
                n = prev["n_nodes"][b]; ne = prob["n_events"][b]
                x0[b], _, _ = oracle.evaluate_policy(prev["t"][b, :n], prev["event"][b, :n], prev["x"][b, :n], prev["u"][b, :n], prob["event_times"][b, :ne], prob["modes"][b, :ne + 1], prob["t0"][b])
            prob["x0"] = x0
        out = s.mpc_solve(prob); ref = oracle.mpc_solve_batch(prob, s.nmax, prev=prev, nthreads=8); res.append((out, ref)); prev = ref; s.mpc_set_solution(ref)
    return s, prob, res


def test_ipm_variant_uses_the_ipm_block_and_matches_the_oracle(oracle):
    ipm = _block("ipm"); assert ipm["g_max"] == 10.0 and ipm["ipmIteration"] == 1
    try:
        oracle.mpc_set_solver(solver=1, iterations=int(ipm["ipmIteration"]), delta_tol=ipm["deltaTol"], g_max=ipm["g_max"], g_min=ipm["g_min"])
        s, prob, res = _run(oracle, "ipm", config=5, B=9)
        got = s.mpc_get_solver(); assert got == dict(solver=1, iterations=1, delta_tol=ipm["deltaTol"], g_max=ipm["g_max"], g_min=ipm["g_min"])
        for tick, (out, ref) in enumerate(res):
            assert np.all((out["status"] & ~16) == 0); np.testing.assert_array_equal(out["step_info"][:, 0], ref["dbg"][:, 0]); assert_traj(out, ref, MPC_TOL, tag="ipm tick %d" % tick)
    finally:
        sq = _block("sqp"); oracle.mpc_set_solver(solver=0, iterations=1, delta_tol=sq["deltaTol"], g_max=sq["g_max"], g_min=sq["g_min"])


def test_ddp_variant_matches_the_oracle_and_descends(oracle):
    ddp = _block("ddp"); ls = {"minStepLength": 1e-2, "maxStepLength": 1.0}; assert ddp["constraintPenaltyInitialValue"] == 20.0 and ddp["maxNumIterations"] == 1
    try:
        oracle.mpc_set_solver(solver=2, iterations=int(ddp["maxNumIterations"]), ddp_penalty=ddp["constraintPenaltyInitialValue"], ddp_min_step=ls["minStepLength"], ddp_max_step=ls["maxStepLength"])
        s, prob, res = _run(oracle, "ddp", config=5, B=9)
        for tick, (out, ref) in enumerate(res):
            assert np.all((out["status"] & ~16) == 0), np.unique(out["status"])
            np.testing.assert_array_equal(out["step_info"][:, 0], ref["dbg"][:, 0])                    # accepted step length
            assert_traj(out, ref, MPC_TOL, tag="ddp tick %d" % tick)                                   # observed 1e-12 on B200 (profiles/r02d_parity_levels.txt)
            acc = ref["dbg"][:, 0] > 0; assert acc.all()
            np.testing.assert_allclose(out["step_info"][acc, 1], ref["dbg"][acc, 4], rtol=1e-8, atol=1e-9)   # cost of the accepted rollout
            assert np.all(out["step_info"][:, 2] == 0.0)                                               # single shooting: the accepted trajectory is a rollout, no dynamics defect
            merit0 = ref["dbg"][:, 1] + 20.0 * np.sqrt(ref["dbg"][:, 3]); merit = out["step_info"][:, 1] + 20.0 * np.sqrt(out["step_info"][:, 3])
            assert np.all(merit < merit0), (merit, merit0)                                             # descent of the penalty merit
    finally:
        sq = _block("sqp"); oracle.mpc_set_solver(solver=0, iterations=1, delta_tol=sq["deltaTol"], g_max=sq["g_max"], g_min=sq["g_min"])
