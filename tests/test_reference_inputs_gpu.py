"""A handle created from byte-identical copies of the reference's own task.info / reference.info / robot.urdf (tests/golden/ref_inputs/) solves the same
tick, bit for bit, as the handle every other test creates from the derived assets/ files (tests/test_reference_inputs_cpu.py checks the parsed constants)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
REF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_inputs")


def test_tick_on_the_reference_files_is_bit_identical_to_the_assets():
    import qm_control_b200 as q
    from qm_control_b200 import synthetic
    B = 16; prob, wbc = synthetic.make_batch(np.arange(B), config=5, gait_file=os.path.join(REF, "gait.info"), task_file=os.path.join(REF, "task.info"), reference_file=os.path.join(REF, "reference.info"))
    prob_a, _ = synthetic.make_batch(np.arange(B), config=5)
    for k in prob:
        np.testing.assert_array_equal(prob[k], prob_a[k])                     # the synthetic batch itself reads initialState / defaultJointState / gait templates
    ref_if = q.QMInterface(taskFile=os.path.join(REF, "task.info"), urdfFile=os.path.join(REF, "robot.urdf"), referenceFile=os.path.join(REF, "reference.info"))
    outs = []
    for iface in (ref_if, None):
        s = q.Solver(iface, batch=B); cmd, status = s.tick(prob, prob["t0"] + 0.002, wbc["rbd"], wbc["period"]); sol = s.mpc_get_solution()
        outs.append((cmd, status, sol["x"], sol["u"], sol["n_nodes"]))
    assert np.all((outs[0][1] & ~(16 << 8)) == 0)
    for a, b in zip(*outs):
        assert np.array_equal(a, b)
