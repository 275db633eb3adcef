"""The PRODUCT's host parser (csrc/host/qm_config.cpp) on the reference's own input files.

Every other test feeds the derived files under assets/ (tools/make_assets.py: comments stripped, the unused ddp / ipm / rollout blocks and the visual /
collision / gazebo elements dropped).  Here byte-identical copies of the reference's task.info, reference.info, gait.info and robot.urdf
(tests/golden/ref_inputs/, md5 pinned below) go through the same parser — host only, no GPU — and must produce the same model + settings block,
byte for byte, that is replicated to every GPU; the oracle's own parser must agree on the quantities both expose."""
import ctypes as C
import hashlib
import os

import numpy as np

from qm_control_b200 import _lib

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(HERE, "golden", "ref_inputs")
MD5 = {"task.info": "47e417bf5dea44b5bcb85f43dc792c4f", "reference.info": "650b9c7f61c223c013eed33f58389054", "gait.info": "ad3bcc5374db06f6ff8b20eba56a0b59",
       "robot.urdf": "2438ccb67bb3b37781c4cd7f6bf56919"}   # of the files in skywoodsz/qm_control @ 67247bb


def _blob(task, urdf, reference, gains=None, dt=0.0):
    lib = _lib.load_library()
    cfg = _lib.Config(task.encode(), urdf.encode(), reference.encode(), gains.encode() if gains else None, 1, 0, 0.0, dt, 0, 0)
    n = lib.qmb200_debug_model_blob(C.byref(cfg), None, 0)
    assert n > 0, lib.qmb200_last_error(None).decode()
    buf = (C.c_ubyte * n)(); assert lib.qmb200_debug_model_blob(C.byref(cfg), buf, n) == n
    return bytes(buf)


def test_fixture_files_are_the_reference_files():
    for name, md5 in MD5.items():
        assert hashlib.md5(open(os.path.join(REF, name), "rb").read()).hexdigest() == md5, name


def test_product_parser_gives_identical_constants_on_the_reference_files():
    ref = _blob(os.path.join(REF, "task.info"), os.path.join(REF, "robot.urdf"), os.path.join(REF, "reference.info"))
    ass = _blob(_lib.asset("qm_task.info"), _lib.asset("qm_robot.urdf"), _lib.asset("qm_reference.info"))
    assert len(ref) == len(ass) > 10000
    if ref != ass:
        a = np.frombuffer(ref, dtype=np.uint8); b = np.frombuffer(ass, dtype=np.uint8); bad = np.nonzero(a != b)[0]
        raise AssertionError("model blocks differ at %d bytes, first offsets %s" % (len(bad), bad[:8]))
    # the dt override of qmb200_config reaches the block (so the comparison above is not vacuous)
    assert _blob(os.path.join(REF, "task.info"), os.path.join(REF, "robot.urdf"), os.path.join(REF, "reference.info"), dt=0.01) != ref


def test_oracle_parser_agrees_on_the_reference_files():
    from _oracle import Oracle, GAINS
    o_ref = Oracle(os.path.join(REF, "robot.urdf"), os.path.join(REF, "task.info"), os.path.join(REF, "reference.info"), GAINS); o_ass = Oracle()
    ia, ib = o_ref.model_info(), o_ass.model_info()
    assert abs(ia["mass"] - 27.371574) < 1e-6 and ia["mass"] == ib["mass"]                       # SURVEY Appendix B: total mass of robot.urdf
    np.testing.assert_array_equal(ia["effort"], ib["effort"])
    Qa, Ra = o_ref.mpc_weights(); Qb, Rb = o_ass.mpc_weights(); np.testing.assert_array_equal(Qa, Qb); np.testing.assert_array_equal(Ra, Rb)


def test_gait_templates_of_the_reference_file_match_the_asset():
    """gait.info feeds the mode schedules (QMInterface.cpp:444-480): every template of the original file tiles to the same schedule as the asset's."""
    lib = _lib.load_library()
    for gait in ("stance", "trot", "flying_trot", "standing_trot", "pace", "standing_pace", "dynamic_walk", "static_walk", "amble", "lindyhop", "skipping", "pawup"):
        out = []
        for path in (os.path.join(REF, "gait.info"), _lib.asset("qm_gait.info")):
            ev = np.zeros(_lib.EMAX); md = np.zeros(_lib.EMAX + 1, dtype=np.int32)
            n = lib.qmb200_gait_schedule(path.encode(), gait.encode(), C.c_double(10.0), C.c_double(11.0), C.c_double(13.0), ev.ctypes.data_as(_lib.dp), md.ctypes.data_as(_lib.ip))
            out.append((n, ev.copy(), md.copy()))
        if out[0][0] < 0 and out[1][0] < 0:
            continue                                            # a template neither file defines
        assert out[0][0] == out[1][0] > 0, gait
        np.testing.assert_array_equal(out[0][1], out[1][1]); np.testing.assert_array_equal(out[0][2], out[1][2])
