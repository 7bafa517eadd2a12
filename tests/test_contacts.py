"""Contact output without a GPU: the geom names and sizes the C header and the Python side share, and the oracle's restatement of
mj_contactForce (tests/contact_oracle.py), whose decoded forces must reproduce the contacts' share of qfrc_constraint."""
import os
import re

import numpy as np
import pytest

from mycobotgym_b200 import _lib, flatten, mjcf
from oracle.oracle import OracleEnv, OracleSim

from contact_oracle import contact_forces, generalized_force, slots, world_force

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _header_define(name):
    with open(_lib.HDR) as f:
        m = re.search(rf"#define {name} (\d+)", f.read())
    return int(m.group(1))


@pytest.mark.parametrize("path", [mjcf.COMPILED_JOINT, mjcf.COMPILED_MOCAP])
def test_geom_names_match_the_compiled_model(path):
    fm = mjcf.load_compiled(path)
    assert int(fm["ngeom"]) == flatten.NGEOM == len(flatten.GEOM_NAMES)
    for g, name in enumerate(flatten.GEOM_NAMES):
        own, body = str(fm["geom_names"][g]), str(fm["body_names"][fm["geom_bodyid"][g]])
        if own:
            assert own == name
        elif body == "world":
            assert name == "floor" and fm["geom_type"][g] == 0       # the ground plane
        else:
            assert body == name                                       # the table's unnamed box
    desc = flatten.reduce_model(fm)
    assert [desc.geom_finger_r, desc.geom_finger_l, desc.geom_object] == [flatten.GEOM_NAMES.index(n) for n in
                                                                          ("right_finger_layer", "left_finger_layer", "object0")]


def test_sizes_and_exports_match_the_header():
    assert _header_define("MCB_MAXCON") == flatten.MAXCON == 24
    assert _header_define("MCB_CONTACT_DOUBLES") == flatten.CONTACT_DOUBLES == 1 + 3 + 9 + 6
    with open(_lib.HDR) as f:
        assert "int32_t mcb_set_contact_output(" in f.read()
    assert "mcb_set_contact_output" in _lib.EXPORTS


def _grasp_sim(fm):
    g = np.load(os.path.join(GOLDEN, "grasp_pick_sparse.npz"))
    s = OracleSim(fm)
    s.set_state(g["qpos0"], g["qvel0"], g["ctrl0"], g["warm0"])
    s.forward()
    return s


def _settled_cube_sim(fm, steps=40):
    e = OracleEnv(fm, has_object=True, reward_type="sparse")
    e.reset(object_xy=np.array([0.05, -0.03]), goal=np.array([0.0, 0.0, 0.3]))
    for _ in range(steps):
        e.step(np.zeros(7, dtype=np.float32))
    e.sim.forward()
    return e.sim


def _check_identity(s):
    cons = contact_forces(s)
    assert cons
    J, f, t = s.efc("J"), s.efc("force"), s.efc("type")
    other = np.flatnonzero(t != 2)                           # equality and limit rows
    expected = np.array(s.qfrc_constraint) - J[other].T @ f[other]
    got = generalized_force(s, cons)
    scale = max(1.0, np.abs(expected).max())
    np.testing.assert_allclose(got, expected, rtol=0, atol=1e-10 * scale)
    return cons


def test_decoded_forces_reproduce_qfrc_constraint_in_a_grasp():
    fm = mjcf.load_compiled()
    s = _grasp_sim(fm)
    cons = _check_identity(s)
    names = [(flatten.GEOM_NAMES[c["geom1"]], flatten.GEOM_NAMES[c["geom2"]]) for c in cons]
    assert any("right_finger_layer" in n and "object0" in n for n in names)
    assert any("left_finger_layer" in n and "object0" in n for n in names)
    assert any(c["dim"] == 4 and abs(c["force"][3]) > 0 for c in cons) or all(c["dim"] == 3 for c in cons)


def test_decoded_forces_reproduce_qfrc_constraint_for_a_cube_on_the_table():
    fm = mjcf.load_compiled()
    s = _settled_cube_sim(fm)
    cons = _check_identity(s)
    cube = flatten.GEOM_NAMES.index("object0")
    on_cube = [c for c in cons if cube in (c["geom1"], c["geom2"])]
    assert len(on_cube) >= 3
    # a resting cube: the contact forces on it carry its weight, and the frame is orthonormal with the normal first
    F = sum(world_force(c) * (1.0 if c["geom2"] == cube else -1.0) for c in on_cube)
    m = float(fm["body_mass"][list(fm["body_names"]).index("object0")])
    g = float(-np.asarray(fm["gravity"])[2])
    assert abs(F[2] - m * g) < 0.02 * m * g, (F, m * g)
    for c in on_cube:
        np.testing.assert_allclose(c["frame"] @ c["frame"].T, np.eye(3), atol=1e-12)
        assert c["force"][0] >= 0 and np.all(c["force"][c["dim"]:] == 0)


def test_decoded_forces_use_the_mixed_friction_of_a_baked_model():
    # the mixed friction comes from the (baked) model: a friction multiplier on the cube changes mu of its pairs
    fm = mjcf.load_compiled()
    p = np.ones(flatten.NPARAM)
    p[flatten.P_FRICTION + flatten.GEOM_NAMES.index("object0")] = 1.7
    fm2 = flatten.apply_params_flat(fm, p)
    s = _grasp_sim(fm2)
    cons = _check_identity(s)
    fr = np.asarray(fm2["geom_friction"])
    for c in cons:
        assert c["friction"][0] == max(fr[c["geom1"], 0], fr[c["geom2"], 0])


def test_slots_layout():
    fm = mjcf.load_compiled()
    cons = contact_forces(_grasp_sim(fm))
    sl = slots(cons)
    n = sl["ncon"]
    assert n == len(cons) and np.all(sl["geom"][n:] == -1) and np.all(sl["dim"][n:] == 0) and not sl["force"][n:].any()
    assert np.array_equal(sl["dim"][:n], [c["dim"] for c in cons])
