"""Model compiler + flattening (north-star subsystem 1) against the reference's own known answers."""
import ctypes
import os

import numpy as np
import pytest

from mycobotgym_b200 import flatten, mjcf

# MyCobotGym's MJCF tree (mycobotgym/envs/assets) is not part of this repository: set MYCOBOT_ASSETS to recompile it
REF_XML = os.path.join(os.environ["MYCOBOT_ASSETS"], "mycobot280.xml") if os.environ.get("MYCOBOT_ASSETS") else None


@pytest.fixture(scope="module")
def flat():
    return mjcf.load_compiled()


def test_sizes_match_reference_keyframe_lengths(flat):
    # qpos 19 / qvel 18 / ctrl 7 from the keyframe (mycobot280.xml:6-8); SURVEY A.1
    assert (flat.nq, flat.nv, flat.nu, flat.nbody, flat.njnt, flat.nsite, flat.neq) == (19, 18, 7, 25, 13, 3, 3)
    assert flat.nM == 86
    assert flat.key_qpos.shape == (1, 19) and flat.key_ctrl.shape == (1, 7)
    assert list(flat.dof_parentid) == [-1, 0, 1, 2, 3, 4, 5, 6, 5, 8, 5, 5, -1, 12, 13, 14, 15, 16]


def test_fk_known_answers(flat):
    # EEF at qpos0 == mocap body pos (mocap.xml:3); EEF at the keyframe == mpos (mycobot280_mocap.xml:8)
    s = flat.site_names.index("EEF")
    b = flat.site_bodyid[s]
    fk = mjcf.fk_numpy(flat, flat.qpos0)
    eef = fk[0][b] + fk[2][b] @ flat.site_pos[s]
    np.testing.assert_allclose(eef, [0.0138673, 0.01864658, 0.61236], atol=5e-9)
    fk = mjcf.fk_numpy(flat, flat.key_qpos[0])
    eef = fk[0][b] + fk[2][b] @ flat.site_pos[s]
    np.testing.assert_allclose(eef, [-0.05154491, 0.01053502, 0.3448586], atol=5e-9)
    q = fk[1][flat.body_names.index("gripper_tcp")]
    np.testing.assert_allclose(q, [0.01762876, -0.70526013, 0.0078235, 0.70868623], atol=5e-8)
    # reference known answer (SURVEY 8c (2)): at the keyframe the tool orientation is the fetch IK target [0, -0.707, 0, 0.707]
    # (mycobot.py:140) to two digits
    np.testing.assert_allclose(q, [0.0, -0.707, 0.0, 0.707], atol=0.02)


def test_mocap_keyframe_orientation_known_answer():
    # mycobot280_mocap.xml:8: the keyframe's mocap quaternion (0.50235287 -0.499 -0.5 0.49764296), composed with the weld's
    # relative pose, is the orientation of gripper_tcp at that keyframe's qpos -- an independent check of the FK rotations,
    # the weld relpose computed by the set_const restatement and the quaternion conventions
    fm = mjcf.load_compiled(mjcf.COMPILED_MOCAP)
    fk = mjcf.fk_numpy(fm, fm.key_qpos[0])
    tcp = fm.body_names.index("gripper_tcp")
    want = mjcf.quat_mul(fm.key_mquat[0], fm.eq_data[0, 6:10])
    got = fk[1][tcp]
    if np.dot(want, got) < 0:
        want = -want
    np.testing.assert_allclose(got, want, atol=5e-3)
    np.testing.assert_allclose(fk[0][tcp], fm.key_mpos[0], atol=2e-3)        # and the mocap body sits on the tool (weld at rest)


def test_classes_and_defaults(flat):
    # joint classes (mycobot280_main.xml:57-77)
    np.testing.assert_array_equal(flat.dof_armature[:6], 0.1)
    np.testing.assert_array_equal(flat.dof_damping[:6], 1.0)
    assert flat.dof_armature[6] == 0.005 and flat.dof_damping[6] == 0.1 and flat.dof_armature[7] == 0
    np.testing.assert_array_equal(flat.jnt_range[6], [0, 0.7])
    np.testing.assert_array_equal(flat.jnt_limited, [1] * 10 + [0, 0, 0])
    np.testing.assert_array_equal(flat.jnt_solref[6], [0.005, 1])
    np.testing.assert_array_equal(flat.jnt_solref[0], [0.02, 1])
    np.testing.assert_array_equal(flat.dof_damping[12:], 0.01)
    # actuators (joint_actuators.xml:3-22)
    np.testing.assert_array_equal(flat.actuator_gain, [4500, 4500, 3500, 2000, 2000, 2000, 70])
    np.testing.assert_array_equal(flat.actuator_forcerange[:, 1], [87, 87, 87, 12, 12, 12, 5])
    np.testing.assert_array_equal(flat.actuator_moment[6, [6, 8]], [0.5, 0.5])
    np.testing.assert_array_equal(flat.actuator_biasprm[6], [0, -100, -10])
    # cube (mycobot280_main.xml:260-265)
    assert abs(flat.body_mass[24] - 0.008) < 1e-15
    np.testing.assert_allclose(flat.body_inertia[24], 0.008 / 3 * 2e-4, rtol=1e-12)
    g = flat.geom_names.index("object0")
    np.testing.assert_array_equal(flat.geom_friction[g], [0.95, 0.3, 0.1])
    assert flat.geom_condim[g] == 4
    np.testing.assert_array_equal(flat.geom_solref[flat.geom_names.index("right_finger_layer")], [-20000, -500])


def test_setconst_products(flat):
    assert abs(flat.body_invweight0[24, 0] - 125.0) < 1e-9          # 1/m for the free cube
    assert abs(flat.dof_invweight0[12] - 125.0) < 1e-9
    assert np.all(flat.body_invweight0[:3] == 0)                     # static bodies
    assert 0.01 < flat.stat_meaninertia < 0.1
    # connect anchors coincide at qpos0
    fk = mjcf.fk_numpy(flat, flat.qpos0)
    for e in range(2):
        b1, b2 = flat.eq_obj1id[e], flat.eq_obj2id[e]
        p1 = fk[0][b1] + fk[2][b1] @ flat.eq_data[e, :3]
        p2 = fk[0][b2] + fk[2][b2] @ flat.eq_data[e, 3:6]
        np.testing.assert_allclose(p1, p2, atol=1e-15)
    M = flat.M0
    assert np.allclose(M, M.T) and np.all(np.linalg.eigvalsh(M) > 0)


@pytest.mark.skipif(not (REF_XML and os.path.exists(REF_XML)), reason="reference MJCF tree not found (set MYCOBOT_ASSETS)")
def test_committed_json_matches_recompile(flat):
    log = []
    fresh = mjcf.compile_mjcf(REF_XML, log)
    for k, v in fresh.items():
        if isinstance(v, np.ndarray):
            assert np.array_equal(flat[k], v), k
        elif k != "compile_log":
            assert flat[k] == v, k
    assert any("base_link" in line for line in log)  # documented deviation: mesh absent from the mount


def test_compiler_on_the_stored_mjcf_tree(tmp_path):
    """compile_mjcf end to end on tests/golden/mjcf_tree (an include tree with the constructs of the reference's model: default
    classes and childclass, box / mesh / explicit inertia, a missing mesh, duplicate mesh geoms, free and mocap bodies, exclude,
    fixed tendon, connect, keyframe) against answers worked out by hand from the XML, then through the JSON round trip."""
    log = []
    m = mjcf.compile_mjcf(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mjcf_tree", "model.xml"), log)
    assert (m.nq, m.nv, m.nbody, m.njnt, m.nu, m.nsite, m.neq, m.nmocap, m.ntendon, m.ngeom, m.nM) == (11, 10, 7, 5, 2, 1, 1, 1, 1, 5, 30)
    assert m.timestep == 0.004
    np.testing.assert_array_equal(m.body_parentid, [0, 0, 1, 2, 2, 0, 0])
    np.testing.assert_array_equal(m.body_weldid, [0, 1, 2, 3, 4, 5, 0])
    np.testing.assert_array_equal(m.body_rootid, [0, 1, 1, 1, 1, 5, 6])
    np.testing.assert_array_equal(m.body_mocapid, [-1, -1, -1, -1, -1, -1, 0])
    np.testing.assert_array_equal(m.dof_parentid, [-1, 0, 1, 1, -1, 4, 5, 6, 7, 8])
    np.testing.assert_array_equal(m.qpos0, [0, 0, 0, 0, 0.3, 0, 0.02, 1, 0, 0, 0])
    np.testing.assert_allclose(m.body_quat[2], [np.sqrt(0.5), 0, 0, np.sqrt(0.5)], atol=1e-15)
    # joint defaults: class "arm" on the links, "finger" (nested in "arm") on the fingers, built-ins on the free joint
    np.testing.assert_array_equal(m.jnt_axis[0], [0, 0, 1])
    np.testing.assert_array_equal(m.dof_armature, [0.1, 0.1, 0.005, 0.005, 0, 0, 0, 0, 0, 0])
    np.testing.assert_array_equal(m.dof_damping, [1, 1, 0.1, 0.1, 0, 0, 0, 0, 0, 0])
    np.testing.assert_array_equal(m.jnt_limited, [1, 1, 1, 1, 0])
    np.testing.assert_array_equal(m.jnt_range[[0, 2]], [[-3, 3], [0, 0.7]])
    np.testing.assert_array_equal(m.jnt_solref[[0, 2]], [[0.02, 1], [0.005, 1]])
    # masses: boxes at density 500 (pad_b's mass given), the cube mesh (side 0.04) at 500, the missing mesh and the density-0
    # copy add nothing; box inertia m/3 (b^2 + c^2) in decreasing order, cube m a^2 / 6 about its centroid
    np.testing.assert_allclose(m.body_mass, [0, 0.04, 0.032, 0.004, 0.02, 0.008, 0], rtol=1e-6)
    np.testing.assert_allclose(m.body_inertia[1], np.array([29, 26, 5]) * 1e-4 * 0.04 / 3, rtol=1e-12)
    np.testing.assert_allclose(m.body_inertia[2], [0.032 * 0.04 ** 2 / 6] * 3, rtol=1e-6)
    np.testing.assert_allclose(m.body_ipos[2], [0.03, 0, 0], atol=1e-9)
    np.testing.assert_allclose(m.body_inertia[3:6], [[0.004 / 3 * 2e-4] * 3, [0.02 / 3 * 2e-4] * 3, [1e-6] * 3], rtol=1e-12)
    np.testing.assert_allclose(m.body_subtreemass[:3], [0.104, 0.096, 0.056], rtol=1e-6)
    assert any("mesh gone: file missing" in line for line in log)
    # collision: plane / box geoms with their classes, one hull for the two cube geoms
    assert m.geom_names == ["floor", "box1", "pad_a", "pad_b", "object0"]
    np.testing.assert_array_equal(m.geom_friction[[1, 2]], [[1, 0.005, 0.0001], [0.95, 0.3, 0.1]])
    np.testing.assert_array_equal(m.geom_condim, [3, 3, 4, 4, 3])
    assert (m.nhull, list(m.hull_mult), list(m.hull_vertnum), m.hull_names) == (1, [2], [8], ["link2"])
    hv = m.hull_vert[np.lexsort(m.hull_vert.T)]
    want = np.array([[x, y, z] for z in (-0.02, 0.02) for y in (-0.02, 0.02) for x in (0.01, 0.05)])
    np.testing.assert_allclose(hv, want, atol=1e-9)
    np.testing.assert_allclose(m.hull_center[0], [0.03, 0, 0], atol=1e-9)
    np.testing.assert_allclose(m.hull_rbound, [0.02 * np.sqrt(3)], rtol=1e-6)
    # site, exclude, tendon, actuators, connect anchor 2 (set_const), keyframe
    fk = mjcf.fk_numpy(m, m.qpos0)
    np.testing.assert_allclose(fk[0][2] + fk[2][2] @ m.site_pos[0], [0.1, 0.05, 0.1], atol=1e-15)
    np.testing.assert_array_equal(m.exclude, [[1, 2]])
    np.testing.assert_array_equal(m.ten_J, [[0, 0, 0.5, 0.5, 0, 0, 0, 0, 0, 0]])
    np.testing.assert_array_equal(m.actuator_moment, [[1, 0, 0, 0, 0, 0, 0, 0, 0, 0], [0, 0, 1, 1, 0, 0, 0, 0, 0, 0]])
    np.testing.assert_array_equal(m.actuator_gain, [100, 70])
    np.testing.assert_array_equal(m.actuator_biasprm, [[0, -100, -10]] * 2)
    np.testing.assert_array_equal(m.actuator_forcelimited, [1, 0])
    np.testing.assert_array_equal(m.actuator_ctrlrange, [[-3, 3], [0, 0.7]])
    np.testing.assert_allclose(m.eq_data[0, :6], [0, 0.01, 0, 0, -0.01, 0], atol=1e-15)
    np.testing.assert_array_equal(m.key_qpos, [[0.1, -0.2, 0.3, 0.3, 0.3, 0, 0.02, 1, 0, 0, 0]])
    np.testing.assert_array_equal(m.key_ctrl, [[0.5, 0.2]])
    np.testing.assert_array_equal(m.key_mpos, [[0, 0, 0.5]])
    # set_const on the free body (centroid at its origin: translation and rotation decouple)
    np.testing.assert_allclose(m.M0[4:7, 4:7], 0.008 * np.eye(3), rtol=1e-12)
    np.testing.assert_allclose([m.body_invweight0[5, 0], m.dof_invweight0[4], m.dof_invweight0[7]], [125, 125, 1e6], rtol=1e-9)
    assert np.allclose(m.M0, m.M0.T) and np.all(np.linalg.eigvalsh(m.M0) > 0)
    # the committed assets are written and read through the same JSON + hull side file
    m.to_json(str(tmp_path / "model.json"))
    back = mjcf.FlatModel.from_json(str(tmp_path / "model.json"))
    assert mjcf.diff_flatmodels(m, back, rtol=0) == {} and back.compile_log == m.compile_log


def test_reduced_model_is_consistent(flat):
    d = flatten.reduce_model(flat)
    assert list(d.parent) == [-1, 0, 1, 2, 3, 4, 5, 6, 5, 8, 5, 5, -1]
    assert list(d.subtree_size) == [12, 11, 10, 9, 8, 7, 2, 1, 2, 1, 1, 1, 1]
    # merged masses conserve total mass per weld group
    total = sum(flat.body_mass[b] for b in range(flat.nbody) if flat.body_weldid[b] != 0)
    assert abs(sum(d.mass) - total) < 1e-15
    # link6 composite = link6 + flange + gripper_base
    names = flat.body_names
    m6 = sum(flat.body_mass[names.index(n)] for n in ("link6", "flange", "gripper_base"))
    assert abs(d.mass[5] - m6) < 1e-15
    assert d.npair == 9 and ctypes.sizeof(d) % 8 == 0
    # the composite inertia must reproduce M(qpos0) of the unmerged model: checked end-to-end on the GPU
    # (tests/test_gpu_parity.py) and here through a numpy CRBA on the reduced tree
    fk = mjcf.fk_numpy(flat, flat.qpos0)
    jb = [b for b in range(flat.nbody) if flat.body_jntnum[b] > 0]
    M = np.diag(np.array(d.armature[:]))
    for k, b in enumerate(jb):
        R, p = fk[2][b], fk[0][b]
        com = p + R @ np.array(d.ipos[k][:])
        I6 = np.array(d.inertia[k][:])
        Ib = np.array([[I6[0], I6[3], I6[4]], [I6[3], I6[1], I6[5]], [I6[4], I6[5], I6[2]]])
        jp, jr = mjcf.jac_point(flat, fk, b, com)
        M += d.mass[k] * jp.T @ jp + jr.T @ (R @ Ib @ R.T) @ jr
    np.testing.assert_allclose(M, flat.M0, atol=1e-16, rtol=1e-12)


@pytest.mark.parametrize("which", ["joint", "mocap"])
def test_live_mjmodel_loader_path_executes(which):
    """north_star subsystem 1 ("takes the reference's compiled mjModel"): `flatmodel_from_mjmodel` + `diff_flatmodels` + the
    flattening into the device descriptor, executed against an MjModel-shaped stand-in (tests/fake_mujoco.py)."""
    import ctypes

    import fake_mujoco
    from mycobotgym_b200 import flatten, mjcf

    compiled = mjcf.load_compiled(mjcf.COMPILED_MOCAP if which == "mocap" else mjcf.COMPILED_JOINT)
    mjm = fake_mujoco.model_from_flat(compiled)
    assert mjm.ngeom == compiled["ngeom"] + 2 * compiled["nhull"]   # two mesh geoms per robot body in the "live" model ...
    live = mjcf.flatmodel_from_mjmodel(mjm, mujoco=fake_mujoco)
    assert live["ngeom"] == compiled["ngeom"] and live["geom_names"] == compiled["geom_names"]      # ... become one hull each
    assert live["nhull"] == 14 and np.all(live["hull_mult"] == 2)
    assert mjcf.diff_flatmodels(compiled, live) == {}
    a, b = flatten.reduce_model(compiled), flatten.reduce_model(live)
    assert bytes(ctypes.string_at(ctypes.addressof(a), ctypes.sizeof(a))) == bytes(ctypes.string_at(ctypes.addressof(b), ctypes.sizeof(b)))
    # the diff tool does flag a wrong field
    live["body_mass"] = live["body_mass"] * 1.01
    assert "body_mass" in mjcf.diff_flatmodels(compiled, live)
