"""Live parity against MuJoCo itself -- auto-enabled when `import mujoco` succeeds (SURVEY.md 8c, oracle plan (ii)).

MuJoCo 2.3.2 is not installable in the build image (no wheel, no network), so in this repo's own runs every test
below SKIPS and the oracle stays "parity unpinned" (oracle/mjc_oracle.c header, DESIGN.md section 5).  On a machine
that has `mujoco` and the reference's MJCF tree these tests pin the three layers in turn:

  1. the MJCF mini-compiler (mycobotgym_b200/mjcf.py) against MuJoCo's compiled mjModel, field by field;
  2. the CPU oracle's mj_forward / mj_step against MuJoCo's, from injected (qpos, qvel, ctrl, qacc_warmstart);
  3. nothing GPU-side: the CUDA engine is compared with the oracle in tests/test_gpu_parity.py.

The MJCF tree is looked up in $MYCOBOT_ASSETS, an installed `mycobotgym` package, or baseline/_ref.
Mesh geoms do not collide in the oracle (documented gap), so the stepping comparison disables their contype /
conaffinity on the MuJoCo side -- that isolates the gap instead of hiding it: `test_mesh_contacts_are_the_gap`
reports how often the unmodified model produces a mesh contact on the same states.
"""
import os
import random

import numpy as np
import pytest

mujoco = pytest.importorskip("mujoco", reason="MuJoCo is not installable in this image; parity stays unpinned")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _assets_dir():
    cands = [os.environ.get("MYCOBOT_ASSETS"), os.path.join(ROOT, "baseline", "_ref", "mycobotgym", "envs", "assets")]
    try:
        import mycobotgym  # noqa: F401  (needs gymnasium + glfw at import time, usually absent)

        cands.insert(1, os.path.join(os.path.dirname(mycobotgym.__file__), "envs", "assets"))
    except Exception:
        pass
    for c in cands:
        if c and os.path.exists(os.path.join(c, "mycobot280.xml")):
            return c
    pytest.skip("reference MJCF tree not found (set MYCOBOT_ASSETS)")


@pytest.fixture(scope="module", params=["mycobot280.xml", "mycobot280_mocap.xml"])
def pair(request):
    from mycobotgym_b200 import mjcf

    path = os.path.join(_assets_dir(), request.param)
    mjm = mujoco.MjModel.from_xml_path(path)
    return mjm, mjcf.compile_mjcf(path), mjcf.flatmodel_from_mjmodel(mjm)


def test_mini_compiler_matches_mjmodel(pair):
    from mycobotgym_b200 import mjcf

    mjm, ours, live = pair
    diff = mjcf.diff_flatmodels(ours, live, rtol=1e-9)
    diff.pop("M0", None)                      # derived; compared through the inertias below
    for k in ("hull_vert", "hull_vertnum", "hull_vertadr", "hull_center", "hull_rbound"):
        diff.pop(k, None)                     # hull vertex order / count may differ (qhull options, float32 mesh storage): compared as point sets below
    assert not diff, diff
    assert ours["nhull"] == live["nhull"]
    for h in range(int(ours["nhull"])):
        a = ours["hull_vert"][ours["hull_vertadr"][h]:ours["hull_vertadr"][h] + ours["hull_vertnum"][h]]
        b = live["hull_vert"][live["hull_vertadr"][h]:live["hull_vertadr"][h] + live["hull_vertnum"][h]]
        d_ab = np.sqrt(((a[:, None, :] - b[None, :, :]) ** 2).sum(-1))
        assert d_ab.min(1).max() < 1e-5 and d_ab.min(0).max() < 1e-5, (ours["hull_names"][h], d_ab.min(1).max(), d_ab.min(0).max())
        np.testing.assert_allclose(ours["hull_center"][h], live["hull_center"][h], atol=1e-6)


def test_reference_keyframes_are_equilibria_of_mujoco():
    """The premise of tests/test_keyframe_equilibria.py (the oracle's weld rows were chosen so that the mocap keyframe is an
    equilibrium): MuJoCo itself must be at rest there, and must rest the cube 1.9e-5 m deep."""
    path = os.path.join(_assets_dir(), "mycobot280_mocap.xml")
    mjm = mujoco.MjModel.from_xml_path(path)
    mjd = mujoco.MjData(mjm)
    mujoco.mj_resetDataKeyframe(mjm, mjd, 0)
    mujoco.mj_forward(mjm, mjd)
    assert np.abs(mjd.qacc[:6]).max() < 0.5, mjd.qacc[:6]
    for _ in range(3000):
        mujoco.mj_step(mjm, mjd)
    tcp = mujoco.mj_name2id(mjm, mujoco.mjtObj.mjOBJ_BODY, "gripper_tcp")
    off = mjd.xpos[tcp] - mjd.mocap_pos[0]
    assert abs(np.linalg.norm(off) - 1.1486e-3) < 2e-5, off
    assert abs(mjd.qpos[14] - 0.209981) < 1e-6, mjd.qpos[14]


def _no_mesh_contacts(mjm):
    import copy

    m2 = copy.copy(mjm)
    for g in range(m2.ngeom):
        if m2.geom_type[g] == mujoco.mjtGeom.mjGEOM_MESH:
            m2.geom_contype[g] = 0
            m2.geom_conaffinity[g] = 0
    return m2


def _random_state(rng, mjm, flat):
    q = np.array(mjm.qpos0)
    q[:6] = rng.uniform(-1.0, 1.0, 6)
    g = rng.uniform(0.0, 0.6)
    q[6:12] = [g, g, g, g, g, -g]             # respects the gripper's closed-loop equalities
    q[12:14] = rng.uniform(-0.1, 0.1, 2)
    v = np.zeros(mjm.nv)
    v[:6] = rng.uniform(-0.5, 0.5, 6)
    return q, v


def test_oracle_step_matches_mujoco(pair):
    from oracle.oracle import OracleSim

    mjm, ours, live = pair
    mjm = _no_mesh_contacts(mjm)
    d = mujoco.MjData(mjm)
    sim = OracleSim(live)
    rng = np.random.default_rng(0)
    for trial in range(20):
        q, v = _random_state(rng, mjm, live)
        ctrl = rng.uniform(-1, 1, mjm.nu)
        mujoco.mj_resetData(mjm, d)
        d.qpos[:], d.qvel[:], d.ctrl[:] = q, v, ctrl
        mujoco.mj_forward(mjm, d)
        sim.set_state(q, v, ctrl, np.zeros(mjm.nv))
        if mjm.nmocap:
            sim.mocap_pos[:], sim.mocap_quat[:] = d.mocap_pos[0], d.mocap_quat[0]
        sim.forward()
        np.testing.assert_allclose(sim.xpos, d.xpos, atol=1e-12)
        np.testing.assert_allclose(sim.qacc_smooth, d.qacc_smooth, rtol=1e-8, atol=1e-8)
        assert sim.nefc == d.nefc, (trial, sim.nefc, d.nefc)
        np.testing.assert_allclose(sim.qacc, d.qacc, rtol=1e-6, atol=1e-6)
        sim.set_state(q, v, ctrl, np.array(d.qacc_warmstart))
        for _ in range(20):
            mujoco.mj_step(mjm, d)
        sim.step(20)
        np.testing.assert_allclose(sim.qpos, d.qpos, atol=1e-7, err_msg=f"trial {trial}")
        np.testing.assert_allclose(sim.qvel, d.qvel, atol=1e-5, err_msg=f"trial {trial}")


def test_mesh_contacts_are_the_gap(pair):
    """How often does the UNMODIFIED reference model put a mesh geom in contact on the benchmark's state distribution?"""
    mjm, ours, live = pair
    d = mujoco.MjData(mjm)
    rng = np.random.default_rng(1)
    random.seed(1)
    hits = 0
    for trial in range(200):
        q, v = _random_state(rng, mjm, live)
        mujoco.mj_resetData(mjm, d)
        d.qpos[:], d.qvel[:] = q, v
        mujoco.mj_forward(mjm, d)
        for c in range(d.ncon):
            con = d.contact[c]
            if mjm.geom_type[con.geom1] == mujoco.mjtGeom.mjGEOM_MESH or mjm.geom_type[con.geom2] == mujoco.mjtGeom.mjGEOM_MESH:
                hits += 1
                break
    print(f"states with at least one mesh contact: {hits}/200")
    assert hits <= 200
