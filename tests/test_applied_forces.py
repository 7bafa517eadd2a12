"""Applied forces, host side: the oracle's restatement (zero forces are the plain step, J' xfrc is the virtual work of the wrench,
a force at the cube's centre of mass is the same generalized force on its translation dofs), the body table and the argument checks
of MyCobotVectorEnv.set_applied_forces."""
import numpy as np
import pytest
import torch

from applied_oracle import AppliedOracleSim, applied_oracle_env, set_engine_forces
from mycobotgym_b200 import flatten, mjcf
from oracle.oracle import OracleEnv

CONTROLLERS = [("joint", False, 7), ("IK", False, 7), ("mocap", False, 8)]


def _flat(ctrl="joint"):
    return mjcf.load_compiled(mjcf.COMPILED_MOCAP if ctrl == "mocap" else mjcf.COMPILED_JOINT)


def _pair(ctrl, fetch, seed):
    """A plain oracle and one with (zero) applied forces switched on, in the same reset state."""
    flat = _flat(ctrl)
    kw = dict(has_object=True, reward_type="dense", controller_type=ctrl, fetch_env=fetch, control_steps=2)
    a, b = OracleEnv(flat, **kw), applied_oracle_env(flat, **kw)
    a.reset(seed=seed)
    b.reset(seed=seed)
    b.sim.set_state(**a.sim.get_state())
    b.sim.mocap_pos[:], b.sim.mocap_quat[:] = a.sim.mocap_pos, a.sim.mocap_quat
    b.goal = a.goal.copy()
    a.sim.forward()
    b.sim.forward()
    b.sim.applied = True
    return a, b


@pytest.mark.parametrize("ctrl,fetch,adim", CONTROLLERS)
def test_zero_forces_are_the_plain_step(ctrl, fetch, adim):
    a, b = _pair(ctrl, fetch, 3)
    rng = np.random.default_rng(0)
    for _ in range(4):
        act = rng.uniform(-1, 1, adim).astype(np.float32)
        oa, ra, *_ = a.step(act)
        ob, rb, *_ = b.step(act)
        assert np.array_equal(oa["observation"], ob["observation"]) and ra == rb
        for x, y in ((a.sim.qpos, b.sim.qpos), (a.sim.qvel, b.sim.qvel), (a.sim.ctrl, b.sim.ctrl), (a.sim.qacc_warmstart, b.sim.qacc_warmstart)):
            assert np.array_equal(x, y)


def _posed_sim(seed):
    """An oracle sim at a random arm pose with the cube at a random pose, kinematics current."""
    flat = _flat()
    sim = AppliedOracleSim.attach(OracleEnv(flat, has_object=True).sim)
    rng = np.random.default_rng(seed)
    q = np.array(flat["qpos0"], dtype=np.float64)
    q[:12] += rng.uniform(-0.5, 0.5, 12)
    q[12:15] = rng.uniform(-0.3, 0.3, 3)
    quat = rng.normal(size=4)
    q[15:19] = quat / np.linalg.norm(quat)
    sim.qpos[:] = q
    sim.kinematics()
    return flat, sim


def _point(sim, b):
    return sim.xpos[b] + sim.xmat[b] @ sim.xfrc_point[b]


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_xfrc_is_the_virtual_work_of_the_wrench(seed):
    """F . dp/dq_j and tau . dtheta/dq_j by central differences of the application point p and of the body's orientation, over the
    twelve hinges and the cube's three translation dofs (qpos index == dof index there), for every jointed body."""
    flat, sim = _posed_sim(seed)
    rng = np.random.default_rng(100 + seed)
    jointed = [b for b in range(int(flat["nbody"])) if flat["body_jntnum"][b] > 0]
    q0 = sim.qpos.copy()
    h = 1e-6
    for b in jointed:
        w = rng.normal(size=6)
        sim.xfrc_applied[:] = 0
        sim.xfrc_applied[b] = w
        sim.qpos[:] = q0
        sim.kinematics()
        got = sim.applied_qfrc()
        R0 = sim.xmat[b].copy()
        for j in range(15):
            pts, mats = [], []
            for sgn in (1, -1):
                sim.qpos[:] = q0
                sim.qpos[j] += sgn * h
                sim.kinematics()
                pts.append(_point(sim, b).copy())
                mats.append(sim.xmat[b].copy())
            dp = (pts[0] - pts[1]) / (2 * h)
            dR = (mats[0] - mats[1]) / (2 * h)
            W = dR @ R0.T                                              # skew-symmetric: the angular velocity per unit dq_j
            dth = np.array([W[2, 1], W[0, 2], W[1, 0]])
            want = w[:3] @ dp + w[3:] @ dth
            assert abs(got[j] - want) < 1e-7 * (1 + np.abs(w).sum()), (b, j, got[j], want)
        sim.qpos[:] = q0
        sim.kinematics()
        if b != jointed[-1]:
            assert np.all(got[12:] == 0), b                            # a wrench on the robot does not reach the cube's dofs


def test_cube_force_at_its_centre_is_the_translation_qfrc():
    flat, sim = _posed_sim(7)
    cube = [b for b in range(int(flat["nbody"])) if flat["body_jntnum"][b] > 0][-1]
    F = np.array([0.3, -1.2, 4.5])
    sim.xfrc_applied[cube, :3] = F
    via_x = sim.applied_qfrc()
    sim.xfrc_applied[:] = 0
    sim.qfrc_applied[12:15] = F
    via_q = sim.applied_qfrc()
    assert np.abs(via_x - via_q).max() < 1e-12, via_x - via_q

    # and one step of the dynamics from a state in the air: the two ways agree
    a, b = (AppliedOracleSim.attach(OracleEnv(flat, has_object=True).sim) for _ in range(2))
    for s in (a, b):
        s.qpos[:] = sim.qpos
        s.qpos[14] = 0.5
        s.applied = True
    a.xfrc_applied[cube, :3] = F
    b.qfrc_applied[12:15] = F
    a.step(20)
    b.step(20)
    assert np.abs(a.qpos - b.qpos).max() < 1e-12 and np.abs(a.qvel - b.qvel).max() < 1e-12


def test_engine_forces_map_to_the_jointed_bodies():
    flat = _flat()
    desc = flatten.reduce_model(flat)
    sim = AppliedOracleSim.attach(OracleEnv(flat, has_object=True).sim)
    x = np.arange(13 * 6, dtype=np.float64).reshape(13, 6) + 1
    set_engine_forces(sim, desc, np.ones(18), x)
    jointed = [b for b in range(int(flat["nbody"])) if flat["body_jntnum"][b] > 0]
    assert sim.applied and np.array_equal(sim.xfrc_applied[jointed], x) and np.count_nonzero(sim.xfrc_applied.any(axis=1)) == 13
    assert np.array_equal(sim.xfrc_point[jointed], np.array([desc.ipos[k][:] for k in range(13)]))


def test_body_names_are_the_reduced_bodies():
    for variant in (mjcf.COMPILED_JOINT, mjcf.COMPILED_MOCAP):
        flat = mjcf.load_compiled(variant)
        jointed = [flat["body_names"][b] for b in range(int(flat["nbody"])) if flat["body_jntnum"][b] > 0]
        assert list(flatten.BODY_NAMES) == jointed
    assert len(flatten.BODY_NAMES) == flatten.NB and flatten.BODY_NAMES.index("object0") == flatten.CUBE_BODY


def test_applied_forces_are_validated():
    n = 4
    q, x = flatten.applied_forces(np.zeros((n, 18), dtype=np.float32), torch.ones(n, 13, 6), n)
    assert q.dtype == torch.float64 and x.dtype == torch.float64 and q.is_contiguous() and tuple(x.shape) == (n, 13, 6)
    assert flatten.applied_forces(None, None, n) == (None, None)
    assert flatten.applied_forces(None, np.zeros((n, 13, 6)), n)[0] is None
    bad = [
        (np.zeros((n, 17)), None), (np.zeros((n + 1, 18)), None), (np.zeros(18), None), (None, np.zeros((n, 12, 6))),
        (None, np.zeros((n, 13, 3))), (None, np.zeros((n, 78))), (np.full((n, 18), np.nan), None), (None, np.full((n, 13, 6), np.inf)),
        (np.zeros((n, 18), dtype=bool), None), (np.zeros((n, 18), dtype=np.complex128), None),
    ]
    for qf, xf in bad:
        with pytest.raises(ValueError):
            flatten.applied_forces(qf, xf, n)
    with pytest.raises(ValueError, match="mesh_collision"):
        flatten.applied_forces(np.zeros((n, 18)), None, n, mesh_collision=True)
