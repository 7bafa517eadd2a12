"""Actuation latency, host side: the range parser, and the oracle's restatement (a latency of 0 is the plain step, a latency of one
full control period delays the joint controller's commands by exactly one step)."""
import numpy as np
import pytest

from mycobotgym_b200 import flatten, mjcf
from latency_oracle import LatencyOracleEnv
from oracle.oracle import OracleEnv


def test_latency_bounds_parses_and_rejects():
    assert flatten.latency_bounds(None, 20) is None
    assert flatten.latency_bounds(7, 20) == (7, 7)
    assert flatten.latency_bounds(np.int64(3), 20) == (3, 3)
    assert flatten.latency_bounds((0, 20), 20) == (0, 20)
    assert flatten.latency_bounds([2, 5], 10) == (2, 5)
    for bad in (1.0, (0, 2.5), "3", (True, 4), True, (1,), (1, 2, 3), -1, (-1, 3), (5, 4), 21, (0, 21), (3, None)):
        with pytest.raises(ValueError):
            flatten.latency_bounds(bad, 20)
    with pytest.raises(ValueError):
        flatten.latency_bounds((0, 11), 10)
    with pytest.raises(ValueError, match="mesh_collision"):
        flatten.latency_bounds((0, 5), 20, mesh_collision=True)


CONTROLLERS = [("joint", False, 7), ("IK", False, 7), ("mocap", False, 8), ("IK", True, 4), ("mocap", True, 4)]


def _oracle(ctrl, fetch, cls=LatencyOracleEnv, **kw):
    flat = mjcf.load_compiled(mjcf.COMPILED_MOCAP if ctrl == "mocap" else mjcf.COMPILED_JOINT)
    return cls(flat, has_object=True, reward_type="dense", controller_type=ctrl, fetch_env=fetch, control_steps=2, **kw)


def _pair(ctrl, fetch, seed, **kw):
    """Two oracles in the same reset state (the reference sampler draws x, y from the global `random`: reset one, copy it)."""
    a, b = _oracle(ctrl, fetch, cls=OracleEnv, **kw), _oracle(ctrl, fetch, **kw)
    a.reset(seed=seed)
    b.reset(seed=seed)
    b.sim.set_state(**a.sim.get_state())
    b.sim.mocap_pos[:], b.sim.mocap_quat[:] = a.sim.mocap_pos, a.sim.mocap_quat
    b.goal = a.goal.copy()
    a.sim.forward()
    b.sim.forward()
    return a, b


def _state(e):
    s = e.sim
    return [s.qpos.copy(), s.qvel.copy(), s.ctrl.copy(), s.qacc_warmstart.copy(), s.mocap_pos.copy(), s.mocap_quat.copy()]


@pytest.mark.parametrize("ctrl,fetch,adim", CONTROLLERS)
def test_latency_zero_is_the_plain_step(ctrl, fetch, adim):
    a, b = _pair(ctrl, fetch, 3)
    rng = np.random.default_rng(0)
    for _ in range(4):
        act = rng.uniform(-1, 1, adim).astype(np.float32)
        oa, ra, *_ = a.step(act)
        ob, rb, *_ = b.step(act, latency=0)
        assert np.array_equal(oa["observation"], ob["observation"]) and ra == rb
        for x, y in zip(_state(a), _state(b)):
            assert np.array_equal(x, y)


def test_latency_changes_the_trajectory():
    a, b = _pair("joint", False, 1)
    act = np.full(7, 0.5, dtype=np.float32)
    a.step(act)
    b.step(act, latency=7)
    assert not np.array_equal(a.sim.qpos, b.sim.qpos)
    assert np.array_equal(a.sim.ctrl, b.sim.ctrl)                    # the same command is in force at the end


def test_full_period_latency_is_a_one_step_delay():
    """Joint controller, latency = frame_skip, fed a_1..a_T, against the plain step fed c_0, a_1..a_{T-1}: bit for bit in qpos, qvel
    and qacc_warmstart after every step (c_0: the command in force at the start, float32-representable and inside [-1, 1]).  Without
    block_gripper: its forward pass comes after the commit and sees the newer command."""
    fs, T = 20, 6
    plain, late = _pair("joint", False, 5)
    rng = np.random.default_rng(2)
    c0 = rng.uniform(-1, 1, 7).astype(np.float32)
    late.sim.ctrl[:] = c0.astype(np.float64)
    plain.sim.ctrl[:] = c0.astype(np.float64)
    acts = [rng.uniform(-1, 1, 7).astype(np.float32) for _ in range(T)]
    fed = [c0] + acts[:-1]
    for t in range(T):
        ol, *_ = late.step(acts[t], latency=fs)
        op, *_ = plain.step(fed[t])
        assert np.array_equal(late.sim.qpos, plain.sim.qpos), t
        assert np.array_equal(late.sim.qvel, plain.sim.qvel), t
        assert np.array_equal(late.sim.qacc_warmstart, plain.sim.qacc_warmstart), t
        assert np.array_equal(ol["observation"], op["observation"]), t
        assert np.array_equal(late.sim.ctrl, acts[t].astype(np.float64))   # the newest command, one step ahead


@pytest.mark.parametrize("ctrl,fetch,adim", CONTROLLERS)
def test_latency_is_bounded_by_the_control_period(ctrl, fetch, adim):
    e = _oracle(ctrl, fetch)
    e.reset(seed=0)
    with pytest.raises(AssertionError):
        e.step(np.zeros(adim, dtype=np.float32), latency=21)
