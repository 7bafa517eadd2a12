"""GPU parity tests proper: the CUDA path (through the C ABI) against the CPU oracle and the committed
golden fixtures.  Tolerances are the north star's: single-step qpos/qvel within 1e-9 abs in contact-free
motion and 1e-5 with contact, rewards within 1e-9, success/done flags exact, injected goals bit-exact.
Nothing here reads /root/reference."""
import os
import random

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL_FREE, TOL_CONTACT, TOL_REWARD = 1e-9, 1e-5, 1e-9


@pytest.fixture(scope="module")
def flat():
    from mycobotgym_b200 import mjcf

    return mjcf.load_compiled()


def _env(**kw):
    from mycobotgym_b200.vector_env import MyCobotVectorEnv

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return MyCobotVectorEnv(**kw)


def _states(flat, n, seed, has_object=True, airborne=False):
    rng = np.random.default_rng(seed)
    qpos = np.tile(flat["qpos0"], (n, 1))
    qvel = np.zeros((n, 18))
    ctrl = np.zeros((n, 7))
    for i in range(1, n):
        qpos[i, :6] = rng.uniform(-1, 1, 6)
        gq = rng.uniform(0.0, 0.5)                       # four-bar closure kept consistent: fingers / hinges follow the gears
        qpos[i, 6:12] = [gq, gq, gq, gq, gq, -gq]
        qvel[i, :6] = rng.normal(size=6) * 0.5
        ctrl[i] = rng.uniform(-1, 1, 7)
        if has_object:
            qpos[i, 12:14] = rng.uniform(-0.1, 0.1, 2)
            qpos[i, 14] = 0.45 if airborne else 0.21 - 1e-5
            if i % 2 == 0:
                qvel[i, 12:18] = rng.normal(size=6) * 0.05
            if i % 3 == 0:
                q = np.array([1.0, 0, 0, 0]) + rng.normal(size=4) * 0.02
                qpos[i, 15:19] = q / np.linalg.norm(q)
    return qpos, qvel, ctrl


def test_native_library_is_loaded():
    from mycobotgym_b200 import _lib

    L = _lib.load()
    assert b"sm_100a" in L.mcb_version()
    with open("/proc/self/maps") as f:
        assert "libmycobot_b200.so" in f.read()


@pytest.mark.parametrize("has_object", [True, False])
def test_forward_stages_match_oracle(flat, has_object):
    from oracle.oracle import OracleSim

    n = 8
    qpos, qvel, ctrl = _states(flat, n, 3, has_object)
    env = _env(num_envs=n, has_object=has_object, reward_type="dense", auto_reset=False)
    jb = [b for b in range(flat["nbody"]) if flat["body_jntnum"][b] > 0]
    nva, nba = (18, 13) if has_object else (12, 12)
    for i in range(n):
        env.set_state(qpos=qpos, qvel=qvel, ctrl=ctrl, qacc_warmstart=np.zeros((n, 18)))
        sim = OracleSim(flat, disable_cube=not has_object)
        sim.set_state(qpos[i], qvel[i], ctrl[i], np.zeros(18))
        sim.forward()
        d = env.debug_forward(i)
        assert d["nefc"] == sim.nefc and d["ncon"] == sim.ncon and d["overflow"] == 0
        np.testing.assert_allclose(d["xpos"][:nba], sim.xpos[jb][:nba], atol=1e-13)
        np.testing.assert_allclose(d["xmat"][:nba], sim.xmat[jb][:nba], atol=1e-13)
        np.testing.assert_allclose(d["M"][:nva, :nva], sim.M[:nva, :nva], atol=1e-14, rtol=1e-11)
        sc = max(1.0, np.abs(sim.qfrc_smooth).max())
        np.testing.assert_allclose(d["qfrc_bias"][:nva], sim.qfrc_bias[:nva], atol=1e-12)
        np.testing.assert_allclose(d["qfrc_smooth"][:nva], sim.qfrc_smooth[:nva], atol=1e-11 * sc)
        np.testing.assert_allclose(d["efc_J"][:, :nva], sim.efc("J")[:, :nva], atol=1e-12)
        np.testing.assert_allclose(d["efc_D"], sim.efc("D"), rtol=1e-10)
        np.testing.assert_allclose(d["efc_aref"], sim.efc("aref"), atol=1e-9 * max(1.0, np.abs(sim.efc("aref")).max()))
        sa = max(1.0, np.abs(sim.qacc).max())
        np.testing.assert_allclose(d["qacc_smooth"][:nva], sim.qacc_smooth[:nva], atol=1e-10 * sa)
        np.testing.assert_allclose(d["qacc"][:nva], sim.qacc[:nva], atol=1e-7 * sa)
    env.close()


def _oracle_step(flat, has_object, block_gripper, reward_type, qpos, qvel, ctrl, goal, act, tolerance=None):
    """One env-step of the oracle from an injected state; also reports whether any inequality row (limit or
    contact) was ever active, i.e. whether the step was contact-free in the north star's sense."""
    from mycobotgym_b200 import mjcf
    from oracle.oracle import OracleEnv

    f = flat
    if tolerance is not None:
        f = mjcf.FlatModel(flat)
        f["tolerance"] = tolerance
    oe = OracleEnv(f, has_object=has_object, block_gripper=block_gripper, reward_type=reward_type)
    oe.sim.set_state(qpos, qvel, ctrl, np.zeros(18))
    oe.goal = goal.copy()
    # probe pass: per-substep row counts
    probe = OracleEnv(f, has_object=has_object, block_gripper=block_gripper, reward_type=reward_type)
    probe.sim.set_state(qpos, qvel, ctrl, np.zeros(18))
    probe.sim.ctrl[:] = np.clip(act, -1, 1).astype(np.float64)
    free = True
    for _ in range(probe.frame_skip):
        probe.sim.step(1)
        free &= probe.sim.nefc == 7
    o, r, te, tr, inf = oe.step(act)
    return oe, o, r, te, tr, inf, free


def _step_compare(flat, has_object, block_gripper, reward_type, qpos, qvel, ctrl, goals, acts, require_free=False, max_hatch=0):
    n = qpos.shape[0]
    env = _env(num_envs=n, has_object=has_object, block_gripper=block_gripper, reward_type=reward_type, auto_reset=False)
    env.set_state(qpos=qpos, qvel=qvel, ctrl=ctrl, qacc_warmstart=np.zeros((n, 18)), goal=goals, elapsed=np.zeros(n, dtype=np.int32))
    obs, rew, term, trunc, info = env.step(torch.as_tensor(acts))
    st = env.get_state()
    gq, gv = st["qpos"].cpu().numpy(), st["qvel"].cpu().numpy()
    nq, nv = (19, 18) if has_object else (12, 12)
    nfree, hatch = 0, 0
    for i in range(n):
        oe, o, r, te, tr, inf, free = _oracle_step(flat, has_object, block_gripper, reward_type, qpos[i], qvel[i], ctrl[i], goals[i], acts[i])
        tol = TOL_FREE if free else TOL_CONTACT        # north star: 1e-9 contact-free, 1e-5 with contact -- qpos, qvel and observations alike
        eq = np.abs(gq[i, :nq] - oe.sim.qpos[:nq]).max()
        ev = np.abs(gv[i, :nv] - oe.sim.qvel[:nv]).max()
        eo = max(np.abs(obs["observation"][i].cpu().numpy() - o["observation"]).max(), np.abs(obs["achieved_goal"][i].cpu().numpy() - o["achieved_goal"]).max())
        if max(eq, ev, eo) > tol:
            # counted escape: the reference algorithm stops its Newton solve at a cost tolerance of 1e-8; where that alone moves
            # the oracle's own result by more than the bound, the case is ill-conditioned and the bound is 10x that sensitivity
            oe2 = _oracle_step(flat, has_object, block_gripper, reward_type, qpos[i], qvel[i], ctrl[i], goals[i], acts[i], tolerance=1e-13)[0]
            sens = max(np.abs(oe2.sim.qpos - oe.sim.qpos).max(), np.abs(oe2.sim.qvel - oe.sim.qvel).max())
            assert max(eq, ev, eo) <= max(tol, 10 * sens), f"env {i} free={free}: qpos {eq:.2e} qvel {ev:.2e} obs {eo:.2e} sensitivity {sens:.2e}"
            hatch += 1
        nfree += free
        assert np.array_equal(obs["desired_goal"][i].cpu().numpy(), goals[i])          # goals bit-exact
        assert abs(float(rew[i]) - float(r)) <= (TOL_REWARD if free or reward_type == "sparse" else tol)
        assert bool(term[i]) == te and bool(trunc[i]) == tr and bool(info["is_success"][i]) == inf["is_success"]
    assert hatch <= max_hatch, f"{hatch} of {n} envs needed the sensitivity-scaled bound (allowed: {max_hatch})"
    assert rew.dtype == (torch.float32 if reward_type == "sparse" else torch.float64)
    if require_free:
        assert nfree >= n // 2, f"only {nfree}/{n} test states were contact-free"
    env.close()
    return nfree


def test_single_step_contact_free_reach(flat):
    # BASELINE config 2: reach, contact-free dynamics, dense reward -- 1e-9 abs
    n = 16
    qpos, qvel, ctrl = _states(flat, n, 5, has_object=False)
    rng = np.random.default_rng(6)
    goals = rng.uniform(-0.1, 0.1, (n, 3)) + np.array([0, 0, 0.3])
    acts = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
    _step_compare(flat, False, False, "dense", qpos, qvel, ctrl, goals, acts, require_free=True)


def test_single_step_contact_free_airborne_cube(flat):
    n = 8
    qpos, qvel, ctrl = _states(flat, n, 7, has_object=True, airborne=True)
    rng = np.random.default_rng(8)
    goals = rng.uniform(-0.1, 0.1, (n, 3)) + np.array([0, 0, 0.3])
    acts = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
    _step_compare(flat, True, False, "dense", qpos, qvel, ctrl, goals, acts, require_free=True)


@pytest.mark.parametrize("block_gripper", [False, True])
def test_single_step_with_table_contact(flat, block_gripper):
    # BASELINE configs 3 (push = block_gripper) and 4 (pick-and-place): 1e-5 with contact
    n = 16
    qpos, qvel, ctrl = _states(flat, n, 9, has_object=True)
    rng = np.random.default_rng(10)
    goals = rng.uniform(-0.1, 0.1, (n, 3)) + np.array([0, 0, 0.21])
    acts = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
    _step_compare(flat, True, block_gripper, "sparse", qpos, qvel, ctrl, goals, acts, max_hatch=1)


@pytest.mark.parametrize("name", ["reach_dense_seed0", "reach_dense_seed1_perturbed", "pick_sparse_seed0",
                                  "pick_sparse_seed4_perturbed", "push_sparse_seed2", "grasp_pick_sparse"])
def test_against_committed_golden_rollouts(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    has_object, block = bool(g["has_object"]), bool(g["block_gripper"])
    env = _env(num_envs=1, has_object=has_object, block_gripper=block, reward_type=str(g["reward_type"]), auto_reset=False)
    env.set_state(qpos=g["qpos0"][None], qvel=g["qvel0"][None], ctrl=g["ctrl0"][None], qacc_warmstart=g["warm0"][None],
                  goal=g["goal"][None], elapsed=np.zeros(1, dtype=np.int32))
    nq, nv = (19, 18) if has_object else (12, 12)
    tol = TOL_CONTACT if has_object else TOL_FREE
    for t in range(len(g["actions"])):
        obs, rew, term, trunc, info = env.step(torch.as_tensor(g["actions"][t][None]))
        st = env.get_state()
        # the GPU state is re-injected from the golden trajectory every step => every step is a single-step test
        np.testing.assert_allclose(st["qpos"][0, :nq].cpu().numpy(), g["qpos"][t][:nq], atol=tol, rtol=0)
        np.testing.assert_allclose(st["qvel"][0, :nv].cpu().numpy(), g["qvel"][t][:nv], atol=tol, rtol=0)
        np.testing.assert_allclose(obs["observation"][0].cpu().numpy(), g["obs"][t], atol=tol, rtol=0)
        assert abs(float(rew[0]) - float(g["reward"][t])) <= TOL_REWARD
        assert bool(term[0]) == bool(g["terminated"][t]) and bool(info["is_success"][0]) == bool(g["success"][t])
        warm = g["warm"][t][None].copy()
        env.set_state(qpos=g["qpos"][t][None], qvel=g["qvel"][t][None], qacc_warmstart=warm)
    env.close()


@pytest.mark.parametrize("name", ["ik_pick_dense_seed3", "ik_fetch_pick_dense_seed5", "mocap_pick_dense_seed6", "mocap_fetch_pick_dense_seed7"])
def test_against_committed_controller_golden(name):
    # IK / mocap fixtures: every step starts from its recorded state (stale-frame configuration qprev and the mocap pose
    # included).  Bound per step: 1e-7 or 100x the oracle's own recorded sensitivity to a one-ulp velocity perturbation.
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    controller, fetch = str(g["controller"]), bool(g["fetch"])
    kw = dict(model_path="./assets/mycobot280_mocap.xml") if controller == "mocap" else {}
    env = _env(num_envs=1, has_object=True, reward_type="dense", controller_type=controller, fetch_env=fetch, auto_reset=False, **kw)
    nu = 1 if controller == "mocap" else 7
    for t in range(len(g["actions"])):
        ctrl = np.zeros((1, 7)); ctrl[0, :nu] = g["ctrl0"][t]
        env.set_state(qpos=g["qpos0"][t][None], qvel=g["qvel0"][t][None], ctrl=ctrl, qacc_warmstart=g["warm0"][t][None],
                      goal=g["goal"][None], elapsed=np.zeros(1, dtype=np.int32), qprev=g["qprev0"][t][None], mocap=g["mocap0"][t][None])
        obs, rew, term, trunc, info = env.step(torch.as_tensor(g["actions"][t][None]))
        st = env.get_state()
        tol = min(max(1e-7, 100 * float(g["sens"][t])), TOL_CONTACT)
        np.testing.assert_allclose(st["qpos"][0].cpu().numpy(), g["qpos"][t], atol=tol, rtol=0, err_msg=f"step {t}")
        np.testing.assert_allclose(st["ctrl"][0, :nu].cpu().numpy(), g["ctrl"][t], atol=tol, rtol=0)
        np.testing.assert_allclose(st["qprev"][0].cpu().numpy(), g["qprev"][t], atol=tol, rtol=0)
        np.testing.assert_allclose(st["mocap"][0].cpu().numpy(), g["mocap"][t], atol=1e-12 if controller == "mocap" else 1.0, rtol=0)
        np.testing.assert_allclose(obs["observation"][0].cpu().numpy(), g["obs"][t], atol=tol, rtol=0)
        assert abs(float(rew[0]) - float(g["reward"][t])) <= tol
    env.close()


def test_reference_seeded_goals_are_bit_exact(flat):
    # goals injected from the reference's seeded sampling protocol (random.seed(k) and reset(seed=k), SURVEY 0.5)
    from oracle.oracle import OracleEnv

    env = _env(num_envs=1, has_object=True, reward_type="sparse", goal_source="reference")
    oe = OracleEnv(flat, has_object=True)
    for seed in (0, 4):
        random.seed(seed)
        oe.reset(seed=seed)
        want_xy, want_goal = oe.sim.qpos[12:14].copy(), oe.goal.copy()
        random.seed(seed)
        obs, _ = env.reset(seed=seed)
        st = env.get_state()
        assert np.array_equal(obs["desired_goal"][0].cpu().numpy(), want_goal)
        assert np.array_equal(st["qpos"][0, 12:14].cpu().numpy(), want_xy)
        assert np.array_equal(st["goal"][0].cpu().numpy(), want_goal)
    # observation right after reset is fresh and matches the oracle's reset observation
    random.seed(0)
    o_ref, _ = oe.reset(seed=0)
    random.seed(0)
    obs, _ = env.reset(seed=0)
    np.testing.assert_allclose(obs["observation"][0].cpu().numpy(), o_ref["observation"], atol=1e-12)
    st = env.get_state()
    np.testing.assert_allclose(st["qacc_warmstart"][0].cpu().numpy(), oe.sim.qacc_warmstart, atol=1e-6 * np.abs(oe.sim.qacc_warmstart).max())
    env.close()


def test_time_limit_auto_reset_and_stats():
    n = 64
    env = _env(num_envs=n, has_object=True, reward_type="sparse", seed=11)
    obs, _ = env.reset()
    g0 = obs["desired_goal"].clone()
    xy = env.get_state()["qpos"][:, 12:14]
    grip = torch.as_tensor(env.initial_gripper_xpos[:2], device="cuda")
    assert bool(((xy - grip).norm(dim=1) >= 0.1).all()) and bool(((g0[:, :2] - xy).norm(dim=1) >= 0.1).all())
    assert bool((g0[:, 2] >= 0.21).all()) and bool((g0[:, 2] <= 0.31 + 1e-12).all())
    assert 0 < int((g0[:, 2] > 0.21).sum()) < n                      # target_in_the_air coin
    act = torch.zeros(n, 7, device="cuda")
    for t in range(50):
        obs, rew, term, trunc, info = env.step(act)
        if t < 49:
            assert not bool(trunc.any()) and not bool(term.any())
    assert bool(trunc.all()) and not bool(term.any())                # TimeLimit(50)
    assert bool(info["_final_observation"].all())
    st = env.get_state()
    assert bool((st["elapsed"] == 0).all()) and bool((st["qvel"] == 0).all())
    assert not torch.equal(obs["desired_goal"], g0)                  # goals resampled on device
    assert not torch.equal(info["final_observation"], obs["observation"])
    s = env.stats().cpu().numpy()
    assert s[0] == n and s[3] == 50 * n and s[4] == 50 * n and s[2] == -50.0 * n and s[5] == 0
    env.close()


def test_success_terminates_and_sparse_reward_is_negative_zero(flat):
    n = 4
    env = _env(num_envs=n, has_object=True, reward_type="sparse", auto_reset=False)
    env.reset()
    obs, *_ = env.step(torch.zeros(n, 7))
    goal = obs["achieved_goal"].clone()
    goal[1:, 0] += torch.tensor([0.0099, 0.0101, 0.5], device="cuda", dtype=torch.float64)
    st = env.get_state()
    env.set_state(goal=goal, qvel=torch.zeros(n, 18), elapsed=np.zeros(n, dtype=np.int32))
    obs, rew, term, trunc, info = env.step(torch.zeros(n, 7))
    d = (obs["achieved_goal"] - goal).norm(dim=1).cpu().numpy()
    want = d < 0.01
    assert np.array_equal(info["is_success"].cpu().numpy(), want)
    assert np.array_equal(term.cpu().numpy(), want) and np.array_equal(trunc.cpu().numpy(), want)
    r = rew.cpu().numpy()
    assert np.array_equal(r, -(d > 0.01).astype(np.float32)) and np.signbit(r[0])
    env.close()


def test_compute_reward_matches_reference_formula():
    env = _env(num_envs=2, has_object=True, reward_type="sparse")
    envd = _env(num_envs=2, has_object=False, reward_type="dense")
    rng = np.random.default_rng(0)
    ag = rng.normal(size=(4, 16384, 3)) * 0.01
    g = rng.normal(size=(4, 16384, 3)) * 0.01
    g[0, 0] = ag[0, 0] + [0.01, 0, 0]          # d == threshold (up to rounding): compare with numpy on the same inputs
    d = np.linalg.norm(ag - g, axis=-1)
    r = env.compute_reward(ag, g, {})
    assert r.dtype == np.float32 and r.shape == (4, 16384)
    mism = r != -(d > 0.01).astype(np.float32)
    assert np.all(np.abs(d[mism] - 0.01) < 1e-9)                       # flags exact except within 1e-9 of the threshold
    rd = envd.compute_reward(torch.as_tensor(ag, device="cuda"), torch.as_tensor(g, device="cuda"), None)
    assert rd.dtype == torch.float64
    np.testing.assert_allclose(rd.cpu().numpy(), -d, atol=TOL_REWARD)
    assert env.compute_reward(np.zeros((0, 3)), np.zeros((0, 3)), None).shape == (0,)
    env.close(); envd.close()


def test_host_buffer_entry_point_equals_device_entry_point():
    n = 256
    a = np.random.default_rng(3).uniform(-1, 1, (n, 7)).astype(np.float32)
    e1 = _env(num_envs=n, has_object=True, reward_type="sparse", seed=5)
    e2 = _env(num_envs=n, has_object=True, reward_type="sparse", seed=5)
    e3 = _env(num_envs=n, has_object=True, reward_type="sparse", seed=5)
    e1.reset(); e2.reset(); e3.reset()
    pageable = dict(observation=np.empty((n, 25)), achieved_goal=np.empty((n, 3)), desired_goal=np.empty((n, 3)), reward=np.empty(n, np.float32),
                    terminated=np.empty(n, np.uint8), truncated=np.empty(n, np.uint8), is_success=np.empty(n, np.uint8))
    for _ in range(3):
        o1, r1, t1, tr1, i1 = e1.step(torch.as_tensor(a))
        out = e2.step_host(a)                              # page-locked result buffers: direct copies
        out3 = e3.step_host(a, pageable)                   # pageable buffers: through the batch's pinned staging
    assert np.array_equal(o1["observation"].cpu().numpy(), out["observation"])
    assert np.array_equal(r1.cpu().numpy(), out["reward"]) and np.array_equal(t1.cpu().numpy(), out["terminated"].astype(bool))
    for k in pageable:
        assert np.array_equal(out[k], out3[k]), k
    e3.close()
    assert e1.last_step_launches == 3          # one kernel per layout tier
    e1.close(); e2.close()


def test_full_size_batch_is_deterministic_and_well_formed(flat):
    # BASELINE config 4 size: 16384 envs.  Same state + same action in every env => bit-identical results
    n = 16384
    env = _env(num_envs=n, has_object=True, reward_type="sparse", auto_reset=False)
    qpos, qvel, ctrl = _states(flat, 2, 21)
    env.set_state(qpos=np.repeat(qpos[1:2], n, 0), qvel=np.repeat(qvel[1:2], n, 0), ctrl=np.repeat(ctrl[1:2], n, 0),
                  qacc_warmstart=np.zeros((n, 18)), goal=np.tile([0.05, 0.0, 0.25], (n, 1)), elapsed=np.zeros(n, dtype=np.int32))
    act = torch.full((n, 7), 0.3, device="cuda")
    for _ in range(2):
        obs, rew, term, trunc, info = env.step(act)
    st = env.get_state()
    for k in ("qpos", "qvel", "qacc_warmstart"):
        assert bool((st[k] == st[k][0:1]).all()), k
    assert bool((obs["observation"] == obs["observation"][0:1]).all())
    # random rollout: finite state, unit quaternions, cube never below the table top by more than the soft-contact depth
    env2 = _env(num_envs=n, has_object=True, reward_type="sparse", seed=1)
    env2.reset()
    gen = torch.Generator(device="cuda"); gen.manual_seed(1234)
    for _ in range(5):
        a = torch.rand(n, 7, device="cuda", generator=gen) * 2 - 1
        obs, rew, term, trunc, info = env2.step(a)
    st = env2.get_state()
    assert bool(torch.isfinite(st["qpos"]).all()) and bool(torch.isfinite(st["qvel"]).all())
    assert float((st["qpos"][:, 15:19].norm(dim=1) - 1).abs().max()) < 1e-12
    assert float(st["qpos"][:, 14].min()) > 0.2099
    s = env2.stats().cpu().numpy()
    assert s[4] == 5 * n and s[5] == 0
    env.close(); env2.close()


def test_state_roundtrip_and_ragged_sizes(flat):
    for n in (1, 3, 33):
        env = _env(num_envs=n, has_object=False, reward_type="dense", auto_reset=False)
        qpos, qvel, ctrl = _states(flat, max(n, 2), 13, has_object=False)
        qpos, qvel, ctrl = qpos[:n], qvel[:n], ctrl[:n]
        env.set_state(qpos=qpos, qvel=qvel, ctrl=ctrl, qacc_warmstart=np.ones((n, 18)), goal=np.ones((n, 3)), elapsed=np.arange(n, dtype=np.int32))
        st = env.get_state()
        assert np.array_equal(st["qpos"].cpu().numpy(), qpos) and np.array_equal(st["qvel"].cpu().numpy(), qvel)
        assert np.array_equal(st["elapsed"].cpu().numpy(), np.arange(n))
        obs, rew, *_ = env.step(torch.zeros(n, 7))
        assert obs["observation"].shape == (n, 10) and rew.shape == (n,) and rew.dtype == torch.float64
        with pytest.raises(ValueError):
            env.step(torch.zeros(n, 6))
        env.close()


def test_tiered_layouts_are_bit_identical(flat):
    # the same states through (a) the tiered launch (48-row common layout, then 88-row middle tier, then 176-row last tier),
    # (b) the middle tier only and (c) the last tier only
    n = 64
    qpos, qvel, ctrl = _states(flat, n, 31)
    g = np.load(os.path.join(GOLDEN, "grasp_pick_sparse.npz"))      # a grasp: coupled rows overflow the common layout
    qpos[5], qvel[5], ctrl[5] = g["qpos0"], g["qvel0"], g["ctrl0"]
    acts = np.random.default_rng(32).uniform(-1, 1, (n, 7)).astype(np.float32)
    acts[5] = g["actions"][0]
    outs = []
    for nefc_max in (0, 88, 128):
        env = _env(num_envs=n, has_object=True, reward_type="sparse", auto_reset=False, nefc_max=nefc_max)
        env.set_state(qpos=qpos, qvel=qvel, ctrl=ctrl, qacc_warmstart=np.zeros((n, 18)), goal=np.tile([0.0, 0.0, 0.3], (n, 1)),
                      elapsed=np.zeros(n, dtype=np.int32))
        obs, rew, term, trunc, info = env.step(torch.as_tensor(acts))
        st = env.get_state()
        if nefc_max == 0:
            assert env.last_fallback_envs() == (1, 1)          # one env left the common layout; a short list goes straight to the last tier
        outs.append((st["qpos"].cpu().numpy(), st["qvel"].cpu().numpy(), obs["observation"].cpu().numpy(), env.stats().cpu().numpy()))
        env.close()
    for o in outs[1:]:
        assert np.array_equal(outs[0][0], o[0]) and np.array_equal(outs[0][1], o[1]) and np.array_equal(outs[0][2], o[2])
        assert o[3][4] == n and o[3][5] == 0                    # every env stepped exactly once, nothing dropped


def test_many_grasps_take_the_middle_tier():
    # a batch in which every env holds the cube (what a trained pick-and-place policy looks like): the list is long enough
    # for the middle tier (> 2 x 5 x SM count); results equal the last-tier-only run bit for bit
    n = 1600
    g = np.load(os.path.join(GOLDEN, "grasp_pick_sparse.npz"))
    rep = lambda x: np.repeat(np.asarray(x)[None], n, 0)
    rng = np.random.default_rng(7)
    qvel = rep(g["qvel0"]) + 1e-3 * rng.normal(size=(n, 18))
    acts = np.zeros((n, 7), dtype=np.float32)
    acts[:, 6] = 0.8
    acts[:, :6] = rng.uniform(-0.05, 0.05, (n, 6)).astype(np.float32) + g["qpos0"][:6].astype(np.float32)
    outs = []
    for nefc_max in (0, 128):
        env = _env(num_envs=n, has_object=True, reward_type="sparse", auto_reset=False, nefc_max=nefc_max, lockstep_warps=16)
        env.set_state(qpos=rep(g["qpos0"]), qvel=qvel, ctrl=rep(g["ctrl0"]), qacc_warmstart=rep(g["warm0"]), goal=rep(g["goal"]),
                      elapsed=np.zeros(n, dtype=np.int32), qprev=rep(g["qpos0"][:6]))
        obs, rew, term, trunc, info = env.step(torch.as_tensor(acts))
        if nefc_max == 0:
            left_common, left_middle = env.last_fallback_envs()
            assert left_common > 1500 and left_middle < 50, (left_common, left_middle)
        st = env.get_state()
        outs.append((st["qpos"].cpu().numpy(), st["qvel"].cpu().numpy(), obs["observation"].cpu().numpy(), env.stats().cpu().numpy()))
        env.close()
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1]) and np.array_equal(outs[0][2], outs[1][2])
    assert outs[0][3][4] == n and outs[0][3][5] == 0


def test_staged_reward_matches_oracle(flat):
    # SURVEY 8f-3 (reward_shaping): contact-pair flags exported from the collision stage + tanh shaping
    from oracle.oracle import OracleEnv

    n = 8
    qpos, qvel, ctrl = _states(flat, n, 41)
    g = np.load(os.path.join(GOLDEN, "grasp_pick_sparse.npz"))
    qpos[3], qvel[3], ctrl[3] = g["qpos0"], g["qvel0"], g["ctrl0"]
    acts = np.random.default_rng(42).uniform(-1, 1, (n, 7)).astype(np.float32)
    acts[3] = g["actions"][0]
    env = _env(num_envs=n, has_object=True, reward_type="reward_shaping", auto_reset=False)
    env.set_state(qpos=qpos, qvel=qvel, ctrl=ctrl, qacc_warmstart=np.zeros((n, 18)), goal=np.tile([0.0, 0.0, 0.3], (n, 1)),
                  elapsed=np.zeros(n, dtype=np.int32))
    obs, rew, term, trunc, info = env.step(torch.as_tensor(acts))
    assert rew.dtype == torch.float64
    for i in range(n):
        oe = OracleEnv(flat, has_object=True, reward_type="reward_shaping")
        oe.sim.set_state(qpos[i], qvel[i], ctrl[i], np.zeros(18))
        oe.goal = np.array([0.0, 0.0, 0.3])
        o, r, te, tr, inf = oe.step(acts[i])
        assert abs(float(rew[i]) - float(r)) < 1e-7, (i, float(rew[i]), float(r))
    assert float(rew[3]) > 50 and float(rew[0]) < 20              # env 3 holds the cube, env 0 does not
    with pytest.raises(NotImplementedError):
        env.compute_reward(np.zeros((2, 3)), np.zeros((2, 3)), None)
    env.close()


def test_sb3_shaped_adapter():
    # SURVEY 8f-4: VecEnv call pattern of scripts/train.py:80-97 and the info keys scripts/eval_model.py:131 reads
    from mycobotgym_b200.sb3_adapter import MyCobotSB3VecEnv

    n = 32
    ve = MyCobotSB3VecEnv(n, has_object=True, reward_type="sparse", seed=2)
    obs = ve.reset()
    assert obs["observation"].shape == (n, 25) and obs["observation"].dtype == np.float64
    for t in range(50):
        ve.step_async(np.zeros((n, 7), dtype=np.float32))
        obs, rew, dones, infos = ve.step_wait()
    assert dones.all() and rew.dtype == np.float32 and len(infos) == n
    assert infos[0]["TimeLimit.truncated"] and infos[0]["is_success"] is False
    assert infos[0]["episode"] == {"r": -50.0, "l": 50} and infos[0]["terminal_observation"]["observation"].shape == (25,)
    assert not np.array_equal(infos[0]["terminal_observation"]["observation"], obs["observation"][0])
    r = ve.env_method("compute_reward", np.zeros((7, 3)), np.full((7, 3), 0.1), None)[0]
    assert r.shape == (7,) and np.all(r == -1.0)
    ve.close()


@pytest.mark.parametrize("fetch_env,has_object", [(False, True), (True, True), (False, False)])
def test_ik_controller_matches_oracle(flat, fetch_env, has_object):
    # SURVEY 8f-1: IK controller (mycobot.py:134-170, utils.py:499-556), 5 x (DLS solve + 20 substeps) per env-step.
    # Every step is a single-step comparison: before it the oracle is re-synchronised to the GPU state, including the
    # STALE site frames the reference's IK reads (kinematics at qprev).  Step 0 starts from fresh frames (reset).
    from oracle.oracle import OracleEnv

    n, adim = 6, (4 if fetch_env else 7)
    env = _env(num_envs=n, has_object=has_object, reward_type="dense", controller_type="IK", fetch_env=fetch_env, auto_reset=False,
               goal_source="reference")
    assert env.action_dim == adim and env.single_action_space.shape == (adim,)
    oes = [OracleEnv(flat, has_object=has_object, reward_type="dense", controller_type="IK", fetch_env=fetch_env) for _ in range(n)]
    ftight = mjcf_tight(flat)
    oes_tight = [OracleEnv(ftight, has_object=has_object, reward_type="dense", controller_type="IK", fetch_env=fetch_env) for _ in range(n)]
    random.seed(11)
    xy, goals = [], []
    for i, oe in enumerate(oes):
        oe.reset(seed=100 + i)
        xy.append(oe.sim.qpos[12:14].copy()); goals.append(oe.goal.copy())
        oes_tight[i].goal = oe.goal.copy()
    obs, _ = env.reset(object_xy=np.array(xy) if has_object else None, goals=np.array(goals))
    assert abs(env.height_offset - oes[0].height_offset) < 1e-12
    np.testing.assert_allclose(env.initial_gripper_xpos, oes[0].initial_gripper_xpos, atol=1e-12)
    rng = np.random.default_rng(12)
    nq, nv = (19, 18) if has_object else (12, 12)

    def sync(oe, st, i):
        q_stale = st["qpos"][i].copy()
        q_stale[:6] = st["qprev"][i]
        oe.sim.set_state(q_stale, st["qvel"][i], st["ctrl"][i], st["qacc_warmstart"][i])
        oe.sim.kinematics()                                   # the frames the reference still holds from its last mj_step
        oe.sim.qpos[:] = st["qpos"][i]

    for t in range(3):
        st = {k: v.cpu().numpy() for k, v in env.get_state().items()}
        for i in range(n):
            sync(oes[i], st, i)
            sync(oes_tight[i], st, i)
            oes_tight[i].sim.qvel[:6] *= 1 + 2.2e-16          # ... and a one-ulp perturbation of the arm velocities
        assert t == 0 or np.abs(st["qprev"] - st["qpos"][:, :6]).max() > 1e-6        # stale path really exercised
        acts = rng.uniform(-1, 1, (n, adim)).astype(np.float32)
        obs, rew, term, trunc, info = env.step(torch.as_tensor(acts))
        after = env.get_state()
        for i, oe in enumerate(oes):
            o, r, te, tr, inf = oe.step(acts[i])
            oes_tight[i].step(acts[i])
            # 100 substeps of the bang-bang PD loop (SURVEY 0.10) are chaotic: a one-ulp change of qvel can move the result by
            # 1e-7.  The bound is 1e-7 or 100x what a one-ulp perturbation + solver tolerance 1e-13 moves the oracle itself (<= 1e-5, the north star's with-contact bound).
            sens = np.abs(oes_tight[i].sim.qpos[:nq] - oe.sim.qpos[:nq]).max()
            tol = min(max(1e-7, 100 * sens), TOL_CONTACT)      # the GPU differs from the oracle in many roundings, not in one ulp
            np.testing.assert_allclose(after["qpos"][i, :nq].cpu().numpy(), oe.sim.qpos[:nq], atol=tol, rtol=0, err_msg=f"step {t} env {i}")
            np.testing.assert_allclose(after["ctrl"][i].cpu().numpy(), oe.sim.ctrl, atol=tol, rtol=0, err_msg=f"ctrl step {t} env {i}")
            np.testing.assert_allclose(obs["observation"][i].cpu().numpy(), o["observation"], atol=tol, rtol=0)
            assert abs(float(rew[i]) - float(r)) <= tol and bool(term[i]) == te
    env.close()


@pytest.mark.parametrize("fetch_env,has_object", [(False, True), (True, True), (False, False)])
def test_mocap_controller_matches_oracle(fetch_env, has_object):
    # SURVEY 8f-2: mocap controller on the mocap model variant (mycobot.py:172-189, mycobot280_mocap.xml): the mocap body is
    # placed at the STALE gripper_tcp pose + action and a weld equality (6 rows ahead of the connects) drags the arm there.
    # Single-step comparisons with the oracle re-synchronised before each step, as for the IK controller.
    from mycobotgym_b200 import mjcf
    from oracle.oracle import OracleEnv

    fm = mjcf.load_compiled(mjcf.COMPILED_MOCAP)
    n, adim = 6, (4 if fetch_env else 8)
    kw = dict(has_object=has_object, reward_type="dense", controller_type="mocap", fetch_env=fetch_env)
    env = _env(num_envs=n, model_path="./assets/mycobot280_mocap.xml", auto_reset=False, goal_source="reference", **kw)
    assert env.action_dim == adim and env.single_action_space.shape == (adim,)
    oes = [OracleEnv(fm, **kw) for _ in range(n)]
    ftight = mjcf_tight(fm)
    oes_tight = [OracleEnv(ftight, **kw) for _ in range(n)]
    random.seed(21)
    xy, goals = [], []
    for i, oe in enumerate(oes):
        oe.reset(seed=200 + i)
        xy.append(oe.sim.qpos[12:14].copy()); goals.append(oe.goal.copy())
        oes_tight[i].goal = oe.goal.copy()
    obs, _ = env.reset(object_xy=np.array(xy) if has_object else None, goals=np.array(goals))
    assert abs(env.height_offset - oes[0].height_offset) < 1e-12
    np.testing.assert_allclose(env.initial_gripper_xpos, oes[0].initial_gripper_xpos, atol=1e-12)
    st0 = env.get_state()
    np.testing.assert_allclose(st0["mocap"][0].cpu().numpy(), np.concatenate((oes[0].sim.mocap_pos, oes[0].sim.mocap_quat)), atol=1e-15)
    np.testing.assert_allclose(obs["observation"][0].cpu().numpy(), oes[0]._get_obs()["observation"], atol=1e-9)
    rng = np.random.default_rng(22)
    nq = 19 if has_object else 12
    tcp = fm["body_names"].index("gripper_tcp")

    def sync(oe, st, i):
        q_stale = st["qpos"][i].copy()
        q_stale[:6] = st["qprev"][i]
        oe.sim.set_state(q_stale, st["qvel"][i], st["ctrl"][i, :1], st["qacc_warmstart"][i])
        oe.sim.kinematics()                                   # stale gripper_tcp pose, as the reference holds it
        oe.sim.qpos[:] = st["qpos"][i]
        oe.sim.mocap_pos[:] = st["mocap"][i, :3]
        oe.sim.mocap_quat[:] = st["mocap"][i, 3:]

    for t in range(4):
        st = {k: v.cpu().numpy() for k, v in env.get_state().items()}
        for i in range(n):
            sync(oes[i], st, i)
            sync(oes_tight[i], st, i)
            oes_tight[i].sim.qvel[:6] *= 1 + 2.2e-16
        assert t == 0 or np.abs(st["qprev"] - st["qpos"][:, :6]).max() > 1e-6
        acts = rng.uniform(-1, 1, (n, adim)).astype(np.float32)
        if not fetch_env:
            # orientation commands near the current tool orientation for half the envs, arbitrary for the rest
            for i in range(0, n, 2):
                acts[i, 3:7] = (oes[i].sim.xquat[tcp] + 0.1 * rng.uniform(-1, 1, 4)).astype(np.float32)
        obs, rew, term, trunc, info = env.step(torch.as_tensor(acts))
        after = env.get_state()
        for i, oe in enumerate(oes):
            o, r, te, tr, inf = oe.step(acts[i])
            oes_tight[i].step(acts[i])
            sens = np.abs(oes_tight[i].sim.qpos[:nq] - oe.sim.qpos[:nq]).max()
            tol = min(max(1e-7, 100 * sens), TOL_CONTACT)
            np.testing.assert_allclose(after["mocap"][i].cpu().numpy(), np.concatenate((oe.sim.mocap_pos, oe.sim.mocap_quat)), atol=1e-13,
                                       err_msg=f"mocap pose step {t} env {i}")
            np.testing.assert_allclose(after["qpos"][i, :nq].cpu().numpy(), oe.sim.qpos[:nq], atol=tol, rtol=0, err_msg=f"step {t} env {i}")
            assert abs(float(after["ctrl"][i, 0]) - oe.sim.ctrl[0]) == 0.0
            np.testing.assert_allclose(obs["observation"][i].cpu().numpy(), o["observation"], atol=tol, rtol=0)
            assert abs(float(rew[i]) - float(r)) <= tol and bool(term[i]) == te
    assert np.abs(after["qpos"][:, :6].cpu().numpy() - st0["qpos"][:, :6].cpu().numpy()).max() > 0.05     # the weld really moved the arm
    env.close()


def mjcf_tight(flat):
    from mycobotgym_b200 import mjcf

    f = mjcf.FlatModel(flat)
    f["tolerance"] = 1e-13
    return f


def test_bad_simulation_guard_resets_the_env():
    # the role of mj_checkPos / mj_checkVel in mj_step: a non-finite state must not poison the batch
    n = 8
    env = _env(num_envs=n, has_object=True, reward_type="sparse", seed=9)
    env.reset()
    st = env.get_state()
    qvel = st["qvel"].clone()
    qvel[2, 0] = float("nan")
    qvel[5, 3] = 1e30
    env.set_state(qvel=qvel)
    obs, rew, term, trunc, info = env.step(torch.zeros(n, 7))
    assert trunc[2] and trunc[5] and not term[2] and int(trunc.sum()) == 2
    st = env.get_state()
    assert bool(torch.isfinite(st["qpos"]).all()) and bool(torch.isfinite(st["qvel"]).all()) and bool(torch.isfinite(obs["observation"]).all())
    assert env.stats().cpu().numpy()[5] == 2
    env.close()


def test_autotune_restores_state_and_grouping_is_scheduling_only():
    # the lockstep grouping of the step kernel (mcb_autotune) must not change a single bit of the results, and tuning must
    # leave state, episode clocks, RNG streams and statistics exactly as they were
    n = 96
    gen = torch.Generator(device="cuda").manual_seed(5)
    acts = torch.rand(4, n, 7, device="cuda", generator=gen) * 2 - 1
    runs = []
    for lw in (1, 4, 16, 0):
        env = _env(num_envs=n, has_object=True, reward_type="sparse", seed=3, max_episode_steps=3, lockstep_warps=lw)
        env.reset()
        if lw == 0:
            before = {k: v.clone() for k, v in env.get_state().items()}
            stats0 = env.stats(reset=False).clone()
            chosen = env.autotune()
            assert chosen in (1, 4, 16) and env.lockstep_warps == chosen
            after = env.get_state()
            for k in before:
                assert torch.equal(before[k], after[k]), k
            assert torch.equal(stats0, env.stats(reset=False))
        else:
            assert env.lockstep_warps == lw
        obs = None
        for t in range(4):                                   # crosses an auto-reset (TimeLimit 3): the RNG streams matter
            obs, rew, term, trunc, info = env.step(acts[t])
        st = env.get_state()
        runs.append((st["qpos"].clone(), st["qvel"].clone(), st["goal"].clone(), obs["observation"].clone(), env.stats().clone()))
        env.close()
    for r in runs[1:]:
        for a, b in zip(runs[0], r):
            assert torch.equal(a, b)
    with pytest.raises(RuntimeError):
        _env(num_envs=2, lockstep_warps=3)


def test_make_registry_ids_and_reference_goal_autoreset():
    from mycobotgym_b200.vector_env import make

    for env_id, obs_dim, adim, rdtype in [("MyCobotPickAndPlace-Sparse-joint-v0", 25, 7, torch.float32),
                                          ("MyCobotReach-Dense-joint-v0", 10, 7, torch.float64),
                                          ("MyCobotPickAndPlace-RewardShaping-joint-v0", 25, 7, torch.float64),
                                          ("MyCobotFetchReach-Sparse-IK-v0", 10, 4, torch.float32),
                                          ("MyCobotReach-Dense-mocap-v0", 10, 8, torch.float64),
                                          ("MyCobotFetchPickAndPlace-Sparse-mocap-v0", 25, 4, torch.float32)]:
        env = make(env_id, num_envs=4)
        obs, info = env.reset(seed=0)
        assert obs["observation"].shape == (4, obs_dim) and info == {} and env.action_dim == adim
        obs, rew, term, trunc, inf = env.step(torch.zeros(4, adim))
        assert rew.dtype == rdtype and rew.shape == (4,) and term.dtype == torch.bool and "is_success" in inf
        env.close()
    with pytest.raises(NotImplementedError):
        make("MyCobotReach-Dense-joint-v1", num_envs=1)           # image envs are out of scope
    # auto-reset with the reference's (host-side, seeded) sampling protocol: goals change at the TimeLimit, state restarts
    env = make("MyCobotPickAndPlace-Sparse-joint-v0", num_envs=3, goal_source="reference", max_episode_steps=3)
    random.seed(5)
    obs, _ = env.reset(seed=5)
    g0 = obs["desired_goal"].clone()
    for t in range(3):
        obs, rew, term, trunc, inf = env.step(torch.zeros(3, 7))
    assert bool(trunc.all()) and bool(inf["_final_observation"].all())
    assert not torch.equal(obs["desired_goal"], g0) and bool((env.get_state()["elapsed"] == 0).all())
    assert not torch.equal(inf["final_observation"], obs["observation"])
    env.close()


def test_reach_reward_shaping_matches_oracle(flat):
    # the 5 MyCobot[Fetch]Reach-RewardShaping-* ids: the hidden cube is simulated (zero-size box), the reward reads its position
    from mycobotgym_b200 import vector_env
    from oracle.oracle import OracleEnv

    n = 8
    env = _env(num_envs=n, has_object=False, reward_type="reward_shaping", auto_reset=False, goal_source="reference")
    oes = [OracleEnv(flat, has_object=False, reward_type="reward_shaping") for _ in range(n)]
    random.seed(3)
    env.reset(seed=3)
    st = {k: v.cpu().numpy() for k, v in env.get_state().items()}
    for i, oe in enumerate(oes):
        oe.reset(seed=0, goal=st["goal"][i])
    rng = np.random.default_rng(12)
    for t in range(4):
        acts = rng.uniform(-1, 1, (n, 7)).astype(np.float32)
        st = {k: v.cpu().numpy() for k, v in env.get_state().items()}
        obs, rew, term, trunc, info = env.step(torch.as_tensor(acts))
        after = env.get_state()
        assert rew.dtype == torch.float64 and obs["observation"].shape == (n, 10)
        for i, oe in enumerate(oes):
            oe.sim.set_state(st["qpos"][i], st["qvel"][i], st["ctrl"][i], st["qacc_warmstart"][i])
            o, r, te, tr, inf = oe.step(acts[i])
            np.testing.assert_allclose(after["qpos"][i].cpu().numpy(), oe.sim.qpos, atol=TOL_CONTACT, rtol=0)     # cube included
            np.testing.assert_allclose(obs["observation"][i].cpu().numpy(), o["observation"], atol=TOL_CONTACT, rtol=0)
            assert abs(float(rew[i]) - float(r)) < 1e-7 and bool(term[i]) == te
    assert float(after["qpos"][:, 14].max()) < 0.2001                      # the point cube rests on the table top
    env.close()
    for name in ("MyCobotReach-RewardShaping-joint-v0", "MyCobotFetchReach-RewardShaping-IK-v0", "MyCobotReach-RewardShaping-mocap-v0"):
        e = vector_env.make(name, num_envs=2, autotune=False)
        e.reset()
        e.step(torch.zeros(2, e.action_dim))
        e.close()
