"""Per-env applied forces on the device: zero forces change nothing, the free cube obeys the force / torque it is given, the two ways
of pushing the cube agree, every controller matches the oracle's restatement in every layout tier, results do not depend on the
tier, resets clear the forces, and checkpoints, autotune, CUDA graphs and the guard-word build carry them."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PICK = dict(has_object=True, reward_type="sparse")
CONTROLLERS = {
    "joint": (dict(controller_type="joint"), 7),
    "IK": (dict(controller_type="IK"), 7),
    "mocap": (dict(controller_type="mocap", model_path="./assets/mycobot280_mocap.xml"), 8),
}
STATE_KEYS = ("qpos", "qvel", "ctrl", "qacc_warmstart", "goal", "elapsed", "qprev", "mocap")
FORCE_KEYS = {"qfrc_applied", "xfrc_applied"}


def _env(n, **kw):
    from mycobotgym_b200.vector_env import MyCobotVectorEnv

    kw.setdefault("autotune", False)
    return MyCobotVectorEnv(num_envs=n, **kw)


def _actions(gen, n, adim):
    return torch.rand(n, adim, device="cuda", generator=gen) * 2 - 1


def _forces(gen, n, k=3):
    """Random pushes: per env `k` random dofs with a generalized force and `k` random bodies with a wrench (arm: ~0.5 N, 0.02 N m;
    cube: ~0.05 N, 5e-4 N m -- its weight is 0.08 N)."""
    q = torch.zeros(n, 18, dtype=torch.float64, device="cuda")
    x = torch.zeros(n, 13, 6, dtype=torch.float64, device="cuda")
    rows = torch.arange(n, device="cuda")[:, None]
    dofs = torch.rand(n, 18, device="cuda", generator=gen).argsort(dim=1)[:, :k]
    q[rows, dofs] = torch.randn(n, k, dtype=torch.float64, device="cuda", generator=gen) * 0.05
    bodies = torch.rand(n, 13, device="cuda", generator=gen).argsort(dim=1)[:, :k]
    scale = torch.tensor([0.5] * 3 + [0.02] * 3, dtype=torch.float64, device="cuda").repeat(13, 1)
    scale[12] = torch.tensor([0.05] * 3 + [5e-4] * 3, dtype=torch.float64)
    x[rows, bodies] = torch.randn(n, k, 6, dtype=torch.float64, device="cuda", generator=gen) * scale[bodies]
    return q, x


def _rollout(env, n, adim, steps, seed):
    gen = torch.Generator(device="cuda")
    gen.manual_seed(seed)
    out = []
    for _ in range(steps):
        obs, rew, term, trunc, info = env.step(_actions(gen, n, adim))
        out += [obs["observation"].clone(), obs["desired_goal"].clone(), rew.clone(), term.clone(), trunc.clone(),
                info["is_success"].clone(), info["final_observation"].clone()]
    return out


@pytest.mark.parametrize("ctrl", ["joint", "IK", "mocap"])
def test_zero_forces_change_nothing(ctrl):
    """All-zero forces (set again before every step: every reset clears them anyway) against a plain batch and a batch with nominal
    parameters, 60 steps with auto-resets: bit for bit the same outputs, state and statistics."""
    from mycobotgym_b200 import flatten

    kw, adim = CONTROLLERS[ctrl]
    n = 2048
    plain, nominal, zero = (_env(n, seed=11, **kw, **PICK) for _ in range(3))
    nominal.set_params(torch.ones(n, flatten.NPARAM, dtype=torch.float64))
    zq, zx = torch.zeros(n, 18, dtype=torch.float64, device="cuda"), torch.zeros(n, 13, 6, dtype=torch.float64, device="cuda")
    zero.set_applied_forces(zq, zx)
    for e in (plain, nominal, zero):
        e.reset()
        e.set_state(elapsed=torch.arange(n, dtype=torch.int32) % 50)
    gen = [torch.Generator(device="cuda").manual_seed(3) for _ in range(3)]
    done = 0
    for t in range(60):
        zero.set_applied_forces(zq, zx)
        outs = []
        for e, g in zip((plain, nominal, zero), gen):
            obs, rew, term, trunc, info = e.step(_actions(g, n, adim))
            outs.append([obs["observation"].clone(), obs["desired_goal"].clone(), rew.clone(), term.clone(), trunc.clone(),
                         info["is_success"].clone(), info["final_observation"].clone()])
        done += int((outs[0][3] | outs[0][4]).sum())
        for other in outs[1:]:
            for k, (x, y) in enumerate(zip(outs[0], other)):
                assert torch.equal(x, y), (ctrl, t, k)
    assert done > 0
    sp, sn, sz = plain.get_state(), nominal.get_state(), zero.get_state()
    assert set(sz) - set(sp) == FORCE_KEYS and set(sp) <= set(sz)
    for k in sp:
        assert torch.equal(sp[k], sz[k]) and torch.equal(sp[k], sn[k]), (ctrl, k)
    assert torch.equal(plain.stats(), zero.stats())
    q, x = plain.get_applied_forces()                                  # a batch without forces reports zeros
    assert not bool(q.any()) and not bool(x.any()) and tuple(x.shape) == (n, 13, 6)


def _air_state(env, n):
    """The reset state with the cube upright, at rest, in the air away from the table and the arm; actions that hold the arm."""
    env.reset(seed=1)
    st = env.get_state()
    q = st["qpos"].clone()
    q[:, 12:15] = torch.tensor([0.25, -0.25, 0.4], dtype=torch.float64, device="cuda")
    q[:, 15:19] = torch.tensor([1.0, 0.0, 0.0, 0.0], dtype=torch.float64, device="cuda")
    qv = st["qvel"].clone()
    qv[:, 12:] = 0
    env.set_state(qpos=q, qvel=qv, qacc_warmstart=torch.zeros_like(qv))
    return st["ctrl"].float()


def test_free_cube_obeys_the_applied_force_and_torque():
    from mycobotgym_b200 import flatten, mjcf

    desc = flatten.reduce_model(mjcf.load_compiled())
    m, izz, h, fs = desc.mass[12], desc.inertia[12][2], desc.timestep, 20
    d = [desc.damping[j] for j in range(12, 18)]
    assert [desc.armature[j] for j in range(12, 18)] == [0.0] * 6 and len(set(d)) == 1 and list(desc.ipos[12]) == [0.0] * 3
    assert len({desc.inertia[12][k] for k in range(3)}) == 1           # isotropic: no gyroscopic term
    d, g = d[0], -desc.gravity[2]
    n = 256
    env = _env(n, auto_reset=False, **PICK)
    act = _air_state(env, n)
    before = env.get_state()

    # weight compensated at the centre of mass: the cube does not move at all
    x = torch.zeros(n, 13, 6, dtype=torch.float64, device="cuda")
    x[:, 12, 2] = m * g
    env.set_applied_forces(xfrc_applied=x)
    env.step(act)
    after = env.get_state()
    assert torch.equal(after["qpos"][:, 12:], before["qpos"][:, 12:]) and not bool(after["qvel"][:, 12:].any())

    # a constant total force F (gravity included) and a torque about world z: implicit-damped velocity recurrence per substep
    _air_state(env, n)
    gen = torch.Generator(device="cuda").manual_seed(5)
    F = torch.randn(n, 3, dtype=torch.float64, device="cuda", generator=gen) * 0.05
    tau = torch.randn(n, dtype=torch.float64, device="cuda", generator=gen) * 1e-4
    x = torch.zeros(n, 13, 6, dtype=torch.float64, device="cuda")
    x[:, 12, :3] = F
    x[:, 12, 2] += m * g
    x[:, 12, 5] = tau
    env.set_applied_forces(xfrc_applied=x)
    env.step(act)
    qv = env.get_state()["qvel"].cpu().numpy()
    F, tau = F.cpu().numpy(), tau.cpu().numpy()
    v, w = np.zeros((n, 3)), np.zeros(n)
    for _ in range(fs):
        v = v + h * (F - d * v) / (m + h * d)
        w = w + h * (tau - d * w) / (izz + h * d)
    assert np.abs(qv[:, 12:15] - v).max() <= 1e-12 * np.abs(v).max(), np.abs(qv[:, 12:15] - v).max()
    assert np.abs(qv[:, 17] - w).max() <= 1e-12 * np.abs(w).max(), np.abs(qv[:, 17] - w).max()
    assert np.abs(qv[:, 15:17]).max() <= 1e-12 * np.abs(w).max()


def test_cube_force_as_xfrc_and_as_qfrc_agree():
    n = 256
    a, b = _env(n, auto_reset=False, **PICK), _env(n, auto_reset=False, **PICK)
    act = _air_state(a, n)
    _air_state(b, n)
    F = torch.randn(n, 3, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2)) * 0.1
    x = torch.zeros(n, 13, 6, dtype=torch.float64, device="cuda")
    q = torch.zeros(n, 18, dtype=torch.float64, device="cuda")
    x[:, 12, :3] = F
    q[:, 12:15] = F
    a.set_applied_forces(xfrc_applied=x)
    b.set_applied_forces(qfrc_applied=q)
    oa, *_ = a.step(act)
    ob, *_ = b.step(act)
    sa, sb = a.get_state(), b.get_state()
    for k in ("qpos", "qvel"):
        err = (sa[k] - sb[k]).abs().max().item()
        assert err <= 1e-12 * max(1.0, sb[k].abs().max().item()), (k, err)
    assert sb["qvel"][:, 12:15].abs().min().item() > 0                 # the force did move the cube
    assert (oa["observation"] - ob["observation"]).abs().max().item() <= 1e-12


@functools.lru_cache(maxsize=None)
def _rollout_state(ctrl):
    """A rollout state of a batch pushed by random forces, the next step's actions and forces (device tensors)."""
    kw, adim = CONTROLLERS[ctrl]
    n = 2048
    env = _env(n, seed=3, **kw, **PICK)
    env.reset()
    env.set_state(elapsed=torch.arange(n, dtype=torch.int32) % 50)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(99)
    for _ in range(12):
        env.set_applied_forces(*_forces(gen, n))
        env.step(_actions(gen, n, adim))
    st = {k: v.clone() for k, v in env.get_state().items() if k not in FORCE_KEYS}
    acts = _actions(gen, n, adim)
    frc = _forces(gen, n)
    env.close()
    return st, acts, frc


@pytest.mark.parametrize("ctrl", ["joint", "IK", "mocap"])
def test_results_do_not_depend_on_the_layout_tier(ctrl):
    """One step with random forces from the same rollout state, tiered (envs that overflow the common layout are redone from
    untouched forces), middle tier first and last tier only: bit for bit the same outputs, state and forces."""
    kw, adim = CONTROLLERS[ctrl]
    st_t, acts_t, (q, x) = _rollout_state(ctrl)
    n = acts_t.shape[0]
    outs, lefts = [], []
    for nefc_max in (0, 88, 128):
        env = _env(n, auto_reset=False, nefc_max=nefc_max, **kw, **PICK)
        env.set_state(**{k: st_t[k] for k in STATE_KEYS}, qfrc_applied=q, xfrc_applied=x)
        obs, rew, term, trunc, info = env.step(acts_t)
        lefts.append(env.last_fallback_envs())
        outs.append([obs["observation"].clone(), rew.clone(), term.clone(), trunc.clone()] + [v.clone() for v in env.get_state().values()])
        env.close()
    assert lefts[1][0] == n and lefts[2][1] == n, lefts
    if ctrl != "joint":
        assert lefts[0][0] > 0, lefts
    for other in outs[1:]:
        for k, (a, b) in enumerate(zip(outs[0], other)):
            assert torch.equal(a, b), (ctrl, k)


@pytest.mark.parametrize("nefc_max", [0, 88, 128])
@pytest.mark.parametrize("ctrl", ["joint", "IK", "mocap"])
def test_matches_the_oracle(ctrl, nefc_max):
    """One step with random forces on random bodies and dofs from rollout states against the oracle's restatement
    (tests/applied_oracle.py), started from the GPU state including the stale frames and the mocap pose.  The bounds of
    tests/test_gpu_latency.py::test_matches_the_oracle: joint 1e-9 contact-free / 1e-5 with contact (counted Newton-tolerance escape),
    IK and mocap min(max(1e-7, 100x the one-ulp sensitivity), 1e-5) or 100x the sensitivity where it alone exceeds 1e-5 (counted)."""
    from applied_oracle import applied_oracle_env, set_engine_forces
    from mycobotgym_b200 import flatten, mjcf

    kw, adim = CONTROLLERS[ctrl]
    okw = dict(PICK, controller_type=ctrl)
    fm = mjcf.load_compiled(mjcf.COMPILED_MOCAP if ctrl == "mocap" else mjcf.COMPILED_JOINT)
    desc = flatten.reduce_model(fm)
    tight = mjcf.FlatModel(fm)
    tight["tolerance"] = 1e-13
    st_t, acts_t, (q_t, x_t) = _rollout_state(ctrl)
    n = acts_t.shape[0]
    env = _env(n, auto_reset=False, nefc_max=nefc_max, **kw, **PICK)
    env.set_state(**{k: st_t[k] for k in STATE_KEYS}, qfrc_applied=q_t, xfrc_applied=x_t)
    obs, rew, term, trunc, info = env.step(acts_t)
    left = env.last_fallback_list()
    after = {k: v.cpu().numpy() for k, v in env.get_state().items()}
    obs_np = obs["observation"].cpu().numpy()
    term_np = term.cpu().numpy()
    env.close()
    assert np.array_equal(after["qfrc_applied"], q_t.cpu().numpy()) and np.array_equal(after["xfrc_applied"], x_t.cpu().numpy())
    st = {k: v.cpu().numpy() for k, v in st_t.items()}
    acts, qf, xf = acts_t.cpu().numpy(), q_t.cpu().numpy(), x_t.cpu().numpy()
    nu = 1 if ctrl == "mocap" else 7

    def start(f, i, ulp=False):
        oe = applied_oracle_env(f, **okw)
        q_stale = st["qpos"][i].copy()
        q_stale[:6] = st["qprev"][i]
        oe.sim.set_state(q_stale, st["qvel"][i], st["ctrl"][i][:nu], st["qacc_warmstart"][i])
        oe.sim.mocap_pos[:], oe.sim.mocap_quat[:] = st["mocap"][i][:3], st["mocap"][i][3:]
        oe.sim.kinematics()
        oe.sim.qpos[:] = st["qpos"][i]
        if ulp:
            oe.sim.qvel[:6] *= 1 + 2.2e-16
        oe.goal = st["goal"][i].copy()
        oe.elapsed = int(st["elapsed"][i])
        set_engine_forces(oe.sim, desc, qf[i], xf[i])
        return oe

    def contact_free(i):
        oe = start(fm, i)
        oe.sim.ctrl[:] = np.clip(acts[i], -1, 1).astype(np.float64)
        free = True
        for _ in range(oe.frame_skip):
            oe.sim.step(1)
            free &= oe.sim.nefc == 7
        return free

    rng = np.random.default_rng(5)
    chosen = sorted(set(rng.choice(n, 24, replace=False).tolist()) | set(left[:24].tolist()))
    failures, hatch, chaotic, ncontact, worst = [], 0, 0, 0, 0.0
    for i in chosen:
        oe = start(fm, i)
        o, r, te, tr, inf = oe.step(acts[i])
        eq = np.abs(after["qpos"][i] - oe.sim.qpos).max()
        ev = np.abs(after["qvel"][i] - oe.sim.qvel).max()
        eo = np.abs(obs_np[i] - o["observation"]).max()
        worst = max(worst, eq)
        if ctrl == "joint":
            free = contact_free(i)
            ncontact += not free
            tol = 1e-9 if free else 1e-5
            if max(eq, ev, eo) > tol:
                oe2 = start(tight, i)
                oe2.step(acts[i])
                sens = max(np.abs(oe2.sim.qpos - oe.sim.qpos).max(), np.abs(oe2.sim.qvel - oe.sim.qvel).max())
                if max(eq, ev, eo) > max(tol, 10 * sens):
                    failures.append((i, bool(free), float(eq), float(ev), float(eo), float(sens)))
                    continue
                hatch += 1
        else:
            oe2 = start(tight, i, ulp=True)
            oe2.step(acts[i])
            sens = np.abs(oe2.sim.qpos - oe.sim.qpos).max()
            if sens > 1e-5:
                chaotic += 1
                tol = 100 * sens
                if eq > tol or eo > 10 * tol:
                    failures.append((i, float(eq), float(eo), float(sens)))
                    continue
            else:
                tol = min(max(1e-7, 100 * sens), 1e-5)
                if eq > tol or eo > min(10 * tol, 1e-5):
                    failures.append((i, float(eq), float(eo), float(sens)))
                    continue
        assert bool(term_np[i]) == te, i
    print(f"\n{ctrl} nefc_max={nefc_max}: {len(chosen)} envs ({len(left)} left the common layout, {ncontact} joint envs with contact), "
          f"worst |qpos gpu - oracle| {worst:.2e}, escape used by {hatch}, one-ulp sensitivity above 1e-5 for {chaotic}")
    assert not failures, failures[:8]
    assert hatch <= max(1, len(chosen) // 50), hatch
    assert chaotic <= max(1, len(chosen) // 6), chaotic
    if nefc_max == 0 and ctrl != "joint":
        assert len(left) > 0


def test_resets_clear_the_forces():
    n = 1024
    gen = torch.Generator(device="cuda").manual_seed(7)
    env = _env(n, seed=21, **PICK)
    env.reset()
    env.set_state(elapsed=torch.arange(n, dtype=torch.int32) % 50)
    q, x = _forces(gen, n)
    q[:, 0] += 1e-3                                                    # every env has a nonzero row
    env.set_applied_forces(q, x)
    _, _, term, trunc, _ = env.step(_actions(gen, n, 7))
    done = term | trunc
    gq, gx = env.get_applied_forces()
    assert 0 < int(done.sum()) < n
    assert not bool(gq[done].any()) and not bool(gx[done].any())
    assert torch.equal(gq[~done], q[~done]) and torch.equal(gx[~done], x[~done])

    # a masked reset clears exactly the masked envs
    env.set_applied_forces(q, x)
    mask = torch.arange(n, device="cuda") % 3 == 0
    env.reset(mask=mask)
    gq, gx = env.get_applied_forces()
    assert not bool(gq[mask].any()) and not bool(gx[mask].any())
    assert torch.equal(gq[~mask], q[~mask]) and torch.equal(gx[~mask], x[~mask])

    # the reset's own forward passes already see zero: its first observation is that of a batch without forces
    plain = _env(n, seed=21, **PICK)
    env.set_applied_forces(q, x)
    o1, _ = env.reset(seed=4)
    o2, _ = plain.reset(seed=4)
    for k in o1:
        assert torch.equal(o1[k], o2[k]), k
    for k, v in plain.get_state().items():
        if k != "qacc_warmstart":          # the solver's warm start comes from each batch's own history (it persists across resets)
            assert torch.equal(v, env.get_state()[k]), k


def test_checkpoint_continues_the_same_trajectory():
    n = 1024
    gen = torch.Generator(device="cuda").manual_seed(8)
    a = _env(n, seed=31, **PICK)
    a.reset()
    a.set_state(elapsed=torch.arange(n, dtype=torch.int32) % 50)
    a.set_applied_forces(*_forces(gen, n))
    a.stats(reset=True)
    ck = {k: v.clone() for k, v in a.get_state().items()}
    assert FORCE_KEYS <= set(ck)
    b = _env(n, seed=777, **PICK)
    b.reset()
    b.set_state(**ck)
    b.stats()
    ra, rb = _rollout(a, n, 7, 40, 12), _rollout(b, n, 7, 40, 12)
    for k, (x, y) in enumerate(zip(ra, rb)):
        assert torch.equal(x, y), k
    sa, sb = a.get_state(), b.get_state()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    assert torch.equal(a.stats(), b.stats())


def test_autotune_restores_the_forces_exactly():
    n = 4096
    gen = torch.Generator(device="cuda").manual_seed(9)
    env = _env(n, seed=6, **PICK)
    env.reset()
    env.set_state(elapsed=torch.arange(n, dtype=torch.int32) % 50)
    env.set_applied_forces(*_forces(gen, n))
    before = {k: v.clone() for k, v in env.get_state().items()}
    stats = env.stats(reset=False).clone()
    env.autotune()
    after = env.get_state()
    for k in before:
        assert torch.equal(before[k], after[k]), k
    assert torch.equal(env.stats(reset=False), stats)


def test_step_graph_replays_like_eager_with_forces_rewritten_between_replays():
    n = 2048
    envs = [_env(n, seed=8, lockstep_warps=1, **PICK) for _ in range(2)]
    gen = torch.Generator(device="cuda")
    gen.manual_seed(4)
    for e in envs:
        e.reset()
        e.set_state(elapsed=torch.arange(n, dtype=torch.int32) % 50)
    acts = [_actions(gen, n, 7) for _ in range(30)]
    frcs = [_forces(gen, n) for _ in range(30)]
    eager = []
    for a, f in zip(acts, frcs):
        envs[0].set_applied_forces(*f)
        obs, rew, _, _, _ = envs[0].step(a)
        eager += [obs["observation"].clone(), rew.clone()]
    g = envs[1]
    g.set_applied_forces(*frcs[0])                                  # the first call turns forces on (it synchronises)
    static_act = acts[0].clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        g.step(static_act)                                          # warm-up outside the capture (step 0)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        obs_g, rew_g, _, _, _ = g.step(static_act)
    replay = [obs_g["observation"].clone(), rew_g.clone()]
    for a, f in zip(acts[1:], frcs[1:]):
        static_act.copy_(a)
        g.set_applied_forces(*f)
        graph.replay()
        replay += [obs_g["observation"].clone(), rew_g.clone()]
    for k, (x, y) in enumerate(zip(eager, replay)):
        assert torch.equal(x, y), k
    for k, v in envs[0].get_state().items():
        assert torch.equal(v, g.get_state()[k]), k


def test_set_applied_forces_validates_and_mesh_batches_refuse():
    from mycobotgym_b200 import _lib

    L = _lib.load()
    env = _env(8, **PICK)
    for q, x in ((torch.zeros(8, 17), None), (None, torch.zeros(8, 13, 5)), (torch.full((8, 18), float("nan")), None),
                 (None, torch.full((8, 13, 6), float("inf")))):
        with pytest.raises(ValueError):
            env.set_applied_forces(q, x)
    assert "qfrc_applied" not in env.get_state()                        # a rejected call turns nothing on
    mesh = _env(8, mesh_collision=True, **PICK)
    with pytest.raises(ValueError, match="mesh_collision"):
        mesh.set_applied_forces(torch.zeros(8, 18))
    assert L.mcb_set_env_applied(mesh._batch, None, None, None) < 0 and b"mesh_collision" in L.mcb_last_error()


def test_canary_build_with_forces():
    from mycobotgym_b200 import _lib

    assert os.path.exists(_lib.CANARY_PATH), "build the canary library first: python -c 'import __graft_entry__ as g; g.build()'"
    env = dict(os.environ, MCB_LIB=_lib.CANARY_PATH)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "canary_workload.py"), "--forces"], env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "CANARY_OK" in r.stdout and "MCB_CANARY:" not in r.stdout, r.stdout[-3000:]
    print(r.stdout)
