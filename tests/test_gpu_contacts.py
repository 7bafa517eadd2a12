"""Contact output on the device (MyCobotVectorEnv(contact_output=True), mcb_set_contact_output): it changes no result, a forward pass
and a step report the oracle's contacts and mj_contactForce (tests/contact_oracle.py), the forces obey the physics they come from,
the buffers do not depend on the layout tier, and resets, set_state, CUDA graphs, autotune and the guard-word build handle them."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
PICK = dict(has_object=True, reward_type="sparse")
PUSH = dict(has_object=True, block_gripper=True, target_in_the_air=False, reward_type="sparse")
MOCAP = dict(controller_type="mocap", model_path="./assets/mycobot280_mocap.xml")
CONTROLLERS = {"joint": (dict(controller_type="joint"), 7), "IK": (dict(controller_type="IK"), 7), "mocap": (MOCAP, 8)}
STATE_KEYS = ("qpos", "qvel", "ctrl", "qacc_warmstart", "goal", "elapsed", "qprev", "mocap")
FIELDS = ("ncon", "geom", "dim", "dist", "pos", "frame", "force")
# forward() on injected states: both sides run the same Newton iterations from the same warm start, so the forces differ only by the
# rounding carried through the solve (measured worst on one B200: 4.4e-14).  Bound on |force gpu - oracle| per component, relative to
# max(1, the env's largest contact force): 1e-11, a hundredfold margin over the measurement and far below the with-contact 1e-5
FORCE_TOL_FORWARD = 1e-11


def _env(n, **kw):
    from mycobotgym_b200.vector_env import MyCobotVectorEnv

    kw.setdefault("autotune", False)
    return MyCobotVectorEnv(num_envs=n, **kw)


def _actions(gen, n, adim):
    return torch.rand(n, adim, device="cuda", generator=gen) * 2 - 1


def _snap(env, final=False):
    return {k: v.clone() for k, v in env.contacts(final).items()}


def _np(c, i):
    return {k: v[i].cpu().numpy() for k, v in c.items()}


def _flat(ctrl):
    from mycobotgym_b200 import mjcf

    return mjcf.load_compiled(mjcf.COMPILED_MOCAP if ctrl == "mocap" else mjcf.COMPILED_JOINT)


def _states(flat, n, seed):
    """Random arm poses with the gripper half open, the cube resting on the table (some tilted, some moving); row 1 holds the cube
    (the grasp fixture)."""
    rng = np.random.default_rng(seed)
    qpos = np.tile(flat["qpos0"], (n, 1))
    qvel = np.zeros((n, 18))
    for i in range(n):
        qpos[i, :6] = rng.uniform(-1, 1, 6)
        gq = rng.uniform(0.0, 0.5)
        qpos[i, 6:12] = [gq, gq, gq, gq, gq, -gq]
        qvel[i, :6] = rng.normal(size=6) * 0.5
        qpos[i, 12:14] = rng.uniform(-0.1, 0.1, 2)
        qpos[i, 14] = 0.21 - 1e-5
        if i % 2 == 0:
            qvel[i, 12:18] = rng.normal(size=6) * 0.05
        if i % 3 == 0:
            q = np.array([1.0, 0, 0, 0]) + rng.normal(size=4) * 0.02
            qpos[i, 15:19] = q / np.linalg.norm(q)
    g = np.load(os.path.join(GOLDEN, "grasp_pick_sparse.npz"))
    qpos[1], qvel[1] = g["qpos0"], g["qvel0"]
    return qpos, qvel, np.tile(g["warm0"], (n, 1))


def _compare(gpu, ref, tol_geom, tol_force, where):
    """gpu: one env's contacts (numpy), ref: contact_oracle.slots(...).  Returns the worst force error relative to the env's scale."""
    assert int(gpu["ncon"]) == ref["ncon"], where
    for k in ("geom", "dim"):
        assert np.array_equal(gpu[k], ref[k]), (where, k, gpu[k], ref[k])
    for k in ("dist", "pos", "frame"):
        err = np.abs(gpu[k] - ref[k]).max()
        assert err <= tol_geom, (where, k, err)
    scale = max(1.0, np.abs(ref["force"]).max())
    err = np.abs(gpu["force"] - ref["force"]).max() / scale
    assert err <= tol_force, (where, "force", err, scale)
    return err


@pytest.mark.parametrize("ctrl", ["joint", "IK", "mocap"])
def test_contact_output_changes_nothing(ctrl):
    """Contact output on, nominal parameters and a plain batch, 60 steps with auto-resets: bit for bit the same outputs, state and
    statistics.  The contact buffers are in use: contacts and terminal contacts are reported."""
    from mycobotgym_b200 import flatten

    kw, adim = CONTROLLERS[ctrl]
    n = 2048
    plain, nominal, con = _env(n, seed=11, **kw, **PICK), _env(n, seed=11, **kw, **PICK), _env(n, seed=11, contact_output=True, **kw, **PICK)
    nominal.set_params(torch.ones(n, flatten.NPARAM, dtype=torch.float64))
    for e in (plain, nominal, con):
        e.reset()
        e.set_state(elapsed=torch.arange(n, dtype=torch.int32) % 50)
    gen = [torch.Generator(device="cuda").manual_seed(3) for _ in range(3)]
    done, seen, seen_final = 0, 0, 0
    for t in range(60):
        outs = []
        for e, g in zip((plain, nominal, con), gen):
            obs, rew, term, trunc, info = e.step(_actions(g, n, adim))
            outs.append([obs["observation"].clone(), obs["achieved_goal"].clone(), obs["desired_goal"].clone(), rew.clone(),
                         term.clone(), trunc.clone(), info["is_success"].clone(), info["final_observation"].clone()])
        d = outs[0][4] | outs[0][5]
        done += int(d.sum())
        seen += int(con.contacts()["ncon"].sum())
        seen_final += int(con.contacts(final=True)["ncon"][d].sum())
        for other in outs[1:]:
            for k, (x, y) in enumerate(zip(outs[0], other)):
                assert torch.equal(x, y), (ctrl, t, k)
    assert done > 0 and seen > 0 and seen_final > 0
    sp, sn, sc = plain.get_state(), nominal.get_state(), con.get_state()
    assert set(sc) == set(sp)                                        # contacts are output, not state
    for k in sp:
        assert torch.equal(sp[k], sc[k]) and torch.equal(sp[k], sn[k]), (ctrl, k)
    assert torch.equal(plain.stats(), con.stats())


@pytest.mark.parametrize("ctrl", ["joint", "mocap"])
def test_forward_matches_the_oracle(ctrl):
    """forward() on injected contact-rich states (cube on the table, tilted or moving; a held grasp; random arm poses) with random
    cube mass and friction multipliers against the oracle's forward on the model with the env's multipliers baked in: ncon, geom ids
    and dim exact, dist / pos / frame to 1e-9, forces to FORCE_TOL_FORWARD of the env's largest contact force."""
    from contact_oracle import contact_forces, slots
    from mycobotgym_b200 import flatten
    from oracle.oracle import OracleSim

    kw, _ = CONTROLLERS[ctrl]
    fm = _flat(ctrl)
    n = 48
    qpos, qvel, warm = _states(fm, n, 17)
    env = _env(n, contact_output=True, **kw, **PICK)
    env.reset()
    st = env.get_state()
    rng = np.random.default_rng(4)
    p = np.ones((n, flatten.NPARAM))
    p[:, flatten.P_CUBE_MASS] = rng.uniform(0.5, 2.0, n)
    p[:, flatten.P_FRICTION:flatten.P_FRICTION + flatten.NGEOM] = rng.uniform(0.5, 1.5, (n, flatten.NGEOM))
    p[0] = 1.0
    env.set_params(torch.as_tensor(p))
    env.set_state(qpos=qpos, qvel=qvel, qacc_warmstart=warm)
    env.forward()
    c = _snap(env)
    ctrl_np, mocap = st["ctrl"].cpu().numpy(), st["mocap"].cpu().numpy()
    nu = 1 if ctrl == "mocap" else 7
    worst, total = 0.0, 0
    for i in range(n):
        s = OracleSim(flatten.apply_params_flat(fm, p[i]))
        s.set_state(qpos[i], qvel[i], ctrl_np[i][:nu], warm[i])
        if ctrl == "mocap":
            s.mocap_pos[:], s.mocap_quat[:] = mocap[i][:3], mocap[i][3:]
        s.forward()
        ref = slots(contact_forces(s))
        total += ref["ncon"]
        worst = max(worst, _compare(_np(c, i), ref, 1e-9, FORCE_TOL_FORWARD, (ctrl, i)))
    print(f"\n{ctrl}: {n} envs, {total} contacts, worst |force gpu - oracle| / max(1, |force|) = {worst:.2e}")
    assert total > 3 * n


@functools.lru_cache(maxsize=None)
def _rollout_state(case):
    """A rollout state (auto-resets on), the next step's actions; a third of the envs are at their last step of the episode."""
    kw, adim = CONTROLLERS["joint" if case in ("pick", "push") else case]
    task = PUSH if case == "push" else PICK
    n = 1024
    env = _env(n, seed=5, **kw, **task)
    env.reset()
    env.set_state(elapsed=torch.arange(n, dtype=torch.int32) % 50)
    gen = torch.Generator(device="cuda").manual_seed(77)
    for _ in range(10):
        env.step(_actions(gen, n, adim))
    st = {k: v.clone() for k, v in env.get_state().items() if k in STATE_KEYS}
    st["elapsed"] = torch.where(torch.arange(n, device="cuda") % 3 == 0, 49, st["elapsed"] % 40).to(torch.int32)
    acts = _actions(gen, n, adim)
    env.close()
    return kw, task, st, acts


@pytest.mark.parametrize("case", ["pick", "push", "IK", "mocap"])
def test_step_matches_the_oracle(case):
    """One step from rollout states against OracleEnv.step: `contacts()` holds the contacts of the step's last forward pass (the
    block_gripper pass for push), or, for envs that auto-reset, those of the reset state; `contacts(final=True)` holds the terminal
    state's for them.  The terminal contacts are compared where the oracle's observation agrees with the engine's to 1e-7 (contacts are
    a function of the state, whose parity is tests/test_gpu_parity.py's): geometry to 1e-6, forces to 1e-4 of the env's largest
    contact force.  The reset state is the same on both sides (its solve starts from each side's warm start, which the step left):
    geometry to 1e-9, forces to 1e-6."""
    from contact_oracle import contact_forces, slots
    from oracle.oracle import OracleEnv

    kw, task, st_t, acts_t = _rollout_state(case)
    ctrl = kw["controller_type"]
    fm = _flat(ctrl)
    n = acts_t.shape[0]
    env = _env(n, contact_output=True, **kw, **task)
    env.reset()
    env.set_state(**st_t)
    obs, rew, term, trunc, info = env.step(acts_t)
    done = (term | trunc).cpu().numpy()
    c, cf = _snap(env), _snap(env, final=True)
    after = {k: v.cpu().numpy() for k, v in env.get_state().items()}
    st = {k: v.cpu().numpy() for k, v in st_t.items()}
    acts = acts_t.cpu().numpy()
    nu = 1 if ctrl == "mocap" else 7
    okw = dict(task, controller_type=ctrl)
    rng = np.random.default_rng(2)
    chosen = sorted(set(rng.choice(np.flatnonzero(done), 12, replace=False).tolist()) |
                    set(rng.choice(np.flatnonzero(~done), 12, replace=False).tolist()))
    obs_np, fobs_np = obs["observation"].cpu().numpy(), info["final_observation"].cpu().numpy()
    compared, skipped, worst, worst_reset = 0, 0, 0.0, 0.0
    for i in chosen:
        oe = OracleEnv(fm, **okw)
        q_stale = st["qpos"][i].copy()
        q_stale[:6] = st["qprev"][i]
        oe.sim.set_state(q_stale, st["qvel"][i], st["ctrl"][i][:nu], st["qacc_warmstart"][i])
        oe.sim.mocap_pos[:], oe.sim.mocap_quat[:] = st["mocap"][i][:3], st["mocap"][i][3:]
        oe.sim.kinematics()
        oe.sim.qpos[:] = st["qpos"][i]
        oe.goal = st["goal"][i].copy()
        oe.elapsed = int(st["elapsed"][i])
        o, _, te, tr, _ = oe.step(acts[i])
        assert bool(te or tr) == bool(done[i]), i
        terminal = slots(contact_forces(oe.sim))
        agree = np.abs(o["observation"] - (fobs_np[i] if done[i] else obs_np[i])).max() <= 1e-7
        if agree:
            worst = max(worst, _compare(_np(cf if done[i] else c, i), terminal, 1e-6, 1e-4, (case, i, "terminal")))
            compared += 1
        else:
            skipped += 1
        if done[i]:
            oe.reset(object_xy=after["qpos"][i][12:14], goal=after["goal"][i])
            assert np.abs(oe.sim.qpos - after["qpos"][i]).max() == 0.0, i
            worst_reset = max(worst_reset, _compare(_np(c, i), slots(contact_forces(oe.sim)), 1e-9, 1e-6, (case, i, "reset")))
    print(f"\n{case}: {len(chosen)} envs ({int(done[chosen].sum())} auto-reset), {compared} terminal sets compared, {skipped} skipped "
          f"(observation apart by > 1e-7), worst force error {worst:.2e}, after the reset {worst_reset:.2e}")
    assert skipped <= len(chosen) // 4, skipped
    # rows of envs that did not reset keep their previous final contacts: the sentinel written before the step survives
    env.contacts(final=True)["dist"].fill_(7.0)
    env.set_state(**st_t)
    _, _, term, trunc, _ = env.step(acts_t)
    d = term | trunc
    assert bool((env.contacts(final=True)["dist"][~d] == 7.0).all())
    assert torch.equal(env.contacts(final=True)["ncon"][d], cf["ncon"][d])


def test_cube_contact_forces_sum_to_its_constraint_force():
    """For every env, the world-frame forces of the cube's contacts (on the cube: + where it is geom2, - where geom1) add up to the
    translational part of its qfrc_constraint (debug_forward), to rounding."""
    from mycobotgym_b200 import flatten

    fm = _flat("joint")
    n = 16
    qpos, qvel, warm = _states(fm, n, 23)
    env = _env(n, contact_output=True, **PICK)
    env.reset()
    env.set_state(qpos=qpos, qvel=qvel, qacc_warmstart=warm)
    cube = flatten.GEOM_NAMES.index("object0")
    checked = 0
    for i in range(n):
        d = env.debug_forward(i)            # a forward pass of every env: the contacts are this pass's
        c = _np(env.contacts(), i)
        F = np.zeros(3)
        for k in range(int(c["ncon"])):
            g1, g2 = c["geom"][k]
            if cube in (g1, g2):
                F += (1.0 if g2 == cube else -1.0) * (c["frame"][k].T @ c["force"][k][:3])
        q = d["qfrc_constraint"][12:15]
        assert np.abs(F - q).max() <= 1e-9 * max(1.0, np.abs(q).max()), (i, F, q)
        checked += int(np.abs(q).max() > 0)
    assert checked >= n // 2


def _cube_normal_sum(env):
    """Per env, the world-z force of the cube's contacts on the cube."""
    from mycobotgym_b200 import flatten

    cube = flatten.GEOM_NAMES.index("object0")
    c = env.contacts()
    wf = torch.einsum("nckj,nck->ncj", c["frame"], c["force"][..., :3])
    sign = torch.where(c["geom"][..., 1] == cube, 1.0, torch.where(c["geom"][..., 0] == cube, -1.0, 0.0)).to(torch.float64)
    return (wf[..., 2] * sign).sum(dim=1)


def test_resting_cube_carries_its_weight_and_a_push():
    """A cube settled on the table: its contacts' normal forces sum to m g for cube mass multipliers 0.5, 1 and 2; a downward
    xfrc_applied of m g on it adds m g."""
    from mycobotgym_b200 import flatten

    desc = flatten.reduce_model(_flat("joint"))
    g = -desc.gravity[2]
    n = 3
    env = _env(n, contact_output=True, auto_reset=False, **PICK)
    env.reset(object_xy=np.tile([0.05, -0.15], (n, 1)), goals=np.tile([0.0, 0.0, 0.4], (n, 1)))
    mult = torch.tensor([0.5, 1.0, 2.0], dtype=torch.float64)
    p = torch.ones(n, flatten.NPARAM, dtype=torch.float64)
    p[:, flatten.P_CUBE_MASS] = mult
    env.set_params(p)
    hold = env.get_state()["ctrl"].float()
    for _ in range(25):
        env.step(hold)
    env.forward()
    W = (mult * desc.mass[12] * g).cuda()
    np.testing.assert_allclose(_cube_normal_sum(env).cpu().numpy(), W.cpu().numpy(), rtol=1e-3)
    x = torch.zeros(n, 13, 6, dtype=torch.float64)
    x[:, 12, 2] = -W.cpu()
    env.set_applied_forces(None, x)
    for _ in range(25):
        env.step(hold)
    env.forward()
    np.testing.assert_allclose(_cube_normal_sum(env).cpu().numpy(), 2 * W.cpu().numpy(), rtol=1e-3)


def test_grasp_reward_agrees_with_the_reported_contacts():
    """reward_shaping: the grasp term (rewards >= 50) is on exactly when both finger-layer x cube pairs are reported, in `contacts()`
    or, for envs that auto-reset, in `contacts(final=True)`."""
    from mycobotgym_b200 import flatten

    n = 512
    g = np.load(os.path.join(GOLDEN, "grasp_pick_sparse.npz"))
    env = _env(n, seed=9, contact_output=True, has_object=True, reward_type="reward_shaping")
    env.reset()
    k = 128
    st = env.get_state()
    rep = lambda x: torch.as_tensor(np.repeat(np.asarray(x)[None], k, 0), device="cuda")
    for key, val in (("qpos", g["qpos0"]), ("qvel", g["qvel0"]), ("ctrl", g["ctrl0"]), ("qacc_warmstart", g["warm0"])):
        st[key][:k] = rep(val)
    st["elapsed"] = torch.arange(n, dtype=torch.int32, device="cuda") % 50
    env.set_state(**{key: st[key] for key in STATE_KEYS})
    gen = torch.Generator(device="cuda").manual_seed(1)
    fr, fl, ob = (flatten.GEOM_NAMES.index(x) for x in ("right_finger_layer", "left_finger_layer", "object0"))
    grasps, resets = 0, 0
    for t in range(8):
        a = _actions(gen, n, 7)
        a[:k, :6] = torch.as_tensor(g["qpos0"][:6], device="cuda", dtype=torch.float32)
        a[:k, 6] = 0.8
        _, rew, term, trunc, _ = env.step(a)
        d = term | trunc
        c = env.contacts()
        cf = env.contacts(final=True)
        geom = torch.where(d[:, None, None], cf["geom"], c["geom"])
        pair = lambda f: ((geom[..., 0] == f) & (geom[..., 1] == ob)) | ((geom[..., 0] == ob) & (geom[..., 1] == f))
        both = pair(fr).any(dim=1) & pair(fl).any(dim=1)
        on = rew >= 50.0
        assert torch.equal(on, both), (t, torch.nonzero(on != both).flatten()[:8])
        grasps += int(on.sum())
        resets += int(d.sum())
    assert grasps > 0 and resets > 0


def test_buffers_do_not_depend_on_the_layout_tier():
    """One step of a push batch from a rollout state, tiered, middle tier first and last tier only: bit for bit the same contacts
    and final contacts; envs left the common layout."""
    kw, task, st_t, acts_t = _rollout_state("push")
    n = acts_t.shape[0]
    outs, lefts = [], []
    for nefc_max in (0, 88, 128):
        env = _env(n, nefc_max=nefc_max, contact_output=True, **kw, **task)
        env.reset()
        env.set_state(**st_t)
        env.step(acts_t)
        lefts.append(env.last_fallback_envs())
        outs.append([v.clone() for v in env.contacts().values()] + [v.clone() for v in env.contacts(final=True).values()])
        env.close()
    assert lefts[0][0] > 0 and lefts[1][0] == n and lefts[2][1] == n, lefts
    for other in outs[1:]:
        for k, (a, b) in enumerate(zip(outs[0], other)):
            assert torch.equal(a, b), k


def test_masked_reset_set_state_and_forward():
    n = 256
    env = _env(n, seed=4, contact_output=True, **PICK)
    env.reset()
    gen = torch.Generator(device="cuda").manual_seed(2)
    for _ in range(5):
        env.step(_actions(gen, n, 7))
    c = env.contacts()
    for v in c.values():
        v.fill_(7)
    mask = torch.arange(n, device="cuda") % 3 == 0
    env.reset(mask=mask)
    c = env.contacts()
    assert bool((c["dist"][~mask] == 7).all()) and bool((c["ncon"][~mask] == 7).all())
    assert not bool((c["dist"][mask][:, 0] == 7).any()) and bool((c["geom"][mask][c["dim"][mask] == 0] == -1).all())
    # set_state writes nothing; forward() refreshes every env, equal to a forward pass of another batch in the same state
    for v in c.values():
        v.fill_(7)
    ref = _env(n, seed=4, contact_output=True, **PICK)
    ref.reset()
    st = ref.get_state()
    env.set_state(**{k: st[k] for k in STATE_KEYS})
    assert bool((env.contacts()["ncon"] == 7).all())
    env.forward()
    ref.forward()
    for k, v in env.contacts().items():
        assert torch.equal(v, ref.contacts()[k]), k


def test_step_graph_updates_the_buffers_on_every_replay():
    n = 1024
    envs = [_env(n, seed=8, lockstep_warps=1, contact_output=True, **PICK) for _ in range(2)]
    gen = torch.Generator(device="cuda").manual_seed(4)
    for e in envs:
        e.reset()
        e.set_state(elapsed=torch.arange(n, dtype=torch.int32) % 50)
    acts = [_actions(gen, n, 7) for _ in range(20)]
    eager = []
    for a in acts:
        envs[0].step(a)
        eager.append((_snap(envs[0]), _snap(envs[0], final=True)))
    g = envs[1]
    static_act = acts[0].clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        g.step(static_act)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g.step(static_act)
    replay = [(_snap(g), _snap(g, final=True))]
    for a in acts[1:]:
        static_act.copy_(a)
        graph.replay()
        replay.append((_snap(g), _snap(g, final=True)))
    for t, (x, y) in enumerate(zip(eager, replay)):
        for final in (0, 1):
            for k in FIELDS:
                assert torch.equal(x[final][k], y[final][k]), (t, final, k)


def test_constructor_autotune_leaves_the_same_contacts():
    n = 2048
    a = _env(n, seed=12, contact_output=True, **PICK)
    b = _env(n, seed=12, contact_output=True, autotune=True, **PICK)
    a.reset()
    b.reset()                                  # ends with the autotune roll-ahead, whose contacts the snapshot restores
    for final in (False, True):
        for k, v in a.contacts(final).items():
            assert torch.equal(v, b.contacts(final)[k]), (final, k)


def test_mesh_collision_refuses_contact_output():
    from mycobotgym_b200 import _lib

    with pytest.raises(ValueError, match="mesh_collision"):
        _env(8, contact_output=True, mesh_collision=True, **PICK)
    L = _lib.load()
    mesh = _env(8, mesh_collision=True, **PICK)
    buf = [torch.zeros(8 * 24 * 19, dtype=torch.float64, device="cuda") for _ in range(3)]
    assert L.mcb_set_contact_output(mesh._batch, *(b.data_ptr() for b in buf), None, None, None) < 0
    assert b"mesh_collision" in L.mcb_last_error()
    plain = _env(8, **PICK)
    with pytest.raises(RuntimeError, match="contact_output"):
        plain.contacts()


def test_canary_build_with_contact_output():
    from mycobotgym_b200 import _lib

    assert os.path.exists(_lib.CANARY_PATH), "build the canary library first: python -c 'import __graft_entry__ as g; g.build()'"
    env = dict(os.environ, MCB_LIB=_lib.CANARY_PATH)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "canary_workload.py"), "--contacts"], env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "CANARY_OK" in r.stdout and "MCB_CANARY:" not in r.stdout, r.stdout[-3000:]
    print(r.stdout)
