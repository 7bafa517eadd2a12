"""Per-env physics parameters on the device: nominal parameters change nothing, an env with parameters p simulates exactly what a
batch on the model with p baked in simulates, the oracle on that model agrees, the draws follow their ranges and their own random
stream, and checkpoints, autotune, CUDA graphs and the guard-word build carry them."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PICK = dict(has_object=True, reward_type="sparse")
WIDE = {"cube_mass": (0.5, 2.0), "friction": (0.7, 1.3), "gain": (0.8, 1.2), "arm_damping": (0.5, 2.0)}
CONTROLLERS = {
    "joint": (dict(controller_type="joint"), 7, "joint"),
    "IK": (dict(controller_type="IK"), 7, "joint"),
    "mocap": (dict(controller_type="mocap", model_path="./assets/mycobot280_mocap.xml"), 8, "mocap"),
}
STATE_KEYS = ("qpos", "qvel", "ctrl", "qacc_warmstart", "goal", "elapsed", "qprev", "mocap")


def _env(n, **kw):
    from mycobotgym_b200.vector_env import MyCobotVectorEnv

    kw.setdefault("autotune", False)
    return MyCobotVectorEnv(num_envs=n, **kw)


def _actions(gen, n, adim):
    return torch.rand(n, adim, device="cuda", generator=gen) * 2 - 1


def _nominal():
    from mycobotgym_b200 import flatten

    return {name: (1.0, 1.0) for name in flatten.PARAM_NAMES}


def _rollout(env, n, adim, steps, seed):
    gen = torch.Generator(device="cuda")
    gen.manual_seed(seed)
    out = []
    for _ in range(steps):
        obs, rew, term, trunc, info = env.step(_actions(gen, n, adim))
        out += [obs["observation"].clone(), obs["desired_goal"].clone(), rew.clone(), term.clone(), trunc.clone(),
                info["is_success"].clone(), info["final_observation"].clone()]
    return out


def test_nominal_parameters_change_nothing():
    n = 2048
    plain, nom = _env(n, seed=11, **PICK), _env(n, seed=11, param_ranges=_nominal(), **PICK)
    for e in (plain, nom):
        e.reset()
        e.set_state(elapsed=torch.arange(n, dtype=torch.int32) % 50)
    a, b = _rollout(plain, n, 7, 60, 3), _rollout(nom, n, 7, 60, 3)
    for k, (x, y) in enumerate(zip(a, b)):
        assert torch.equal(x, y), k
    sa, sb = plain.get_state(), nom.get_state()
    assert set(sb) - set(sa) == {"params", "param_counter"}
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    assert torch.equal(plain.stats(), nom.stats())
    p, c = nom.get_params()
    assert torch.all(p == 1.0)
    assert int(c.min()) >= 14 and int(c.max()) > 14                  # every env drew at reset(), some again at auto-resets
    pp, pc = plain.get_params()
    assert torch.all(pp == 1.0) and torch.all(pc == 0)             # a batch without parameters reports the nominal values


def test_goal_stream_is_independent_of_the_parameters():
    n = 1024
    plain, wide = _env(n, seed=5, **PICK), _env(n, seed=5, param_ranges=WIDE, **PICK)
    for e in (plain, wide):
        e.reset(seed=9)
    assert not torch.all(wide.get_params()[0] == 1.0)
    gp, gw = plain.get_state(), wide.get_state()
    assert torch.equal(gp["goal"], gw["goal"]) and torch.equal(gp["qpos"][:, 12:14], gw["qpos"][:, 12:14])
    mask = torch.arange(n, device="cuda") % 3 == 1
    for e in (plain, wide):
        e.reset(mask=mask)                                         # injected-free masked reset
        e.set_state(elapsed=torch.full((n,), 49, dtype=torch.int32))
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1)
    act = _actions(gen, n, 7)
    _, _, tp, rp, _ = plain.step(act)
    _, _, tw, rw, _ = wide.step(act)
    done = ((tp | rp) & (tw | rw)).cpu()
    assert int(done.sum()) > n // 2                                # the truncation auto-reset every env
    gp, gw = plain.get_state(), wide.get_state()
    assert torch.equal(gp["goal"][done], gw["goal"][done]) and torch.equal(gp["qpos"][done, 12:14], gw["qpos"][done, 12:14])


def test_injected_goals_still_draw_fresh_parameters():
    n = 256
    env = _env(n, seed=2, param_ranges=WIDE, **PICK)
    env.reset()
    p0, c0 = (x.clone() for x in env.get_params())
    goals = np.tile([0.05, 0.0, 0.9], (n, 1))
    xy = np.tile([0.1, 0.05], (n, 1))
    env.reset(object_xy=xy, goals=goals)
    p1, c1 = env.get_params()
    assert torch.all(c1 == c0 + 14) and not torch.equal(p0, p1)
    assert torch.equal(env.get_state()["goal"], torch.as_tensor(goals, device="cuda"))


def test_draws_follow_their_ranges_and_streams():
    from mycobotgym_b200 import flatten

    n = 16384
    ranges = {"cube_mass": (0.5, 2.0), "friction_floor": (0.7, 1.3), "friction_table": (0.7, 1.3), "friction_finger_r": (0.7, 1.3),
              "friction_finger_l": (0.7, 1.3), "friction_cube": (1.25, 1.25), "gain": (0.8, 1.2)}   # arm_damping: (1, 1)
    lo, hi = flatten.param_bounds(ranges)
    env = _env(n, seed=4, param_ranges=ranges, **PICK)
    env.reset()
    p, c = (x.clone() for x in env.get_params())
    lo_t, hi_t = torch.as_tensor(lo, device="cuda"), torch.as_tensor(hi, device="cuda")
    assert torch.all(p >= lo_t) and torch.all(p <= hi_t) and torch.all(c == 14)
    deg = torch.as_tensor(lo == hi, device="cuda")
    assert int(deg.sum()) == 2 and torch.all(p[:, deg] == lo_t[deg])
    mean, mid, sd = p.mean(0).cpu().numpy(), (lo + hi) / 2, (hi - lo) / np.sqrt(12 * n)
    assert np.all(np.abs(mean - mid) <= 4 * sd + 1e-15), (mean, mid)
    assert float(torch.corrcoef(p[:, [1, 2]].T)[0, 1].abs()) < 0.05  # slots of a group are drawn independently

    # across a step, exactly the envs whose episode ended redraw
    env.set_state(elapsed=torch.arange(n, dtype=torch.int32) % 50)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(0)
    _, _, term, trunc, _ = env.step(_actions(gen, n, 7))
    done = term | trunc
    p2, c2 = env.get_params()
    changed = (p2 != p).any(1)
    assert int(done.sum()) > 0 and torch.equal(changed, done) and torch.equal(c2, c + 14 * done.long())

    # reset(seed=s) reproduces, another seed does not, a masked reseed restarts only the masked envs
    env.reset(seed=123)
    a = env.get_params()[0].clone()
    env.reset(seed=123)
    assert torch.equal(env.get_params()[0], a)
    env.reset(seed=124)
    b = env.get_params()[0].clone()
    assert not (b == a).all(1).any()
    mask = torch.arange(n, device="cuda") % 2 == 0
    env.reset(seed=123, mask=mask)
    d = env.get_params()[0]
    assert torch.equal(d[mask], a[mask]) and torch.equal(d[~mask], b[~mask])


def test_ranges_are_validated_in_c_and_python():
    from mycobotgym_b200 import _lib, flatten

    env = _env(8, **PICK)
    L = _lib.load()
    lo, hi = np.ones(flatten.NPARAM), np.ones(flatten.NPARAM)
    ptr = lambda x: x.ctypes.data_as(C.c_void_p)
    for k, (l, h) in enumerate([(2.0, 1.0), (0.0, 1.0), (-1.0, 1.0), (np.nan, 1.0), (1.0, np.inf)]):
        lo2, hi2 = lo.copy(), hi.copy()
        lo2[k % flatten.NPARAM], hi2[k % flatten.NPARAM] = l, h
        assert L.mcb_batch_set_param_ranges(env._batch, ptr(lo2), ptr(hi2)) < 0
    assert L.mcb_batch_set_param_ranges(env._batch, ptr(lo), None) < 0
    p, c = env.get_params()
    assert torch.all(p == 1) and torch.all(c == 0)                 # rejected calls left the batch without parameters
    env.reset()
    assert torch.all(env.get_params()[1] == 0)
    assert L.mcb_batch_set_param_ranges(env._batch, ptr(lo * 0.5), ptr(hi * 2)) == 0
    env.reset()
    p1 = env.get_params()[0].clone()
    assert L.mcb_batch_set_param_ranges(env._batch, None, None) == 0   # stop drawing, values stay
    env.reset()
    assert torch.equal(env.get_params()[0], p1)
    mesh = _env(8, mesh_collision=True, **PICK)
    assert L.mcb_batch_set_param_ranges(mesh._batch, ptr(lo), ptr(hi)) < 0 and b"mesh_collision" in L.mcb_last_error()
    assert L.mcb_set_env_params(mesh._batch, None, None, None) < 0
    with pytest.raises(ValueError):
        _env(8, mesh_collision=True, param_ranges=WIDE, **PICK)


def _param_set(k):
    """k distinct multiplier vectors: the two range extremes, then uniform draws inside WIDE."""
    from mycobotgym_b200 import flatten

    lo, hi = flatten.param_bounds(WIDE)
    rng = np.random.default_rng(17)
    rows = [lo, hi] + [rng.uniform(lo, hi) for _ in range(k - 2)]
    rows[2][[0, 5]] = hi[[0, 5]]
    return np.array(rows)


def _baked_model(dev, variant, p):
    from mycobotgym_b200 import _lib, flatten, mjcf

    L = _lib.load()
    flat = mjcf.load_compiled(mjcf.COMPILED_MOCAP if variant == "mocap" else mjcf.COMPILED_JOINT)
    desc = flatten.apply_params(flatten.reduce_model(flat), p)
    h = C.c_void_p()
    _lib.check(L.mcb_model_create(C.byref(desc), dev, C.byref(h)))
    return h, desc, flat


@pytest.mark.parametrize("nefc_max", [0, 88, 128])
@pytest.mark.parametrize("ctrl", ["joint", "IK", "mocap"])
def test_env_matches_a_batch_on_the_baked_model(monkeypatch, ctrl, nefc_max):
    """The core semantic check: env i of a batch with per-env parameters P[i] and a 1-env batch on the model with P[i] baked in
    (mcb_model_create(apply_params(desc, P[i]))) step bit for bit alike from the same state with the same actions."""
    from mycobotgym_b200 import _lib, vector_env

    kw, adim, variant = CONTROLLERS[ctrl]
    kw = dict(kw, nefc_max=nefc_max, auto_reset=False, **PICK)
    K, steps = 8, 6
    P = _param_set(K)
    src = _env(K, seed=21, **kw)                                   # contact-rich start states: a short rollout ...
    src.reset()
    gen = torch.Generator(device="cuda")
    gen.manual_seed(8)
    for _ in range(12):
        src.step(_actions(gen, K, adim))
    st = src.get_state()
    if ctrl != "mocap":                                            # ... and a held grasp (the golden that reaches the upper tiers)
        g = np.load(os.path.join(ROOT, "tests", "golden", "grasp_pick_sparse.npz"))
        for key, val in (("qpos", "qpos0"), ("qvel", "qvel0"), ("ctrl", "ctrl0"), ("qacc_warmstart", "warm0")):
            st[key][0] = torch.as_tensor(g[val], device="cuda")
        st["qprev"][0] = st["qpos"][0, :6]
    st = {k: st[k] for k in STATE_KEYS}
    acts = [_actions(gen, K, adim) for _ in range(steps)]
    if ctrl != "mocap":
        for a in acts:
            a[0, :6] = torch.as_tensor(g["qpos0"][:6], device="cuda", dtype=torch.float32)
            a[0, 6] = 0.8

    env = _env(K, **kw)
    env.set_state(**st)
    env.set_params(P)
    got = []
    for a in acts:
        obs, rew, term, trunc, info = env.step(a)
        got.append([obs["observation"].clone(), obs["achieved_goal"].clone(), rew.clone(), term.clone(), trunc.clone(), info["is_success"].clone()])
    got_state = env.get_state()
    fallbacks = env.last_fallback_envs()

    dev = torch.cuda.current_device()
    L = _lib.load()
    for i in range(K):
        h, desc, flat = _baked_model(dev, variant, P[i])
        try:
            monkeypatch.setitem(vector_env._MODEL_CACHE, (dev, variant), (h, desc, flat))
            one = _env(1, **kw)
            one.set_state(**{k: v[i:i + 1] for k, v in st.items()})
            for t, a in enumerate(acts):
                obs, rew, term, trunc, info = one.step(a[i:i + 1])
                want = [obs["observation"], obs["achieved_goal"], rew, term, trunc, info["is_success"]]
                for k, (x, y) in enumerate(zip(got[t], want)):
                    assert torch.equal(x[i:i + 1], y), (ctrl, nefc_max, i, t, k)
            one_state = one.get_state()
            for k in STATE_KEYS:
                assert torch.equal(got_state[k][i:i + 1], one_state[k]), (ctrl, nefc_max, i, k)
            one.close()
        finally:
            monkeypatch.undo()
            L.mcb_model_destroy(h)
    print(f"\n{ctrl} nefc_max={nefc_max}: {K} envs x {steps} steps bitwise equal; last step left tier 0 / 1: {fallbacks}")


def test_oracle_parity_with_baked_flat_model():
    """One step from rollout states of a randomised batch against OracleEnv on the flat model with the env's multipliers baked in
    (apply_params_flat); bounds and the sensitivity-scaled escape of tests/test_gpu_rollout_parity.py."""
    from mycobotgym_b200 import flatten, mjcf
    from oracle.oracle import OracleEnv

    flat = mjcf.load_compiled()
    n = 4096
    env = _env(n, seed=3, param_ranges=WIDE, **PICK)
    env.reset()
    env.set_state(elapsed=torch.arange(n, dtype=torch.int32) % 50)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(99)
    for _ in range(25):
        env.step(_actions(gen, n, 7))
    st_t = env.get_state()
    st = {k: v.cpu().numpy() for k, v in st_t.items()}
    acts_t = _actions(gen, n, 7)
    acts = acts_t.cpu().numpy()
    env2 = _env(n, auto_reset=False, **PICK)
    env2.set_state(**{k: st_t[k] for k in STATE_KEYS if k != "mocap"}, params=st_t["params"])
    obs, rew, term, trunc, info = env2.step(acts_t)
    left = env2.last_fallback_list()
    after = {k: v.cpu().numpy() for k, v in env2.get_state().items()}
    obs_np = {k: v.cpu().numpy() for k, v in obs.items()}
    rew_np, term_np, trunc_np = rew.cpu().numpy(), term.cpu().numpy(), trunc.cpu().numpy()

    def oracle(i, tolerance=None):
        f = flatten.apply_params_flat(flat, st["params"][i])
        if tolerance is not None:
            f["tolerance"] = tolerance
        oe = OracleEnv(f, has_object=True, reward_type="sparse")
        oe.sim.set_state(st["qpos"][i], st["qvel"][i], st["ctrl"][i], st["qacc_warmstart"][i])
        oe.goal = st["goal"][i].copy()
        oe.elapsed = int(st["elapsed"][i])
        return oe

    rng = np.random.default_rng(5)
    chosen = sorted(set(rng.choice(n, 48, replace=False).tolist()) | set(left[:48].tolist()))
    hatch, ncontact, failures = 0, 0, []
    for i in chosen:
        probe = oracle(i)
        probe.sim.ctrl[:] = np.clip(acts[i], -1, 1).astype(np.float64)
        free = True
        for _ in range(probe.frame_skip):
            probe.sim.step(1)
            free &= probe.sim.nefc == 7
        oe = oracle(i)
        o, r, te, tr, inf = oe.step(acts[i])
        tol = 1e-9 if free else 1e-5
        eq = np.abs(after["qpos"][i] - oe.sim.qpos).max()
        ev = np.abs(after["qvel"][i] - oe.sim.qvel).max()
        eo = np.abs(obs_np["observation"][i] - o["observation"]).max()
        if max(eq, ev, eo) > tol:
            oe2 = oracle(i, tolerance=1e-13)
            oe2.step(acts[i])
            sens = max(np.abs(oe2.sim.qpos - oe.sim.qpos).max(), np.abs(oe2.sim.qvel - oe.sim.qvel).max())
            if max(eq, ev, eo) > max(tol, 10 * sens):
                failures.append((i, free, float(eq), float(ev), float(eo), float(sens)))
                continue
            hatch += 1
        ncontact += not free
        d = np.linalg.norm(o["achieved_goal"] - st["goal"][i])
        assert float(rew_np[i]) == float(r) or abs(d - 0.01) < 1e-9
        assert bool(term_np[i]) == te and bool(trunc_np[i]) == tr
    assert not failures, failures[:8]
    assert ncontact >= len(chosen) // 4 and hatch <= max(1, len(chosen) // 50), (ncontact, hatch, len(chosen))
    print(f"\noracle parity: {len(chosen)} envs, {ncontact} with contact, sensitivity-scaled bound used by {hatch}")


def test_checkpoint_continues_the_same_trajectory():
    n = 1024
    a = _env(n, seed=31, param_ranges=WIDE, **PICK)
    a.reset()
    a.set_state(elapsed=torch.arange(n, dtype=torch.int32) % 50)
    a.stats(reset=True)
    ck = {k: v.clone() for k, v in a.get_state().items()}
    b = _env(n, seed=777, param_ranges=WIDE, **PICK)
    b.reset()
    b.set_state(**ck)
    b.stats()
    ra, rb = _rollout(a, n, 7, 60, 12), _rollout(b, n, 7, 60, 12)
    for k, (x, y) in enumerate(zip(ra, rb)):
        assert torch.equal(x, y), k
    sa, sb = a.get_state(), b.get_state()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    sta, stb = a.stats().clone(), b.stats().clone()
    assert torch.equal(sta, stb) and sta[0] > 0
    assert int((sa["param_counter"] > ck["param_counter"]).sum()) > n // 2       # the roll redrew parameters


def test_autotune_restores_parameters_exactly():
    n = 4096
    env = _env(n, seed=6, param_ranges=WIDE, **PICK)
    env.reset()
    env.set_state(elapsed=torch.arange(n, dtype=torch.int32) % 50)
    before = {k: v.clone() for k, v in env.get_state().items()}
    stats = env.stats(reset=False).clone()
    env.autotune()
    after = env.get_state()
    for k in before:
        assert torch.equal(before[k], after[k]), k
    assert torch.equal(env.stats(reset=False), stats)


def test_step_is_graph_capturable_and_replays_like_eager():
    n = 2048
    envs = [_env(n, seed=8, param_ranges=WIDE, lockstep_warps=1, **PICK) for _ in range(2)]
    acts = []
    gen = torch.Generator(device="cuda")
    gen.manual_seed(4)
    for e in envs:
        e.reset()
        e.set_state(elapsed=torch.arange(n, dtype=torch.int32) % 50)
    for _ in range(30):
        acts.append(_actions(gen, n, 7))
    eager = []
    for a in acts:
        obs, rew, _, _, _ = envs[0].step(a)
        assert envs[0].last_step_launches == 3
        eager += [obs["observation"].clone(), rew.clone()]
    g = envs[1]
    static_act = acts[0].clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        g.step(static_act)                                          # warm-up outside the capture (step 0)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        obs_g, rew_g, _, _, _ = g.step(static_act)
    replay = [obs_g["observation"].clone(), rew_g.clone()]          # (capture does not run the step: these are step 0's outputs)
    for a in acts[1:]:
        static_act.copy_(a)
        graph.replay()
        replay += [obs_g["observation"].clone(), rew_g.clone()]
    for k, (x, y) in enumerate(zip(eager, replay)):
        assert torch.equal(x, y), k
    for k, v in envs[0].get_state().items():
        assert torch.equal(v, g.get_state()[k]), k


def test_canary_build_with_parameters():
    from mycobotgym_b200 import _lib

    assert os.path.exists(_lib.CANARY_PATH), "build the canary library first: python -c 'import __graft_entry__ as g; g.build()'"
    env = dict(os.environ, MCB_LIB=_lib.CANARY_PATH)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "canary_workload.py"), "--params"], env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "CANARY_OK" in r.stdout and "MCB_CANARY:" not in r.stdout, r.stdout[-3000:]
    print(r.stdout)
