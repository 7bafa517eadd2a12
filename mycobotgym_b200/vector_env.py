"""Host-side mirror of the reference's env API for the hot path, served from device-resident state.

`MyCobotVectorEnv` keeps the reference's gymnasium surface (mycobotgym/envs/mycobot.py:27-205,
506-514: constructor kwargs, `reset(seed=, options=)`, `step(action)`, dict observations with
observation / achieved_goal / desired_goal, `compute_reward`, `observation_space` / `action_space`,
attrs `goal`, `distance_threshold`, `reward_type`) for `num_envs` environments at once.  All physics
and task logic runs in the CUDA library behind include/mycobot_b200.h; torch only owns the device
buffers and the stream.  TimeLimit(50) (mycobotgym/__init__.py:34) is folded into the kernel.

Built controllers: joint (`...-joint-v0`), IK (`...-IK-v0`) and mocap (`...-mocap-v0`, on the mocap model
variant), each incl. its Fetch variant where the reference registers one; the image envs (`-v1`) raise
NotImplementedError (out of scope, SURVEY.md section 8).
"""
from __future__ import annotations

import ctypes as C
import random
import re

import numpy as np
import torch

from . import _lib, flatten, mjcf


class Box:
    """Minimal stand-in for gymnasium.spaces.Box (gymnasium is not installable in this image)."""

    def __init__(self, low, high, shape, dtype):
        self.shape, self.dtype = tuple(shape), np.dtype(dtype)
        self.low = np.full(self.shape, low, dtype=self.dtype)
        self.high = np.full(self.shape, high, dtype=self.dtype)
        self._rng = np.random.default_rng()

    def seed(self, seed=None):
        self._rng = np.random.default_rng(seed)

    def sample(self):
        return self._rng.uniform(self.low, self.high).astype(self.dtype)

    def contains(self, x):
        x = np.asarray(x)
        return x.shape == self.shape and np.all(x >= self.low) and np.all(x <= self.high)

    def __repr__(self):
        return f"Box({self.low.min()}, {self.high.max()}, {self.shape}, {self.dtype})"


class Dict(dict):
    """Minimal stand-in for gymnasium.spaces.Dict."""

    @property
    def spaces(self):
        return self

    def sample(self):
        return {k: v.sample() for k, v in self.items()}


REWARD = {"dense": "Dense", "sparse": "Sparse", "reward_shaping": "RewardShaping"}


def registry():
    """Env ids and kwargs exactly as mycobotgym/__init__.py:5-45 registers them (v0 state envs)."""
    import itertools

    reg = {}
    for reward_type, has_object, controller, fetch in itertools.product(
            ["dense", "sparse", "reward_shaping"], [True, False], ["mocap", "IK", "joint"], [True, False]):
        if fetch and controller == "joint":
            continue
        model_path = f"./assets/mycobot280{'_mocap' if controller == 'mocap' else ''}.xml"
        name = f"MyCobot{'Fetch' if fetch else ''}{'PickAndPlace' if has_object else 'Reach'}"
        reg[f"{name}-{REWARD[reward_type]}-{controller}-v0"] = dict(
            model_path=model_path, reward_type=reward_type, has_object=has_object, controller_type=controller,
            fetch_env=fetch, max_episode_steps=50)
    return reg


def make(env_id, num_envs=1, **kwargs):
    """`gymnasium.make(id)` counterpart returning a device-resident vector env."""
    reg = registry()
    if env_id not in reg:
        if re.match(r"MyCobot.*-v1$", env_id):
            raise NotImplementedError(f"{env_id}: image observation envs (MyCobotImgEnv) are out of scope")
        raise KeyError(f"unknown env id {env_id!r}")
    kw = dict(reg[env_id])
    kw.update(kwargs)
    return MyCobotVectorEnv(num_envs=num_envs, **kw)


class ReferenceGoalSampler:
    """The reference's sampling protocol (mycobot.py:207-243, utils.py:14-21): x, y from the GLOBAL
    stdlib `random`; the in-the-air coin / offset from a per-env numpy Generator seeded the way
    gymnasium's `seeding.np_random(seed)` does (PCG64 over SeedSequence(seed))."""

    def __init__(self, num_envs, height_offset, initial_gripper_xy, has_object, target_in_the_air):
        self.n, self.h, self.gxy = num_envs, height_offset, np.asarray(initial_gripper_xy, dtype=np.float64)
        self.has_object, self.air = has_object, target_in_the_air
        self.rngs = [np.random.Generator(np.random.PCG64(np.random.SeedSequence())) for _ in range(num_envs)]

    def seed(self, seed):
        if seed is None:
            return
        seeds = [seed + i for i in range(self.n)] if np.isscalar(seed) else list(seed)
        for i, s in enumerate(seeds):
            if s is not None:
                self.rngs[i] = np.random.Generator(np.random.PCG64(np.random.SeedSequence(int(s))))

    def _sample_goal(self, i):
        x = random.uniform(-0.12, 0.12)
        y = random.uniform(-0.06, 0.06)
        g = [x, y, self.h]
        if self.air and self.rngs[i].uniform() < 0.5:
            g[2] += self.rngs[i].uniform(0, 0.1)
        return np.array(g)

    def sample(self, env_ids):
        """Returns (obj_xy [N,2], goals [N,3]) with rows filled for env_ids (in index order)."""
        xy = np.zeros((self.n, 2))
        goals = np.zeros((self.n, 3))
        for i in env_ids:
            oxy = self.gxy.copy()
            if self.has_object:
                while np.linalg.norm(oxy - self.gxy) < 0.1:
                    oxy = self._sample_goal(i)[:2]
            g = self._sample_goal(i)
            while np.linalg.norm(g[:2] - oxy) < 0.1:
                g = self._sample_goal(i)
            xy[i], goals[i] = oxy, g
        return xy, goals


_MODEL_CACHE = {}


def _device_model(device_index, variant="joint"):
    """One device copy per (GPU, model variant): mycobot280.xml serves the joint and IK controllers,
    mycobot280_mocap.xml (mocap body + weld, one actuator) the mocap controller."""
    key = (device_index, variant)
    if key not in _MODEL_CACHE:
        L = _lib.load()
        flat = mjcf.load_compiled(mjcf.COMPILED_MOCAP if variant.startswith("mocap") else mjcf.COMPILED_JOINT)
        desc = flatten.reduce_model(flat)
        if variant.endswith("+hidden"):
            # "Hide object in Reach env" (mycobot.py:475-481): geom_size[object0] = 0 AFTER compilation, so geom_rbound keeps the
            # visible cube's value; only the reach + reward_shaping ids simulate this cube (it is frozen otherwise)
            for k in range(3):
                desc.geom_size[desc.geom_object][k] = 0.0
        h = C.c_void_p()
        _lib.check(L.mcb_model_create(C.byref(desc), device_index, C.byref(h)))       # restores the caller's current device
        if int(flat.get("nhull", 0)):
            # convex hulls of the mesh geoms: registered always, collided only by batches created with mesh_collision=True
            hd, verts = flatten.reduce_hulls(flat)
            _lib.check(L.mcb_model_set_hulls(h, C.byref(hd)))
            del verts
        _MODEL_CACHE[key] = (h, desc, flat)
    return _MODEL_CACHE[key]


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


# The optional groups of get_state() / set_state(): group -> (its two keys, the getter, the setter taking the two arrays)
_OPTIONAL = {"params": (("params", "param_counter"), "get_params", "set_params"),
             "latency": (("latency", "latency_counter"), "get_latency", "set_latency"),
             "forces": (("qfrc_applied", "xfrc_applied"), "get_applied_forces", "set_applied_forces")}


class MyCobotVectorEnv:
    metadata = {"render_modes": [], "render_fps": 25}

    def __init__(self, num_envs=1, model_path="./assets/mycobot280.xml", has_object=True, block_gripper=False,
                 control_steps=5, controller_type="joint", obj_range=0.1, target_in_the_air=True,
                 distance_threshold=0.01, initial_qpos=None, fetch_env=False, reward_type="sparse", frame_skip=20,
                 max_episode_steps=50, device="cuda:0", seed=0, auto_reset=True, goal_source="device", nefc_max=0,
                 lockstep_warps=0, autotune=True, mesh_collision=False, param_ranges=None, actuation_latency=None,
                 contact_output=False, **kwargs):
        """Constructor kwargs are the reference's (mycobot.py:30-46).  `obj_range` and `initial_qpos` are accepted and only
        stored, exactly like the reference does (mycobot.py:54,56 assign them; nothing reads them: the cube is placed by
        `generate_random_point_inside_rectangle`, mycobot.py:220-222, and the start pose is qpos0 / keyframe 0).
        `lockstep_warps=0, autotune=True`: the first full `reset()` ends with one explicit `mcb_autotune` call (it
        synchronises and is never hidden inside `step`); `autotune=False` keeps the free-running default.
        `mesh_collision=True`: the convex hulls of the 28 mesh geoms collide too (MuJoCo: mjc_Convex / mjc_PlaneConvex; here one
        MPR contact per hull pair, DESIGN.md section 4); off, only the plane / box primitives collide.
        `param_ranges={name: (lo, hi)}`: per-env physics parameters (domain randomisation), redrawn on the device at every reset of
        an env (`flatten.PARAM_NAMES`, groups 'friction' and 'gain'; DESIGN.md section 9).  Not available with mesh_collision.
        `actuation_latency=d` or `(lo, hi)`: per-env actuation latency in substeps (0 <= lo <= hi <= frame_skip), drawn uniformly from
        the integers [lo, hi] at every reset of an env: each command the controller issues takes effect that many substeps into its
        control period (DESIGN.md section 10).  Not available with mesh_collision.
        `contact_output=True`: every step, reset and forward writes the contacts of each env's last forward pass and their forces
        into persistent device buffers, read with `contacts()` (DESIGN.md section 12).  Not available with mesh_collision."""
        if controller_type not in ("joint", "IK", "mocap"):
            raise ValueError(f"unknown controller_type {controller_type!r}")
        if fetch_env and controller_type == "joint":
            raise AssertionError("Joint controller not supported for Fetch env")        # mycobot.py:96
        if reward_type not in ("sparse", "dense", "reward_shaping"):
            raise ValueError(f"unknown reward_type {reward_type!r}")
        if ("mocap" in model_path) != (controller_type == "mocap"):
            raise ValueError("the mocap controller needs mycobot280_mocap.xml and the joint/IK controllers mycobot280.xml "
                             "(the reference would fail on data.mocap_pos / on the missing actuators)")
        if goal_source not in ("device", "reference"):
            raise ValueError("goal_source must be 'device' or 'reference'")
        bounds = None if param_ranges is None else flatten.param_bounds(param_ranges, mesh_collision)
        lat_bounds = None if actuation_latency is None else flatten.latency_bounds(actuation_latency, int(frame_skip), mesh_collision)
        if contact_output and mesh_collision:
            raise ValueError("contact output is not supported with mesh_collision=True")
        if not torch.cuda.is_available():
            raise RuntimeError("MyCobotVectorEnv needs a CUDA device; there is no CPU fallback")
        self.device = torch.device(device)
        self.num_envs = int(num_envs)
        self.has_object, self.block_gripper = bool(has_object), bool(block_gripper)
        self.target_in_the_air, self.distance_threshold = bool(target_in_the_air), float(distance_threshold)
        self.reward_type, self.frame_skip, self.control_steps = reward_type, int(frame_skip), control_steps
        self.controller_type, self.fetch_env, self.obj_range = controller_type, fetch_env, obj_range
        self.initial_qpos = {} if initial_qpos is None else initial_qpos
        self._want_autotune = bool(autotune) and int(lockstep_warps) == 0 and int(nefc_max) == 0
        self.max_episode_steps = int(max_episode_steps)
        self.goal_source = goal_source
        self.mesh_collision = bool(mesh_collision)
        self.auto_reset = bool(auto_reset)
        self._L = _lib.load()
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self._dev_index = dev_index
        variant = ("mocap" if controller_type == "mocap" else "joint") + ("+hidden" if (reward_type == "reward_shaping" and not has_object) else "")
        self._model, self._desc, self._flat = _device_model(dev_index, variant)
        cfg = flatten.TaskCfg(
            has_object=int(has_object), block_gripper=int(block_gripper), target_in_the_air=int(target_in_the_air),
            reward_type={"sparse": 0, "dense": 1, "reward_shaping": 2}[reward_type], max_episode_steps=self.max_episode_steps,
            frame_skip=self.frame_skip, auto_reset=int(self.auto_reset and goal_source == "device"), nefc_max=int(nefc_max),
            controller_type={"joint": 0, "IK": 1, "mocap": 2}[controller_type], fetch_env=int(bool(fetch_env)), control_steps=int(control_steps),
            mesh_collision=int(bool(mesh_collision)),
            lockstep_warps=int(lockstep_warps), distance_threshold=self.distance_threshold)
        self._cfg = cfg
        with torch.cuda.device(dev_index):
            h = C.c_void_p()
            _lib.check(self._L.mcb_batch_create(self._model, self.num_envs, C.byref(cfg), int(seed), C.byref(h)))
        self._batch = h
        if bounds is not None:
            lo, hi = (np.ascontiguousarray(x, dtype=np.float64) for x in bounds)
            with torch.cuda.device(dev_index):
                _lib.check(self._L.mcb_batch_set_param_ranges(h, lo.ctypes.data_as(C.c_void_p), hi.ctypes.data_as(C.c_void_p)))
        if lat_bounds is not None:
            with torch.cuda.device(dev_index):
                _lib.check(self._L.mcb_batch_set_latency_range(h, *lat_bounds))
        # the optional groups of get_state(): those turned on by a constructor argument or a set_* call
        self._groups = {g for g, on in (("params", bounds is not None), ("latency", lat_bounds is not None)) if on}
        self.obs_dim = self._L.mcb_batch_obs_dim(h)
        self.action_dim = self._L.mcb_batch_action_dim(h)          # 7 (joint, IK), 8 (mocap), 4 (fetch variants) (mycobot.py:90-97)
        N, dev = self.num_envs, self.device
        f64 = torch.float64
        self._obs = torch.zeros(N, self.obs_dim, dtype=f64, device=dev)
        self._ag = torch.zeros(N, 3, dtype=f64, device=dev)
        self._dg = torch.zeros(N, 3, dtype=f64, device=dev)
        self._final_obs = torch.zeros(N, self.obs_dim, dtype=f64, device=dev)
        self._reward = torch.zeros(N, dtype=torch.float32 if reward_type == "sparse" else f64, device=dev)
        self._term = torch.zeros(N, dtype=torch.uint8, device=dev)
        self._trunc = torch.zeros(N, dtype=torch.uint8, device=dev)
        self._succ = torch.zeros(N, dtype=torch.uint8, device=dev)
        self._stats = torch.zeros(8, dtype=f64, device=dev)
        self._contacts = None
        if contact_output:
            # (ncon, geom1 / geom2 / dim, dist pos frame force) for the last forward pass, then for the terminal state of auto-reset envs
            bufs = tuple((torch.zeros(N, dtype=torch.int32, device=dev),
                          torch.full((N, flatten.MAXCON, 3), -1, dtype=torch.int32, device=dev),
                          torch.zeros(N, flatten.MAXCON, flatten.CONTACT_DOUBLES, dtype=f64, device=dev)) for _ in range(2))
            for b in bufs:
                b[1][..., 2] = 0
            torch.cuda.synchronize(dev)
            with torch.cuda.device(dev_index):
                _lib.check(self._L.mcb_set_contact_output(h, *(_ptr(t) for b in bufs for t in b)))
            self._contacts = bufs
        self.initial_gripper_xpos = np.array((self._desc.key_initial_gripper_xpos if fetch_env else self._desc.initial_gripper_xpos)[:])
        self.height_offset = float(self._desc.key_height_offset if fetch_env else self._desc.height_offset)
        self._sampler = ReferenceGoalSampler(N, self.height_offset, self.initial_gripper_xpos[:2], self.has_object,
                                             self.target_in_the_air)
        self.single_action_space = Box(-1.0, 1.0, (self.action_dim,), np.float32)
        self.action_space = Box(-1.0, 1.0, (N, self.action_dim), np.float32)
        self.single_observation_space = Dict(
            desired_goal=Box(-np.inf, np.inf, (3,), np.float64), achieved_goal=Box(-np.inf, np.inf, (3,), np.float64),
            observation=Box(-np.inf, np.inf, (self.obs_dim,), np.float64))
        self.observation_space = Dict(
            desired_goal=Box(-np.inf, np.inf, (N, 3), np.float64), achieved_goal=Box(-np.inf, np.inf, (N, 3), np.float64),
            observation=Box(-np.inf, np.inf, (N, self.obs_dim), np.float64))
        self._closed = False

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _get(self, getter, *arrays):
        """New device tensors [N, *shape] of the given (shape, dtype), filled by one C getter (batch, pointers..., stream)."""
        ts = tuple(torch.empty(self.num_envs, *shape, dtype=dt, device=self.device) for shape, dt in arrays)
        with torch.cuda.device(self._dev_index):
            _lib.check(getter(self._batch, *(_ptr(t) for t in ts), self._stream()))
        return ts

    def _obs_dict(self):
        return {"observation": self._obs, "achieved_goal": self._ag, "desired_goal": self._dg}

    @property
    def goal(self):
        return self._dg

    # ------------------------------------------------------------------ gymnasium surface
    def reset(self, *, seed=None, options=None, mask=None, object_xy=None, goals=None):
        """mycobot.py:506-514.  `mask` restricts the reset to some envs; `object_xy` / `goals` inject sampler
        outputs (float64 [N,2] / [N,3], numpy or torch).  `seed` reseeds the sampler of the (masked) envs like
        `seeding.np_random(seed)` does in the reference: the host protocol sampler (goal_source='reference') and the
        device Philox streams (key := seed, draw counter := 0).  The returned tensors are the env's persistent output
        buffers: the next `reset` / `step` overwrites them (clone to keep)."""
        self._sampler.seed(seed)
        m = None
        if mask is not None:
            m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
        if seed is not None:
            with torch.cuda.device(self._dev_index):
                _lib.check(self._L.mcb_seed(self._batch, int(seed) & 0xFFFFFFFFFFFFFFFF, _ptr(m), self._stream()))
        if self.goal_source == "reference" and goals is None:
            ids = range(self.num_envs) if m is None else torch.nonzero(m).flatten().tolist()
            object_xy, goals = self._sampler.sample(ids)
            if not self.has_object:
                object_xy = None
        xy_t = None if object_xy is None else torch.as_tensor(np.asarray(object_xy) if not torch.is_tensor(object_xy) else object_xy,
                                                              dtype=torch.float64, device=self.device).contiguous()
        g_t = None if goals is None else torch.as_tensor(np.asarray(goals) if not torch.is_tensor(goals) else goals,
                                                         dtype=torch.float64, device=self.device).contiguous()
        with torch.cuda.device(self._dev_index):
            _lib.check(self._L.mcb_reset(self._batch, _ptr(m), _ptr(xy_t), _ptr(g_t), _ptr(self._obs), _ptr(self._ag),
                                        _ptr(self._dg), self._stream()))
        if self._want_autotune and m is None:
            self._want_autotune = False
            self.autotune()
        return self._obs_dict(), {}

    def seed(self, seed=None):
        """Reseed every env's sampler without resetting (SB3 VecEnv.seed)."""
        self._sampler.seed(seed)
        if seed is not None:
            with torch.cuda.device(self._dev_index):
                _lib.check(self._L.mcb_seed(self._batch, int(seed) & 0xFFFFFFFFFFFFFFFF, None, self._stream()))
        return [seed] * self.num_envs

    def reset_host(self, *, seed=None, mask=None, object_xy=None, goals=None):
        """`reset` through HOST buffers (numpy in / numpy out): what a reference-side adapter holding numpy arrays calls."""
        self._sampler.seed(seed)
        N = self.num_envs
        mk = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        if seed is not None:
            md = None if mk is None else torch.as_tensor(mk, device=self.device)
            with torch.cuda.device(self._dev_index):
                _lib.check(self._L.mcb_seed(self._batch, int(seed) & 0xFFFFFFFFFFFFFFFF, _ptr(md), self._stream()))
        if self.goal_source == "reference" and goals is None:
            ids = range(N) if mk is None else np.nonzero(mk)[0].tolist()
            object_xy, goals = self._sampler.sample(ids)
            if not self.has_object:
                object_xy = None
        xy = None if object_xy is None else np.ascontiguousarray(object_xy, dtype=np.float64)
        g = None if goals is None else np.ascontiguousarray(goals, dtype=np.float64)
        out = dict(observation=np.empty((N, self.obs_dim)), achieved_goal=np.empty((N, 3)), desired_goal=np.empty((N, 3)))
        p = lambda x: None if x is None else x.ctypes.data_as(C.c_void_p)
        with torch.cuda.device(self._dev_index):
            _lib.check(self._L.mcb_reset_host(self._batch, p(mk), p(xy), p(g), p(out["observation"]), p(out["achieved_goal"]),
                                             p(out["desired_goal"]), self._stream()))
        return out, {}

    def step(self, actions):
        """mycobot.py:132-205 (joint controller) for all envs; TimeLimit folded in.  `actions`: float32 [N,7]
        torch CUDA tensor (or anything convertible).

        ALIASING CONTRACT: observation / achieved_goal / desired_goal / reward / final_observation are the env's persistent
        device buffers -- the kernel writes straight into them and the next `step` / `reset` overwrites them.  Clone what
        must outlive the next call (`HerReplay.add_step` refuses a `prev_obs` that aliases the new one)."""
        if not torch.is_tensor(actions):
            actions = torch.as_tensor(np.asarray(actions, dtype=np.float32))
        if tuple(actions.shape) != (self.num_envs, self.action_dim):
            raise ValueError(f"Action dimension mismatch. Expected {(self.num_envs, self.action_dim)}, found {tuple(actions.shape)}")
        actions = actions.to(device=self.device, dtype=torch.float32).contiguous()
        with torch.cuda.device(self._dev_index):
            _lib.check(self._L.mcb_step(self._batch, _ptr(actions), _ptr(self._obs), _ptr(self._ag), _ptr(self._dg),
                                       _ptr(self._reward), _ptr(self._term), _ptr(self._trunc), _ptr(self._succ),
                                       _ptr(self._final_obs), self._stream()))
        term, trunc = self._term.bool(), self._trunc.bool()
        info = {"is_success": self._succ.bool()}
        if self.auto_reset:
            done = term | trunc
            if self.goal_source == "reference":
                if bool(done.any()):
                    self._final_obs.copy_(self._obs)
                    if self._contacts is not None:
                        for dst, src in zip(self._contacts[1], self._contacts[0]):
                            dst.copy_(src)
                    self.reset(mask=done)
            info["final_observation"] = self._final_obs
            info["_final_observation"] = done
        return self._obs_dict(), self._reward, term, trunc, info

    def compute_reward(self, achieved_goal, goal, info=None):
        """mycobot.py:289-295 on arbitrary batches (HER relabelling); numpy in -> numpy out, torch in -> torch out."""
        if self.reward_type == "reward_shaping":
            raise NotImplementedError("reward_shaping depends on the live simulation state (mycobot.py:296-298), not on (achieved_goal, goal)")
        is_np = not torch.is_tensor(achieved_goal)
        ag = torch.as_tensor(np.asarray(achieved_goal) if is_np else achieved_goal, dtype=torch.float64, device=self.device).contiguous()
        g = torch.as_tensor(np.asarray(goal) if not torch.is_tensor(goal) else goal, dtype=torch.float64, device=self.device).contiguous()
        if ag.shape != g.shape:
            raise AssertionError("achieved_goal and goal must have the same shape")
        lead = ag.shape[:-1]
        n = int(np.prod(lead)) if len(lead) else 1
        out = torch.empty(lead, dtype=torch.float32 if self.reward_type == "sparse" else torch.float64, device=self.device)
        with torch.cuda.device(self._dev_index):
            _lib.check(self._L.mcb_compute_reward(_ptr(ag), _ptr(g), n, self.distance_threshold,
                                                 0 if self.reward_type == "sparse" else 1, _ptr(out), self._stream()))
        return out.cpu().numpy() if is_np else out

    # ------------------------------------------------------------------ state access (parity replay, checkpointing)
    def get_state(self):
        N, dev = self.num_envs, self.device
        st = dict(qpos=torch.empty(N, 19, dtype=torch.float64, device=dev), qvel=torch.empty(N, 18, dtype=torch.float64, device=dev),
                  ctrl=torch.empty(N, 7, dtype=torch.float64, device=dev), qacc_warmstart=torch.empty(N, 18, dtype=torch.float64, device=dev),
                  goal=torch.empty(N, 3, dtype=torch.float64, device=dev), elapsed=torch.empty(N, dtype=torch.int32, device=dev),
                  qprev=torch.empty(N, 6, dtype=torch.float64, device=dev), mocap=torch.empty(N, 7, dtype=torch.float64, device=dev),
                  env_seed=torch.empty(N, dtype=torch.int64, device=dev), rng_counter=torch.empty(N, dtype=torch.int64, device=dev),
                  ep_return=torch.empty(N, dtype=torch.float64, device=dev))
        for g, (keys, get, _) in _OPTIONAL.items():
            if g in self._groups:
                st.update(zip(keys, getattr(self, get)()))
        with torch.cuda.device(self._dev_index):
            _lib.check(self._L.mcb_get_rng_state(self._batch, _ptr(st["env_seed"]), _ptr(st["rng_counter"]), _ptr(st["ep_return"]), self._stream()))
            _lib.check(self._L.mcb_get_state(self._batch, _ptr(st["qpos"]), _ptr(st["qvel"]), _ptr(st["ctrl"]),
                                            _ptr(st["qacc_warmstart"]), _ptr(st["goal"]), _ptr(st["elapsed"]), _ptr(st["qprev"]),
                                            _ptr(st["mocap"]), self._stream()))
        return st

    def set_state(self, qpos=None, qvel=None, ctrl=None, qacc_warmstart=None, goal=None, elapsed=None, qprev=None, mocap=None,
                  env_seed=None, rng_counter=None, ep_return=None, params=None, param_counter=None, latency=None, latency_counter=None,
                  qfrc_applied=None, xfrc_applied=None):
        """Inverse of `get_state` (a full checkpoint: physics state, goals, episode clocks, RNG streams, running returns, and the
        per-env parameters, actuation latencies and applied forces of a batch that has them)."""
        def prep(x, shape, dt):
            if x is None:
                return None
            t = torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x).to(device=self.device, dtype=dt).contiguous()
            assert tuple(t.shape) == shape, (tuple(t.shape), shape)
            return t

        N = self.num_envs
        ts = [prep(qpos, (N, 19), torch.float64), prep(qvel, (N, 18), torch.float64), prep(ctrl, (N, 7), torch.float64),
              prep(qacc_warmstart, (N, 18), torch.float64), prep(goal, (N, 3), torch.float64), prep(elapsed, (N,), torch.int32),
              prep(qprev, (N, 6), torch.float64), prep(mocap, (N, 7), torch.float64)]
        rs = [prep(env_seed, (N,), torch.int64), prep(rng_counter, (N,), torch.int64), prep(ep_return, (N,), torch.float64)]
        with torch.cuda.device(self._dev_index):
            _lib.check(self._L.mcb_set_state(self._batch, *[_ptr(t) for t in ts], self._stream()))
            if any(t is not None for t in rs):
                _lib.check(self._L.mcb_set_rng_state(self._batch, *[_ptr(t) for t in rs], self._stream()))
        given = dict(params=params, param_counter=param_counter, latency=latency, latency_counter=latency_counter,
                     qfrc_applied=qfrc_applied, xfrc_applied=xfrc_applied)
        for keys, _, set_ in _OPTIONAL.values():
            a, b = (given[k] for k in keys)
            if a is not None or b is not None:
                getattr(self, set_)(a, b)
        torch.cuda.current_stream(self.device).synchronize()

    def get_params(self):
        """(params float64 [N, NPARAM], draw counters int64 [N]) as device tensors: the per-env multipliers (`flatten.PARAM_NAMES`)
        in use and how many parameter draws each env has made since it was seeded.  Without per-env parameters: 1.0 and 0."""
        return self._get(self._L.mcb_get_env_params, ((flatten.NPARAM,), torch.float64), ((), torch.int64))

    def set_params(self, params, draw_counter=None):
        """Fixed per-env multipliers [N, NPARAM] (evaluation, system identification); either argument may be None.  Turns per-env
        parameters on if the batch has none; resets keep redrawing only if `param_ranges` are set."""
        if self.mesh_collision:
            raise ValueError("per-env parameters are not supported with mesh_collision=True")
        N = self.num_envs
        p = c = None
        if params is not None:
            p = torch.as_tensor(np.asarray(params) if not torch.is_tensor(params) else params).to(device=self.device, dtype=torch.float64).contiguous()
            if tuple(p.shape) != (N, flatten.NPARAM):
                raise ValueError(f"params must have shape {(N, flatten.NPARAM)}, got {tuple(p.shape)}")
            if not bool(torch.isfinite(p).all()) or not bool((p > 0).all()):
                raise ValueError("params must be finite and > 0")
        if draw_counter is not None:
            c = torch.as_tensor(np.asarray(draw_counter) if not torch.is_tensor(draw_counter) else draw_counter).to(device=self.device, dtype=torch.int64).contiguous()
            if tuple(c.shape) != (N,):
                raise ValueError(f"draw_counter must have shape {(N,)}, got {tuple(c.shape)}")
        with torch.cuda.device(self._dev_index):
            _lib.check(self._L.mcb_set_env_params(self._batch, _ptr(p), _ptr(c), self._stream()))
        self._groups.add("params")

    def get_latency(self):
        """(latency int32 [N], draw counters int64 [N]) as device tensors: each env's actuation latency in substeps and how many
        latency draws it has made since it was seeded.  Without latency: 0 and 0."""
        return self._get(self._L.mcb_get_env_latency, ((), torch.int32), ((), torch.int64))

    def set_latency(self, latency, draw_counter=None):
        """Fixed per-env actuation latencies [N] in substeps, integers in [0, frame_skip] (evaluation, system identification); either
        argument may be None.  Turns latency on if the batch has none; resets keep redrawing only if `actuation_latency` is set."""
        if self.mesh_collision:
            raise ValueError("actuation latency is not supported with mesh_collision=True")
        N = self.num_envs
        d = c = None
        if latency is not None:
            d = torch.as_tensor(np.asarray(latency) if not torch.is_tensor(latency) else latency)
            if d.dtype.is_floating_point or d.dtype.is_complex or d.dtype == torch.bool:
                raise ValueError(f"latency must be an integer tensor, got {d.dtype}")
            if tuple(d.shape) != (N,):
                raise ValueError(f"latency must have shape {(N,)}, got {tuple(d.shape)}")
            if N and (int(d.min()) < 0 or int(d.max()) > self.frame_skip):
                raise ValueError(f"latency must lie in [0, frame_skip={self.frame_skip}]")
            d = d.to(device=self.device, dtype=torch.int32).contiguous()
        if draw_counter is not None:
            c = torch.as_tensor(np.asarray(draw_counter) if not torch.is_tensor(draw_counter) else draw_counter).to(device=self.device, dtype=torch.int64).contiguous()
            if tuple(c.shape) != (N,):
                raise ValueError(f"draw_counter must have shape {(N,)}, got {tuple(c.shape)}")
        with torch.cuda.device(self._dev_index):
            _lib.check(self._L.mcb_set_env_latency(self._batch, _ptr(d), _ptr(c), self._stream()))
        self._groups.add("latency")

    def get_applied_forces(self):
        """(qfrc_applied float64 [N, 18], xfrc_applied float64 [N, 13, 6]) as device tensors: the forces the step applies (see
        `set_applied_forces`).  Without forces: zeros."""
        return self._get(self._L.mcb_get_env_applied, ((flatten.NV,), torch.float64), ((flatten.NB, 6), torch.float64))

    def set_applied_forces(self, qfrc_applied=None, xfrc_applied=None):
        """Per-env external forces, MuJoCo's `data.qfrc_applied` and `data.xfrc_applied` on the reduced model (DESIGN.md section 11):
        `qfrc_applied` [N, 18] generalized forces, `xfrc_applied` [N, 13, 6] a world-frame force (0:3) and torque (3:6) per body of
        `flatten.BODY_NAMES`, applied at the body's centre of mass.  Torch or numpy input; None leaves that array as it is.  The
        forces persist: they act on every substep of every following step until set again, and every reset of an env sets its
        forces to zero.  In reach envs without reward_shaping the cube is frozen and its forces are ignored.  The first call turns
        forces on (it synchronises).  Every call checks its input on the host (a synchronisation), so it is not capturable itself: call
        it between the replays of a captured step graph, which then use the new values (the C call `mcb_set_env_applied` on checked
        device arrays is one kernel on the stream and can be captured).  Not available with mesh_collision."""
        q, x = flatten.applied_forces(qfrc_applied, xfrc_applied, self.num_envs, self.mesh_collision)
        q = None if q is None else q.to(self.device)
        x = None if x is None else x.to(self.device)
        with torch.cuda.device(self._dev_index):
            _lib.check(self._L.mcb_set_env_applied(self._batch, _ptr(q), _ptr(x), self._stream()))
        self._groups.add("forces")

    def contacts(self, final=False):
        """The contacts of each env's last forward pass (MuJoCo's `data.contact` with `mj_contactForce`), as named views of the env's
        persistent device buffers (batches made with `contact_output=True`; same aliasing contract as `step`: the next step, reset or
        forward overwrites them, clone to keep):
          ncon int32 [N]; geom int32 [N, 24, 2] (geom1, geom2: indices into `flatten.GEOM_NAMES`); dim int32 [N, 24] (condim);
          dist [N, 24]; pos [N, 24, 3] (world); frame [N, 24, 3, 3] (rows: normal from geom1 to geom2, then the two tangents);
          force [N, 24, 6]: the force on geom2 (geom1 takes its opposite) in the contact frame: normal, tangent 1, tangent 2,
          torsional (condim 4), 0, 0.
        Slots >= ncon are zero with geom ids -1.  After a step: the last substep's contacts (the block_gripper forward pass's if
        block_gripper), or the reset's for an env that auto-reset.  `final=True`: for envs that auto-reset in the last step, the
        contacts of the terminal state (those the step's reward saw); rows of other envs are left as they were.  The world-frame
        force of every contact is
          torch.einsum("nckj,nck->ncj", c["frame"], c["force"][..., :3])   # frame[..., :3, :].transpose . force[..., :3]
        Contacts the last layout tier drops for lack of constraint rows are not reported (DESIGN.md section 12)."""
        if self._contacts is None:
            raise RuntimeError("contact output is off: make the env with contact_output=True")
        n, g, c = self._contacts[1 if final else 0]
        return dict(ncon=n, geom=g[..., :2], dim=g[..., 2], dist=c[..., 0], pos=c[..., 1:4], frame=c[..., 4:13].unflatten(-1, (3, 3)),
                    force=c[..., 13:19])

    def autotune(self, actions=None, steps_per_candidate=0):
        """Pick the step kernel's lockstep grouping for this batch (explicit: `step` never tunes; the constructor's
        `autotune=True` calls this once at the end of the first full `reset`).  Synchronises; the state is restored exactly.
        Returns the chosen number of warps per group."""
        self._want_autotune = False
        a = None if actions is None else torch.as_tensor(actions).to(device=self.device, dtype=torch.float32).contiguous()
        with torch.cuda.device(self._dev_index):
            return _lib.check(self._L.mcb_autotune(self._batch, _ptr(a), int(steps_per_candidate), self._stream()))

    @property
    def lockstep_warps(self):
        return int(self._L.mcb_batch_lockstep_warps(self._batch))

    def last_fallback_envs(self):
        """(envs of the most recent step that left the common shared-memory layout for the middle tier, envs that also
        left the middle tier for the last one); synchronises."""
        last = C.c_int32(0)
        with torch.cuda.device(self._dev_index):
            n = _lib.check(self._L.mcb_last_fallback_envs(self._batch, C.byref(last), self._stream()))
        return n, int(last.value)

    def last_fallback_list(self, cap=None):
        """Indices of the envs of the most recent step that left the common layout (host list); synchronises."""
        cap = self.num_envs if cap is None else int(cap)
        buf = np.zeros(max(cap, 1), dtype=np.int32)
        with torch.cuda.device(self._dev_index):
            n = _lib.check(self._L.mcb_last_fallback_list(self._batch, buf.ctypes.data_as(C.c_void_p), cap, self._stream()))
        return buf[:min(n, cap)].copy()

    @property
    def total_launches(self):
        return int(self._L.mcb_total_launches(self._batch))

    def forward(self):
        """mj_forward on every env (refreshes frames, qacc_warmstart and the observation buffers)."""
        with torch.cuda.device(self._dev_index):
            _lib.check(self._L.mcb_forward(self._batch, _ptr(self._obs), _ptr(self._ag), _ptr(self._dg), self._stream()))
        return self._obs_dict()

    def debug_forward(self, env=0):
        """Stage-level tap for parity tests: runs forward and returns intermediate quantities of one env."""
        cap = 4 + 18 * 18 + 5 * 18 + 13 * 12 + 256 * 18 + 2 * 256 + 7 * 32      # at least the library's dump (176 rows, 24 contacts)
        buf = np.zeros(cap)
        with torch.cuda.device(self._dev_index):
            _lib.check(self._L.mcb_debug_forward(self._batch, int(env), 0, buf.ctypes.data_as(C.c_void_p), cap, self._stream()))
        nefc, ncon, iters, overflow = int(buf[0]), int(buf[1]), int(buf[2]), int(buf[3])
        o = 4
        out = dict(nefc=nefc, ncon=ncon, iters=iters, overflow=overflow)
        out["M"] = buf[o:o + 324].reshape(18, 18).copy(); o += 324
        for k in ["qfrc_bias", "qfrc_smooth", "qacc_smooth", "qacc", "qfrc_constraint"]:
            out[k] = buf[o:o + 18].copy(); o += 18
        out["xpos"] = buf[o:o + 39].reshape(13, 3).copy(); o += 39
        out["xmat"] = buf[o:o + 117].reshape(13, 3, 3).copy(); o += 117
        out["efc_J"] = buf[o:o + nefc * 18].reshape(nefc, 18).copy(); o += nefc * 18
        out["efc_aref"] = buf[o:o + nefc].copy(); o += nefc
        out["efc_D"] = buf[o:o + nefc].copy(); o += nefc
        con = buf[o:o + 7 * ncon].reshape(ncon, 7)
        out["contact_dist"], out["contact_pos"], out["contact_normal"] = con[:, 0].copy(), con[:, 1:4].copy(), con[:, 4:7].copy()
        return out

    def stats(self, reset=True):
        """Episode statistics accumulated on device: episodes, successes, return_sum, length_sum, env_steps,
        row_overflows, solver_iterations, substeps."""
        with torch.cuda.device(self._dev_index):
            _lib.check(self._L.mcb_stats(self._batch, _ptr(self._stats), int(reset), self._stream()))
        return self._stats

    def step_host(self, actions_np, out=None, want_final_obs=False):
        """The same step through HOST buffers (numpy): H2D of actions and D2H of all results inside the call."""
        a = np.ascontiguousarray(actions_np, dtype=np.float32)
        assert a.shape == (self.num_envs, self.action_dim)
        N = self.num_envs
        if out is None:
            # page-locked result buffers (numpy views of pinned torch tensors): the library copies into them directly
            pin = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=True).numpy()
            out = dict(observation=pin((N, self.obs_dim), torch.float64), achieved_goal=pin((N, 3), torch.float64),
                       desired_goal=pin((N, 3), torch.float64),
                       reward=pin((N,), torch.float32 if self.reward_type == "sparse" else torch.float64),
                       terminated=pin((N,), torch.uint8), truncated=pin((N,), torch.uint8), is_success=pin((N,), torch.uint8))
            if want_final_obs:
                out["final_observation"] = pin((N, self.obs_dim), torch.float64)
        p = lambda x: x.ctypes.data_as(C.c_void_p)
        with torch.cuda.device(self._dev_index):
            _lib.check(self._L.mcb_step_host(self._batch, p(a), p(out["observation"]), p(out["achieved_goal"]), p(out["desired_goal"]),
                                            p(out["reward"]), p(out["terminated"]), p(out["truncated"]), p(out["is_success"]),
                                            p(out["final_observation"]) if "final_observation" in out else None, self._stream()))
        return out

    @property
    def last_step_launches(self):
        return self._L.mcb_last_step_launches(self._batch)

    def close(self):
        if not self._closed and self._batch:
            self._L.mcb_batch_destroy(self._batch)
            self._closed = True

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ------------------------------------------------------------------ multi-GPU: env-dimension sharding
def shard_envs(total_envs, rank, world_size):
    """Contiguous block of envs owned by `rank` (independent units, no data-path collective)."""
    base, rem = divmod(total_envs, world_size)
    start = rank * base + min(rank, rem)
    return start, base + (1 if rank < rem else 0)


def all_reduce_stats(stats):
    """Sum the 8-double statistics vector over ranks (NCCL on GPU tensors, gloo on CPU tensors)."""
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    return stats
