"""Workload of the guard-word (MCB_CANARY) build: every controller, every layout tier, resets, reward shaping, a held grasp.
Run with MCB_LIB pointing at libmycobot_b200_canary.so; prints `CANARY_OK <anomalies>` (tests/test_gpu_canary.py).
`--params`: the same cases with per-env physics parameters drawn at every reset (tests/test_gpu_env_params.py); the hull-collision
cases, which do not support them, are left out.  `--latency`: the same cases with an actuation latency drawn from (0, frame_skip) at
every reset (tests/test_gpu_latency.py); the hull-collision cases are left out too.  `--forces`: the same cases with random applied
forces (qfrc_applied and xfrc_applied) set before every step (tests/test_gpu_applied_forces.py); the hull-collision cases are left
out too.  `--contacts`: the same cases with contact output on (tests/test_gpu_contacts.py), plus a forward pass; the hull-collision
cases are left out too."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
from mycobotgym_b200 import _lib  # noqa: E402
from mycobotgym_b200.vector_env import MyCobotVectorEnv  # noqa: E402

assert "canary" in _lib.LIB_PATH, _lib.LIB_PATH
PARAMS = "--params" in sys.argv[1:]
LATENCY = "--latency" in sys.argv[1:]
FORCES = "--forces" in sys.argv[1:]
CONTACTS = "--contacts" in sys.argv[1:]
RANGES = {"cube_mass": (0.5, 2.0), "friction": (0.7, 1.3), "gain": (0.8, 1.2), "arm_damping": (0.5, 2.0)}
gen = torch.Generator(device="cuda")
gen.manual_seed(0)
total = 0.0
g = np.load(os.path.join(ROOT, "tests", "golden", "grasp_pick_sparse.npz"))
CASES = [
    ("pick", dict(has_object=True, reward_type="sparse"), 2048, 7, 30),
    ("pick tier 1 only", dict(has_object=True, reward_type="sparse", nefc_max=88), 256, 7, 6),
    ("pick tier 2 only", dict(has_object=True, reward_type="sparse", nefc_max=128), 256, 7, 6),
    ("push", dict(has_object=True, block_gripper=True, target_in_the_air=False, reward_type="sparse", lockstep_warps=16), 2048, 7, 30),
    ("reach", dict(has_object=False, reward_type="dense"), 1024, 7, 20),
    ("reach + reward shaping", dict(has_object=False, reward_type="reward_shaping"), 256, 7, 10),
    ("pick + reward shaping", dict(has_object=True, reward_type="reward_shaping"), 256, 7, 10),
    ("ik", dict(has_object=True, reward_type="sparse", controller_type="IK", lockstep_warps=16), 1024, 7, 8),
    ("fetch ik", dict(has_object=True, reward_type="dense", controller_type="IK", fetch_env=True), 256, 4, 6),
    ("mocap", dict(has_object=True, reward_type="sparse", controller_type="mocap", model_path="./assets/mycobot280_mocap.xml", lockstep_warps=16), 1024, 8, 12),
    ("mocap + hull collisions", dict(has_object=True, reward_type="sparse", controller_type="mocap", model_path="./assets/mycobot280_mocap.xml", lockstep_warps=16,
                                     mesh_collision=True), 128, 8, 10),
    ("push + hull collisions", dict(has_object=True, block_gripper=True, target_in_the_air=False, reward_type="sparse", mesh_collision=True), 128, 7, 8),
    ("fetch mocap", dict(has_object=True, reward_type="dense", controller_type="mocap", fetch_env=True, model_path="./assets/mycobot280_mocap.xml"), 256, 4, 6),
]
for name, kw, n, adim, steps in CASES:
    if PARAMS:
        if kw.get("mesh_collision"):
            continue
        kw = dict(kw, param_ranges=RANGES)
    if LATENCY:
        if kw.get("mesh_collision"):
            continue
        kw = dict(kw, actuation_latency=(0, 20))
    if (FORCES or CONTACTS) and kw.get("mesh_collision"):
        continue
    if CONTACTS:
        kw = dict(kw, contact_output=True)
    env = MyCobotVectorEnv(num_envs=n, seed=3, autotune=False, **kw)
    env.reset()
    env.set_state(elapsed=torch.arange(n, dtype=torch.int32) % 50)
    if name == "pick":          # plus a block of held grasps: coupled rows, middle tier
        st = env.get_state()
        k = 200
        rep = lambda x: torch.as_tensor(np.repeat(np.asarray(x)[None], k, 0), device="cuda")
        for key, val in (("qpos", g["qpos0"]), ("qvel", g["qvel0"]), ("ctrl", g["ctrl0"]), ("qacc_warmstart", g["warm0"])):
            st[key][:k] = rep(val)
        env.set_state(qpos=st["qpos"], qvel=st["qvel"], ctrl=st["ctrl"], qacc_warmstart=st["qacc_warmstart"])
    for t in range(steps):
        a = torch.rand(n, adim, device="cuda", generator=gen) * 2 - 1
        if name == "pick":
            a[:200, :6] = torch.as_tensor(g["qpos0"][:6], device="cuda", dtype=torch.float32)
            a[:200, 6] = 0.8
        if FORCES:
            env.set_applied_forces(torch.randn(n, 18, device="cuda", generator=gen) * 0.05,
                                   torch.randn(n, 13, 6, device="cuda", generator=gen) * torch.tensor([0.2] * 3 + [0.01] * 3, device="cuda"))
        env.step(a)
        if t == 2:
            env.reset(mask=(torch.arange(n) % 3 == 0))
    if CONTACTS:
        env.forward()
    s = env.stats().cpu().numpy()
    print(f"{name:24s} env_steps {int(s[4]):7d}  left tier 0 / 1 in the last step {env.last_fallback_envs()}  anomalies {s[5]:.0f}", flush=True)
    total += s[5]
    env.close()
torch.cuda.synchronize()
print("CANARY_OK" if total < 1e6 else "CANARY_HIT", total)
