"""Cost of the per-env features: pick, push, IK and mocap at the bench.py sizes, each as a set of batch variants timed in one process
with the variants alternated:
  plain          no per-env features (the default step kernels)
  nominal        per-env parameters with every range (1, 1): the step kernels every feature below runs in
  params         per-env parameters drawn from randomised ranges at every reset
  latency        actuation latencies drawn from (0, frame_skip) at every reset
  zero_forces    applied forces on, all zero
  random_forces  random forces rewritten before every step (one mcb_set_env_applied call on device tensors prepared before the timed
                 window: the kernel path, without set_applied_forces' host-side checks)
  contacts       contact output on (contacts and final contacts)
Random pushes change the simulated motion (more contacts, more envs in the upper layout tiers), so `random_forces` measures a different
workload as well as the force path; `left_tier0_tier1` reports how many envs of one more step left the common layout.

    python tools/bench_env_features.py [--steps 20] [--rounds 3] [--preroll 50] [--variants plain,nominal,...] [--workloads pick,...]

Device-event timing of `steps` env-steps per round after `preroll` untimed steps (steady-state episode mix, auto-resets included);
prints the card's name, power limit and max SM clock, then one JSON line per workload with the median ms / step of each variant and
its ratio to `plain` and to `nominal` (where those variants ran)."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
from mycobotgym_b200 import _lib, flatten  # noqa: E402
from mycobotgym_b200.vector_env import MyCobotVectorEnv  # noqa: E402

WORKLOADS = {   # bench.py's workloads and sizes
    "pick": (dict(has_object=True, reward_type="sparse"), 16384, 7),
    "push": (dict(has_object=True, block_gripper=True, target_in_the_air=False, reward_type="sparse"), 16384, 7),
    "ik": (dict(has_object=True, reward_type="sparse", controller_type="IK"), 16384, 7),
    "mocap": (dict(has_object=True, reward_type="sparse", controller_type="mocap", model_path="./assets/mycobot280_mocap.xml"), 16384, 8),
}
FRAME_SKIP = 20
RANDOM = {"cube_mass": (0.5, 2.0), "friction": (0.7, 1.3), "gain": (0.8, 1.2), "arm_damping": (0.5, 2.0)}
VARIANTS = {    # constructor arguments of each variant (the force variants turn forces on after construction)
    "plain": {},
    "nominal": {"param_ranges": {k: (1.0, 1.0) for k in flatten.PARAM_NAMES}},
    "params": {"param_ranges": RANDOM},
    "latency": {"actuation_latency": (0, FRAME_SKIP)},
    "zero_forces": {},
    "random_forces": {},
    "contacts": {"contact_output": True},
}


def ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def make(variant, kw, n):
    e = MyCobotVectorEnv(num_envs=n, seed=1000, frame_skip=FRAME_SKIP, **VARIANTS[variant], **kw)
    if variant.endswith("_forces"):
        e.set_applied_forces(torch.zeros(n, flatten.NV, dtype=torch.float64, device="cuda"))
    return e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--preroll", type=int, default=50)
    ap.add_argument("--variants", default=",".join(VARIANTS))
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    args = ap.parse_args()
    variants = args.variants.split(",")
    for v in variants:
        if v not in VARIANTS:
            ap.error(f"unknown variant {v!r} (known: {', '.join(VARIANTS)})")
    print("card:", card(), flush=True)
    for w in args.workloads.split(","):
        kw, n, adim = WORKLOADS[w]
        envs = {v: make(v, kw, n) for v in variants}
        gen = torch.Generator(device="cuda")
        gen.manual_seed(0)
        acts = [torch.rand(n, adim, device="cuda", generator=gen) * 2 - 1 for _ in range(8)]
        # random pushes: generalized forces on every dof, a wrench on every body (cube: a tenth of its weight; arm: 0.2 N, 0.01 N m)
        scale = torch.tensor([0.2] * 3 + [0.01] * 3, dtype=torch.float64, device="cuda").repeat(flatten.NB, 1)
        scale[flatten.CUBE_BODY] = torch.tensor([0.008] * 3 + [1e-4] * 3)
        qf = [torch.randn(n, flatten.NV, dtype=torch.float64, device="cuda", generator=gen) * 0.02 for _ in range(8)]
        xf = [torch.randn(n, flatten.NB, 6, dtype=torch.float64, device="cuda", generator=gen) * scale for _ in range(8)]

        def step(v, e, t):
            if v == "random_forces":
                _lib.check(e._L.mcb_set_env_applied(e._batch, ptr(qf[t % 8]), ptr(xf[t % 8]), e._stream()))
            e.step(acts[t % 8])

        for v, e in envs.items():
            e.reset()            # (the first full reset autotunes the lockstep grouping, as in bench.py)
            for t in range(args.preroll):
                step(v, e, t)
        torch.cuda.synchronize()
        times = {v: [] for v in envs}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(args.rounds):
            for v, e in envs.items():
                e0.record()
                for t in range(args.steps):
                    step(v, e, t)
                e1.record()
                e1.synchronize()
                times[v].append(e0.elapsed_time(e1) / args.steps)
        med = {v: sorted(x)[len(x) // 2] for v, x in times.items()}
        left = {}        # envs of one more step that left the common layout (contacts): random pushes change the simulated motion
        for v, e in envs.items():
            step(v, e, 0)
            left[v] = e.last_fallback_envs()
        out = dict(workload=w, num_envs=n, ms_per_step=med, all=times, lockstep={v: e.lockstep_warps for v, e in envs.items()},
                   left_tier0_tier1=left)
        if "contacts" in envs:
            out["mean_ncon"] = float(envs["contacts"].contacts()["ncon"].double().mean())
        for base in ("plain", "nominal"):
            if base in med:
                out[f"vs_{base}"] = {v: m / med[base] for v, m in med.items()}
        print(json.dumps(out), flush=True)
        for e in envs.values():
            e.close()


if __name__ == "__main__":
    main()
