"""Cost of the contact output: pick, push, IK and mocap at the bench.py sizes, each as a plain batch, a batch with nominal parameters
(the step kernels the contact output runs in) and a batch with contact output on (contacts and final contacts), timed in one process
with the three alternated.  All three simulate the same motion bit for bit; `left_tier0_tier1` reports how many envs of one more step
left the common layout.

    python tools/bench_contacts.py [--steps 20] [--rounds 3] [--preroll 50]

Device-event timing of `steps` env-steps per round after `preroll` untimed steps (steady-state episode mix, auto-resets included);
prints the card's name, power limit and max SM clock, then one JSON line per workload with the median ms / step of each variant."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
from mycobotgym_b200 import flatten  # noqa: E402
from mycobotgym_b200.vector_env import MyCobotVectorEnv  # noqa: E402

WORKLOADS = {   # bench.py's workloads and sizes
    "pick": (dict(has_object=True, reward_type="sparse"), 16384, 7),
    "push": (dict(has_object=True, block_gripper=True, target_in_the_air=False, reward_type="sparse"), 16384, 7),
    "ik": (dict(has_object=True, reward_type="sparse", controller_type="IK"), 16384, 7),
    "mocap": (dict(has_object=True, reward_type="sparse", controller_type="mocap", model_path="./assets/mycobot280_mocap.xml"), 16384, 8),
}
VARIANTS = ("plain", "nominal", "contacts")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def make(variant, kw, n):
    extra = {"param_ranges": {k: (1.0, 1.0) for k in flatten.PARAM_NAMES}} if variant == "nominal" else {}
    return MyCobotVectorEnv(num_envs=n, seed=1000, contact_output=variant == "contacts", **extra, **kw)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--preroll", type=int, default=50)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    args = ap.parse_args()
    print("card:", card(), flush=True)
    for w in args.workloads.split(","):
        kw, n, adim = WORKLOADS[w]
        envs = {v: make(v, kw, n) for v in VARIANTS}
        gen = torch.Generator(device="cuda")
        gen.manual_seed(0)
        acts = [torch.rand(n, adim, device="cuda", generator=gen) * 2 - 1 for _ in range(8)]
        for v, e in envs.items():
            e.reset()            # (the first full reset autotunes the lockstep grouping, as in bench.py)
            for t in range(args.preroll):
                e.step(acts[t % 8])
        torch.cuda.synchronize()
        times = {v: [] for v in envs}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(args.rounds):
            for v, e in envs.items():
                e0.record()
                for t in range(args.steps):
                    e.step(acts[t % 8])
                e1.record()
                e1.synchronize()
                times[v].append(e0.elapsed_time(e1) / args.steps)
        med = {v: sorted(x)[len(x) // 2] for v, x in times.items()}
        left = {}
        for v, e in envs.items():
            e.step(acts[0])
            left[v] = e.last_fallback_envs()
        c = envs["contacts"].contacts()
        print(json.dumps(dict(workload=w, num_envs=n, ms_per_step=med, all=times, lockstep={v: e.lockstep_warps for v, e in envs.items()},
                              left_tier0_tier1=left, mean_ncon=float(c["ncon"].double().mean()),
                              nominal_vs_plain=med["nominal"] / med["plain"], contacts_vs_nominal=med["contacts"] / med["nominal"],
                              contacts_vs_plain=med["contacts"] / med["plain"])), flush=True)
        for e in envs.values():
            e.close()


if __name__ == "__main__":
    main()
