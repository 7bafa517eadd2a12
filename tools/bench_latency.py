"""Cost of per-env actuation latency: pick, push, IK and mocap at the bench.py sizes, each as a plain batch, a batch with nominal
parameters (the step kernels latency runs in, every latency 0) and a batch with latencies drawn from (0, frame_skip) at every reset,
timed in one process with the three alternated.

    python tools/bench_latency.py [--steps 20] [--rounds 3] [--preroll 50]

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
FRAME_SKIP = 20
VARIANTS = {"plain": {}, "nominal": {"param_ranges": {k: (1.0, 1.0) for k in flatten.PARAM_NAMES}},
            "latency": {"actuation_latency": (0, FRAME_SKIP)}}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


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
        envs = {v: MyCobotVectorEnv(num_envs=n, seed=1000, frame_skip=FRAME_SKIP, **extra, **kw) for v, extra in VARIANTS.items()}
        gen = torch.Generator(device="cuda")
        gen.manual_seed(0)
        acts = [torch.rand(n, adim, device="cuda", generator=gen) * 2 - 1 for _ in range(8)]
        for e in envs.values():
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
        print(json.dumps(dict(workload=w, num_envs=n, ms_per_step=med, all=times, lockstep={v: e.lockstep_warps for v, e in envs.items()},
                              nominal_vs_plain=med["nominal"] / med["plain"], latency_vs_plain=med["latency"] / med["plain"],
                              latency_vs_nominal=med["latency"] / med["nominal"])), flush=True)
        for e in envs.values():
            e.close()


if __name__ == "__main__":
    main()
