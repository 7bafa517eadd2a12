#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched myCobot step on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload pick|reach|push] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one `step()` of every env of the workload = 20 physics substeps (joint controller) +
observation / reward / success / auto-reset, i.e. one launch of the fused env kernel.  Default workload
= BASELINE.json configs[3]: pick-and-place, 16384 envs per GPU, random actions, auto-reset with goal
resampling (weak scaling: per-GPU work fixed).  For N>1 the driver launches this under torchrun, one
rank per GPU; envs are sharded with no data-path collective, NCCL only reduces the 8-double statistics
vector once at the end of the timed region.

`--impl reference`: the reference's CPU path.  MuJoCo 2.3.2 is not installable here, so this arm times the
repo's CPU restatement (oracle/, kind "port") on all host cores, same metric and workload, bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (env kwargs, envs per GPU, algorithmic FLOP per env-step).  FLOP: INSTRUMENTED count of the CPU oracle's arithmetic
    # on the same random-action protocol (tools/count_flops.py: every add / mul / div / sqrt of oracle/mjc_oracle.c counted by a
    # wrapper type; frozen in BASELINE.md section 4; FMA = 2).  Round 1 used the survey's estimates (pick 1.25e6).
    "reach": (dict(has_object=False, reward_type="dense"), 4096, 0.600e6),
    "push": (dict(has_object=True, block_gripper=True, target_in_the_air=False, reward_type="sparse"), 16384, 1.254e6),
    "pick": (dict(has_object=True, reward_type="sparse"), 16384, 1.036e6),
    # IK controller (the reference's default): 5 x (6x6 DLS solve + 20 substeps) per env-step
    "ik": (dict(has_object=True, reward_type="sparse", controller_type="IK"), 16384, 5.180e6),
    # mocap controller on the mocap model variant: a 6-row weld drags the arm (13 equality rows instead of 7)
    "mocap": (dict(has_object=True, reward_type="sparse", controller_type="mocap", model_path="./assets/mycobot280_mocap.xml"), 16384, 1.247e6),
    # contact-rich regime (what a trained pick-and-place policy looks like): EVERY env holds the cube between the finger layers
    # (tests/golden/grasp_pick_sparse.npz replicated + small velocity noise), no auto-reset, the action keeps the grip closed
    "grasp": (dict(has_object=True, reward_type="sparse", auto_reset=False), 16384, 1.406e6),
}
METRIC = "env-steps/sec (pick-and-place, 16K envs/GPU) at 1/2/4/8 B200 vs CPU MuJoCo"
UNIT = "env-steps/s"
DUMP_BYTES = 60 * 10**6      # array data of --dump-outputs: with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir, step_out):
    """Writes what `env.step` returned in the last timed step, one DIR/<name>.npy per array: float64 stays float64, the
    rest becomes float32.  Above DUMP_BYTES in all, every array keeps the same seeded sample of envs (sorted), whose
    indices go to env_index.npy.  Inputs are seeded, so two builds run with the same arguments can be compared file by file."""
    import torch

    obs, reward, term, trunc, info = step_out
    arrays = dict(obs, reward=reward, terminated=term, truncated=trunc, **info)
    arrays = {k: v if v.dtype == torch.float64 else v.to(torch.float32) for k, v in arrays.items()}
    n = reward.shape[0]
    row_bytes = sum(v[0].numel() * v.element_size() for v in arrays.values())
    if n * row_bytes > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // (row_bytes + 8), replace=False))
        rows = torch.as_tensor(idx, device=reward.device)
        arrays = {k: v.index_select(0, rows) for k, v in arrays.items()}
        arrays["env_index"] = torch.as_tensor(idx, dtype=torch.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v.cpu().numpy())


def her_relabel_leg(env, acts, dev, flush):
    """SURVEY 8d config 3 "timed separately": HER relabelling (train.py:93-97, n_sampled_goal=4) of a batch of 4 * N
    transitions out of a device-resident replay ring filled by 52 rollout steps.  HBM-bound gather; reported against
    MEASURED_PEAKS.json's copy bandwidth.  Algorithmic bytes per sample: rows read + rows written (DESIGN.md)."""
    import torch

    from mycobotgym_b200.her import DeviceHerReplayBuffer

    n, T = env.num_envs, 64
    buf = DeviceHerReplayBuffer(T * n, env, seed=7)
    obs = {k: v.clone() for k, v in env._obs_dict().items()}
    for t in range(52):
        a = acts[t % acts.shape[0]]
        out = env.step(a)
        buf.add_step(obs, a, out)
        obs = {k: v.clone() for k, v in out[0].items()}
    def timed(B):
        outb = buf.alloc_batch(B)              # reused output tensors: the timed interval holds the memset + the gather kernel only
        for _ in range(3):
            buf.sample(B, out=outb)
        reps = 10
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for r in range(reps):
            flush.zero_()
            ev[r][0].record()
            buf.sample(B, out=outb)
            ev[r][1].record()
        torch.cuda.synchronize()
        assert buf.failed_samples() == 0
        return sum(a.elapsed_time(b) for a, b in ev) / reps

    B = 4 * n
    ms = timed(B)
    B_large = 64 * n                           # 1 M samples: the same kernel out of the launch-latency regime (the reference's batch is 4 n)
    ms_large = timed(B_large)
    od, ad = env.obs_dim, env.action_dim
    bytes_per_sample = 2 * ((2 * od + 9) * 8 + ad * 4 + 4) + 2 + 8 + 4      # rows read + rows written, flags + episode table, dones out
    peak = None
    try:
        peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass
    gbs = B * bytes_per_sample / (ms * 1e-3) / 1e9
    buf.close()
    return {"batch": B, "ms": ms, "samples_per_s": B / (ms * 1e-3), "bytes_per_sample": bytes_per_sample, "achieved_GBps": gbs,
            "peak_GBps": peak, "frac": (gbs / peak) if peak else None, "ring": f"{T} steps x {n} envs, 52 filled",
            "large_batch": {"batch": B_large, "ms": ms_large, "achieved_GBps": B_large * bytes_per_sample / (ms_large * 1e-3) / 1e9,
                            "frac": (B_large * bytes_per_sample / (ms_large * 1e-3) / 1e9 / peak) if peak else None,
                            "note": "the 4 n batch takes ~0.05 ms: launch-latency scale; at 64 n the gather runs at its bandwidth"},
            "note": "mcb_her_sample: future-strategy relabel + compute_reward, one lane draws a sample, the warp copies 32 rows, 8 in flight; 1 kernel + 1 memset per call"}


def _cpu_worker(job):
    workload, tid, envs_per_worker, steps = job
    from mycobotgym_b200 import mjcf
    from oracle.oracle import OracleEnv

    kw, _, _ = WORKLOADS[workload]
    flat = mjcf.load_compiled(mjcf.COMPILED_MOCAP if kw.get("controller_type") == "mocap" else mjcf.COMPILED_JOINT)
    adim = 8 if kw.get("controller_type") == "mocap" else 7
    okw = dict(has_object=kw.get("has_object", True), block_gripper=kw.get("block_gripper", False),
               target_in_the_air=kw.get("target_in_the_air", True), reward_type=kw.get("reward_type", "sparse"),
               controller_type=kw.get("controller_type", "joint"))
    envs = [OracleEnv(flat, **okw) for _ in range(envs_per_worker)]
    rng = np.random.default_rng(tid)
    for e in envs:
        e.reset(seed=tid)
    envs[0].step(np.zeros(adim, dtype=np.float32))
    t0 = time.perf_counter()
    n = 0
    for _ in range(steps):
        for e in envs:
            a = rng.uniform(-1, 1, adim).astype(np.float32)
            o, r, te, tr, info = e.step(a)
            if te or tr:
                e.reset()
            n += 1
    return n, time.perf_counter() - t0


def cpu_port_throughput(workload, budget_env_steps, workers=None):
    """Times the CPU restatement (oracle/) on the host cores: one process per core (the reference's own
    parallelism is one env per subprocess, scripts/train.py:80-85), each stepping its envs serially with the
    same random-action protocol (50-step TimeLimit, reset on done).  Throughput = sum of env-steps / slowest worker."""
    import multiprocessing as mp

    workers = workers or os.cpu_count() or 1
    steps = 25
    envs_per_worker = max(1, budget_env_steps // (workers * steps))
    ctx = mp.get_context("fork")
    with ctx.Pool(workers) as pool:
        res = pool.map(_cpu_worker, [(workload, t, envs_per_worker, steps) for t in range(workers)])
    total = sum(r[0] for r in res)
    dt = max(r[1] for r in res)
    return total / dt, workers, f"{workers} processes x {envs_per_worker} envs x {steps} steps = {total} env-steps in {dt:.1f}s ({workload})"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe): one `nvidia-smi -lms 100`
    process whose lines are collected until stop()."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index, self.rows, self.proc = gpu_index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))
        except Exception:
            pass

    def stop(self, t0=None, t1=None):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=6)
        sm, mx, reasons = [], 0.0, set()
        for t, r in self.rows:
            if t0 is not None and not (t0 <= t <= t1):
                continue
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
            except Exception:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kw, per_gpu, _ = WORKLOADS[args.workload]
    # each "step" of this arm = a bounded sample of the workload; K steps + W warm-up must end within minutes
    per_step_budget = 20000      # >= 20 k env-steps per timed step (1250 per worker on 16 cores): run-to-run spread ~5 %
    vals = []
    for i in range(args.warmup + args.steps):
        v, cores, sample = cpu_port_throughput(args.workload, per_step_budget)
        if i >= args.warmup:
            vals.append(v)
    value = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * per_step_budget / value, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": {"workload": f"{args.workload}: CPU restatement of the reference step (MuJoCo 2.3.2 not installable), "
                                                    f"random actions, auto-reset, bounded sample of {per_step_budget} env-steps per step"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_ours(args):
    import torch
    import torch.distributed as dist

    from mycobotgym_b200 import _lib
    from mycobotgym_b200.vector_env import MyCobotVectorEnv, all_reduce_stats

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # CPU baseline first (rank 0, N=1 only), before CUDA is initialised in this process (workers are forked)
    cpu_val, cores, sample = cpu_port_throughput(args.workload, 20000) if (world == 1 and not args.no_cpu_baseline) else (None, None, None)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    kw, per_gpu, flop_per_step = WORKLOADS[args.workload]
    n = args.envs_per_gpu or per_gpu
    env = MyCobotVectorEnv(num_envs=n, device=f"cuda:{local}", seed=1000 + rank, lockstep_warps=int(os.environ.get("MCB_LOCKSTEP", "0")),
                           mesh_collision=bool(int(os.environ.get("MCB_MESH", "0"))), **kw)
    env.reset()
    K, W = args.steps, args.warmup
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    if args.workload == "grasp":
        g = np.load(os.path.join(ROOT, "tests", "golden", "grasp_pick_sparse.npz"))
        rep = lambda x: torch.as_tensor(np.repeat(np.asarray(x)[None], n, 0), device=dev)
        qvel = rep(g["qvel0"]) + 1e-3 * torch.randn(n, 18, device=dev, dtype=torch.float64, generator=gen)
        env.set_state(qpos=rep(g["qpos0"]), qvel=qvel, ctrl=rep(g["ctrl0"]), qacc_warmstart=rep(g["warm0"]), goal=rep(g["goal"]),
                      elapsed=torch.zeros(n, dtype=torch.int32), qprev=rep(g["qpos0"][:6]))
        acts = torch.zeros(K + W, n, env.action_dim, device=dev)
        acts[:, :, :6] = torch.as_tensor(g["qpos0"][:6], device=dev, dtype=torch.float32) + float(os.environ.get("MCB_GRASP_NOISE", "0.002")) * (torch.rand(K + W, n, 6, device=dev, generator=gen) * 2 - 1)
        acts[:, :, 6] = 0.8
        args.preroll = 0
        env.autotune(acts[0])
    else:
        # steady-state rollout: episode clocks staggered uniformly over the 50-step horizon, so ~2 % of the envs hit the
        # TimeLimit and auto-reset (two extra forward passes + goal / cube resampling) inside every timed step
        stagger = torch.arange(n, device=dev, dtype=torch.int32) % env.max_episode_steps
        env.set_state(elapsed=stagger)
        acts = torch.rand(K + W, n, env.action_dim, device=dev, generator=gen) * 2 - 1
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2
    # pre-roll one full episode horizon (untimed, before the W warm-up steps): with staggered clocks every env has then been
    # reset at a different step, so the timed steps see the steady-state mix of early- and late-episode states (arm near the
    # cube / table late in an episode costs more: contacts, fallback-layout envs) instead of 16 K freshly reset envs
    for t in range(args.preroll):
        env.step(torch.rand(n, env.action_dim, device=dev, generator=gen) * 2 - 1)
    for t in range(W):
        env.step(acts[t])
    env.stats(reset=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.5)                    # let nvidia-smi start streaming before the timed region
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    torch.cuda.synchronize()
    t_wall0 = time.perf_counter()
    for t in range(K):
        flush.zero_()                      # L2 flush between timed iterations (outside the per-step events)
        ev[t][0].record()
        last = env.step(acts[W + t])
        ev[t][1].record()
    stats = env.stats(reset=False).clone()
    fallback_envs = env.last_fallback_envs()   # after the timed loop's last launch (synchronises; outside the event intervals)
    all_reduce_stats(stats)                # the path's only collective: 8 doubles, once per rollout
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)   # before the e2e and HER legs step the env and overwrite its output buffers
    if world > 1:
        dist.barrier()
    allreduce_us = None
    if world > 1:                          # the "64 B, latency-bound" claim as a number: event-timed all-reduce of the statistics vector
        probe = stats.clone()
        for _ in range(3):
            all_reduce_stats(probe)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); dist.barrier()
        a0.record()
        for _ in range(20):
            all_reduce_stats(probe)
        a1.record()
        torch.cuda.synchronize()
        allreduce_us = a0.elapsed_time(a1) / 20 * 1e3
    ms = torch.tensor([sum(a.elapsed_time(b) for a, b in ev)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    clocks = sampler.stop(t_wall0, t_wall0 + t_wall) if sampler else None
    value = world * n * K / (total_ms * 1e-3)

    # e2e: the same step through host buffers (pinned staging inside the C ABI), H2D + D2H inside the timed region
    a_host = acts[W:].cpu().pin_memory().numpy()      # pinned host actions, as the contract asks
    out = env.step_host(a_host[0])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for t in range(K):
        out = env.step_host(a_host[t], out)
    torch.cuda.synchronize()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * n * K / float(e2e_s.item())
    rbytes = 4 if kw["reward_type"] == "sparse" else 8
    h2d, d2h = n * env.action_dim * 4, n * ((env.obs_dim + 6) * 8 + rbytes + 3)

    her = None
    if rank == 0 and world == 1 and kw["reward_type"] in ("sparse", "dense") and not args.no_her and args.workload != "grasp":
        her = her_relabel_leg(env, acts, dev, flush)

    if rank == 0:
        L = _lib.load()
        import ctypes as C

        traffic = {}
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(f"{args.workload}:{n}", {})
        except Exception:
            pass

        peak = C.c_double(0)
        _lib.check(L.mcb_fp64_peak_probe(local, 20000, C.byref(peak)))
        per_gpu_rate = value / world
        achieved = per_gpu_rate * flop_per_step / 1e12
        st = stats.cpu().numpy()
        state_bytes = 2 * 80 * 8 + 28 + (env.obs_dim + 6) * 8 + rbytes + 3
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": f"{args.workload}: {n} envs/GPU x {world} GPU, {kw.get('controller_type', 'joint')} controller, "
                                   f"{100 if kw.get('controller_type') == 'IK' else 20} substeps/step, uniform random actions "
                                   f"U[-1,1]^{env.action_dim} float32, 50-step TimeLimit (episode clocks staggered, {args.preroll}-step untimed pre-roll), auto-reset with on-device goal resampling",
                       "envs_per_gpu": n, "lockstep_warps": env.lockstep_warps,
                       "mesh_collision": env.mesh_collision,     # False: plane / box primitives only (DESIGN.md section 4); MCB_MESH=1 turns the hulls on "l2": "256 MB memset between timed steps (outside the per-step CUDA events)",
                       "timing": "sum of per-step CUDA-event intervals on the launch stream, max over ranks"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": K * env.last_step_launches,
            "clocks": clocks,
            "roofline": {"bound": "fp64", "achieved": achieved, "peak": peak.value, "unit": "TFLOP/s", "frac": achieved / peak.value,
                         # dram__bytes_read.sum + dram__bytes_write.sum of mcb_env_kernel<0>, read from the committed ncu --set full
                         # capture of this build (profiles/traffic.json, written by tools/ncu_summary.py --traffic)
                         "traffic": traffic.get("bytes_per_launch"), "traffic_unit": "B/launch", "traffic_source": traffic.get("source"),
                         "flop_per_env_step": flop_per_step,
                         "note": "dominant kernel = mcb_env_kernel (the whole step); algorithmic FLOP/env-step = instrumented count of the CPU oracle (tools/count_flops.py, BASELINE.md 4); "
                                 "peak = DFMA micro-kernel measured in this run (FP64 peak is not in MEASURED_PEAKS.json)",
                         "hbm_GBps": per_gpu_rate * state_bytes / 1e9},
            "cpu_baseline": None if cpu_val is None else {"value": cpu_val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "episode_stats": {"episodes": st[0], "successes": st[1], "return_sum": st[2], "length_sum": st[3], "env_steps": st[4],
                              "row_overflows": st[5], "fallback_envs_last_step": fallback_envs[0], "last_tier_envs_last_step": fallback_envs[1], "solver_iters_per_substep": (st[6] / st[7]) if st[7] else None},
            "wall_s_timed_region": t_wall,
            "stats_allreduce_us": allreduce_us,
            "her_relabel": her,
        }
        print(json.dumps(line), flush=True)
    env.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="pick", choices=sorted(WORKLOADS))
    ap.add_argument("--envs-per-gpu", type=int, default=0)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--preroll", type=int, default=50, help="untimed steps before the warm-up (steady-state episode mix)")
    ap.add_argument("--no-her", action="store_true", help="skip the separately timed HER relabel leg")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU-port timing leg (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0's envs) as DIR/<name>.npy, 64 MB at most")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
