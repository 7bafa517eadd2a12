"""Build + ctypes binding of the C-ABI library (include/mycobot_b200.h).

The product path has no CPU fallback: if the shared library is missing or cannot be loaded the
import of the binding raises, it never routes to oracle/.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

from .flatten import HullDesc, ModelDesc, TaskCfg

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
LIB_PATH = os.environ.get("MCB_LIB") or os.path.join(PKG_DIR, "libmycobot_b200.so")   # MCB_LIB: load another build of the library, e.g. the canary build
CANARY_PATH = os.path.join(PKG_DIR, "libmycobot_b200_canary.so")   # -DMCB_CANARY: guard words in the shared-memory records (tests only)
SRC = os.path.join(PKG_DIR, "csrc", "mcb_engine.cu")
SRC_PRM = os.path.join(PKG_DIR, "csrc", "mcb_engine_prm.cu")   # the step kernels of batches with per-env parameters (own module)
HDR = os.path.join(ROOT, "include", "mycobot_b200.h")
DEPS = (SRC, SRC_PRM, HDR, os.path.join(PKG_DIR, "csrc", "mcb_her.cuh"))

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "--fmad=true",
              "-Xcompiler", "-fPIC", "-shared"]

EXPORTS = [
    "mcb_version", "mcb_last_error", "mcb_model_desc_size", "mcb_task_cfg_size", "mcb_model_create",
    "mcb_model_destroy", "mcb_batch_create", "mcb_batch_destroy", "mcb_batch_num_envs", "mcb_batch_obs_dim", "mcb_batch_action_dim",
    "mcb_reset", "mcb_step", "mcb_step_host", "mcb_get_state", "mcb_set_state", "mcb_forward",
    "mcb_compute_reward", "mcb_stats", "mcb_debug_forward", "mcb_last_step_launches", "mcb_fp64_peak_probe",
    "mcb_autotune", "mcb_batch_lockstep_warps", "mcb_last_fallback_envs", "mcb_her_create", "mcb_her_destroy", "mcb_her_add", "mcb_her_size", "mcb_her_episode_table",
    "mcb_her_sample", "mcb_reset_host", "mcb_seed", "mcb_get_rng_state", "mcb_set_rng_state", "mcb_last_fallback_list", "mcb_total_launches", "mcb_hull_desc_size", "mcb_model_set_hulls",
    "mcb_batch_set_param_ranges", "mcb_get_env_params", "mcb_set_env_params",
    "mcb_batch_set_latency_range", "mcb_get_env_latency", "mcb_set_env_latency",
    "mcb_set_env_applied", "mcb_get_env_applied",
    "mcb_set_contact_output",
]


def needs_build(path=None):
    path = path or LIB_PATH
    if not os.path.exists(path):
        return True
    t = os.path.getmtime(path)
    return any(os.path.exists(p) and os.path.getmtime(p) > t for p in DEPS)


def build(force=False, verbose=False):
    """nvcc cross-compiles for sm_100a without a GPU; the .so is built in-tree so it travels with gpurun."""
    if not force and not needs_build():
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + ["-I", os.path.join(ROOT, "include"), "-o", LIB_PATH, SRC, SRC_PRM]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    subprocess.check_call(cmd)
    return LIB_PATH


def build_canary(force=False):
    """The same source with -DMCB_CANARY (guard words between the arrays of every per-env shared-memory record, checked when the
    env is stored): the bounds-check build tests/test_gpu_canary.py runs, since compute-sanitizer is closed on the GPU pool."""
    if not force and not needs_build(CANARY_PATH):
        return CANARY_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    subprocess.check_call([nvcc] + NVCC_FLAGS + ["-DMCB_CANARY", "-I", os.path.join(ROOT, "include"), "-o", CANARY_PATH, SRC, SRC_PRM])
    return CANARY_PATH


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA extension must be built (python -c 'import __graft_entry__ as g; g.build()'); "
            "there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_double
    L.mcb_version.restype = C.c_char_p
    L.mcb_last_error.restype = C.c_char_p
    L.mcb_model_create.argtypes = [C.POINTER(ModelDesc), i32, C.POINTER(vp)]
    L.mcb_model_destroy.argtypes = [vp]
    L.mcb_model_set_hulls.argtypes = [vp, C.POINTER(HullDesc)]
    L.mcb_batch_create.argtypes = [vp, i32, C.POINTER(TaskCfg), u64, C.POINTER(vp)]
    L.mcb_batch_destroy.argtypes = [vp]
    L.mcb_batch_num_envs.argtypes = [vp]
    L.mcb_batch_obs_dim.argtypes = [vp]
    L.mcb_batch_action_dim.argtypes = [vp]
    L.mcb_reset.argtypes = [vp] + [vp] * 7
    L.mcb_step.argtypes = [vp] + [vp] * 10
    L.mcb_step_host.argtypes = [vp] + [vp] * 10
    L.mcb_get_state.argtypes = [vp] + [vp] * 9
    L.mcb_set_state.argtypes = [vp] + [vp] * 9
    L.mcb_forward.argtypes = [vp] + [vp] * 4
    L.mcb_compute_reward.argtypes = [vp, vp, i64, dbl, i32, vp, vp]
    L.mcb_stats.argtypes = [vp, vp, i32, vp]
    L.mcb_debug_forward.argtypes = [vp, i32, i32, vp, i32, vp]
    L.mcb_last_step_launches.argtypes = [vp]
    L.mcb_fp64_peak_probe.argtypes = [i32, i32, C.POINTER(dbl)]
    L.mcb_autotune.argtypes = [vp, vp, i32, vp]
    L.mcb_batch_lockstep_warps.argtypes = [vp]
    L.mcb_last_fallback_envs.argtypes = [vp, C.POINTER(i32), vp]
    L.mcb_reset_host.argtypes = [vp] + [vp] * 7
    L.mcb_seed.argtypes = [vp, u64, vp, vp]
    L.mcb_get_rng_state.argtypes = [vp] + [vp] * 4
    L.mcb_set_rng_state.argtypes = [vp] + [vp] * 4
    L.mcb_last_fallback_list.argtypes = [vp, vp, i32, vp]
    L.mcb_batch_set_param_ranges.argtypes = [vp, vp, vp]
    L.mcb_get_env_params.argtypes = [vp, vp, vp, vp]
    L.mcb_set_env_params.argtypes = [vp, vp, vp, vp]
    L.mcb_batch_set_latency_range.argtypes = [vp, i32, i32]
    L.mcb_get_env_latency.argtypes = [vp, vp, vp, vp]
    L.mcb_set_env_latency.argtypes = [vp, vp, vp, vp]
    L.mcb_set_env_applied.argtypes = [vp, vp, vp, vp]
    L.mcb_get_env_applied.argtypes = [vp, vp, vp, vp]
    L.mcb_set_contact_output.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.mcb_total_launches.argtypes = [vp]
    L.mcb_total_launches.restype = i64
    L.mcb_her_create.argtypes = [i32, i32, i32, i32, i32, i32, dbl, u64, C.POINTER(vp)]
    L.mcb_her_destroy.argtypes = [vp]
    L.mcb_her_destroy.restype = None
    L.mcb_her_add.argtypes = [vp] + [vp] * 7 + [i32, vp, vp, vp]
    L.mcb_her_size.argtypes = [vp]
    L.mcb_her_size.restype = i64
    L.mcb_her_episode_table.argtypes = [vp, vp, vp, C.POINTER(i64), vp]
    L.mcb_her_sample.argtypes = [vp, i32] + [vp] * 13
    assert L.mcb_model_desc_size() == C.sizeof(ModelDesc), (L.mcb_model_desc_size(), C.sizeof(ModelDesc))
    assert L.mcb_task_cfg_size() == C.sizeof(TaskCfg), (L.mcb_task_cfg_size(), C.sizeof(TaskCfg))
    assert L.mcb_hull_desc_size() == C.sizeof(HullDesc), (L.mcb_hull_desc_size(), C.sizeof(HullDesc))
    _lib = L
    return L


def check(rc):
    if rc < 0:
        raise RuntimeError("mycobot_b200: " + load().mcb_last_error().decode())
    return rc
