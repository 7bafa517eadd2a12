"""bench.py --dump-outputs: what the last timed step returned, as .npy files under a size cap (CPU tensors stand in for the
device buffers `MyCobotVectorEnv.step` returns)."""
import os

import numpy as np
import torch

import bench


def _step_out(n, obs_dim=25):
    g = torch.Generator().manual_seed(n)
    f64 = lambda *s: torch.rand(*s, dtype=torch.float64, generator=g)
    flag = lambda: torch.rand(n, generator=g) > 0.5
    obs = {"observation": f64(n, obs_dim), "achieved_goal": f64(n, 3), "desired_goal": f64(n, 3)}
    info = {"is_success": flag(), "final_observation": f64(n, obs_dim), "_final_observation": flag()}
    return obs, torch.rand(n, generator=g), flag(), flag(), info


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_writes_every_returned_array(tmp_path):
    obs, rew, term, trunc, info = out = _step_out(1000)
    bench.dump_outputs(str(tmp_path), out)
    got = _load(tmp_path)
    assert sorted(got) == sorted([*obs, "reward", "terminated", "truncated", *info])
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    np.testing.assert_array_equal(got["observation"], obs["observation"].numpy())
    np.testing.assert_array_equal(got["reward"], rew.numpy())
    np.testing.assert_array_equal(got["truncated"], trunc.numpy().astype(np.float32))


def test_dump_of_a_large_batch_is_a_seeded_sample_under_the_cap(tmp_path, monkeypatch):
    assert bench.DUMP_BYTES + 11 * 4096 < 64 * 10**6     # the real cap leaves room for the .npy headers of the 11 files
    monkeypatch.setattr(bench, "DUMP_BYTES", 20_000)    # 500 envs write ~230 kB of outputs
    n = 500
    obs, rew, term, trunc, info = out = _step_out(n)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), out)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sum(v.nbytes for v in a.values()) <= 20_000
    assert all(np.array_equal(a[k], b[k]) for k in a)
    idx = a["env_index"].astype(np.int64)
    assert 0 < len(idx) < n and np.all(np.diff(idx) > 0)
    np.testing.assert_array_equal(a["final_observation"], info["final_observation"].numpy()[idx])
    np.testing.assert_array_equal(a["terminated"], term.numpy()[idx].astype(np.float32))
