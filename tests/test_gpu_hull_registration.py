"""mcb_model_set_hulls checks a whole descriptor before it changes the model: a rejected descriptor leaves the model's hull tables
and pair parameters exactly as they were."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu


def _fresh_model_with_hulls(dev):
    from mycobotgym_b200 import _lib, flatten, mjcf

    L = _lib.load()
    flat = mjcf.load_compiled(mjcf.COMPILED_JOINT)
    desc = flatten.reduce_model(flat)
    h = C.c_void_p()
    _lib.check(L.mcb_model_create(C.byref(desc), dev, C.byref(h)))
    hd, verts = flatten.reduce_hulls(flat)
    _lib.check(L.mcb_model_set_hulls(h, C.byref(hd)))
    return h, desc, flat, hd, verts


def _push_rollout(monkeypatch, dev, model, desc, flat, mesh_collision=True):
    from mycobotgym_b200 import vector_env

    monkeypatch.setitem(vector_env._MODEL_CACHE, (dev, "joint"), (model, desc, flat))
    n = 512
    env = vector_env.MyCobotVectorEnv(num_envs=n, has_object=True, block_gripper=True, target_in_the_air=False, reward_type="sparse",
                                      mesh_collision=mesh_collision, autotune=False, lockstep_warps=16, seed=5)
    env.reset()
    gen = torch.Generator(device="cuda")
    gen.manual_seed(7)
    outs = []
    for _ in range(16):
        obs, rew, term, trunc, _ = env.step(torch.rand(n, 7, device="cuda", generator=gen) * 2 - 1)
        outs += [obs["observation"].clone(), rew.clone(), term.clone(), trunc.clone()]
    outs += list(env.get_state().values())
    env.close()
    return outs


def test_rejected_hull_descriptor_leaves_the_model_unchanged(monkeypatch):
    from mycobotgym_b200 import _lib
    from mycobotgym_b200.flatten import HullDesc

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    L = _lib.load()
    dev = torch.cuda.current_device()
    clean, desc, flat, _, _ = _fresh_model_with_hulls(dev)
    model, _, _, hd, verts = _fresh_model_with_hulls(dev)      # `bad` below points at `verts`
    try:
        # different hull tables and pair parameters, and a last pair whose second object is a primitive, not a hull
        bad = HullDesc.from_buffer_copy(hd)
        for h in range(bad.nhull):
            bad.rbound[h] *= 2
            bad.center[h][2] += 0.01
            bad.friction[h][0] *= 3
        assert bad.npair > 1
        bad.pair_b[bad.npair - 1] = 0
        assert L.mcb_model_set_hulls(model, C.byref(bad)) < 0
        assert "bad pair" in L.mcb_last_error().decode()

        got = _push_rollout(monkeypatch, dev, model, desc, flat)
        want = _push_rollout(monkeypatch, dev, clean, desc, flat)
        assert len(got) == len(want)
        for k, (a, b) in enumerate(zip(got, want)):
            assert torch.equal(a, b), k
        # the rollout does meet hull contacts: without them it ends elsewhere
        no_mesh = _push_rollout(monkeypatch, dev, clean, desc, flat, mesh_collision=False)
        assert not all(torch.equal(a, b) for a, b in zip(no_mesh, want))
    finally:
        L.mcb_model_destroy(model)
        L.mcb_model_destroy(clean)
