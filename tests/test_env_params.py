"""Per-env physics parameters, host side: the two ways of baking multipliers into a model agree, and the range parser."""
import ctypes

import numpy as np
import pytest

from mycobotgym_b200 import flatten, mjcf


def _fields(d):
    return {name: np.array(np.ctypeslib.as_array(getattr(d, name)) if not isinstance(getattr(d, name), (int, float)) else getattr(d, name))
            for name, _ in flatten.ModelDesc._fields_}


@pytest.mark.parametrize("path", [mjcf.COMPILED_JOINT, mjcf.COMPILED_MOCAP])
def test_baking_commutes_with_the_reduction(path):
    """reduce_model(apply_params_flat(flat, p)) == apply_params(reduce_model(flat), p), bit for bit: the cube (object0) is one body
    with centre of mass at its origin and identity iquat, so the merge copies its mass and inertia unchanged, and every other baked
    field is copied by the reduction."""
    flat = mjcf.load_compiled(path)
    base = flatten.reduce_model(flat)
    rng = np.random.default_rng(1)
    for _ in range(4):
        p = rng.uniform(0.3, 3.0, flatten.NPARAM)
        a = _fields(flatten.reduce_model(flatten.apply_params_flat(flat, p)))
        b = _fields(flatten.apply_params(base, p))
        for name in a:
            assert np.array_equal(a[name], b[name]), name
        changed = [n for n in a if not np.array_equal(a[n], _fields(base)[n])]
        expect = {"mass", "inertia", "geom_friction", "act_gain", "act_bias", "damping"}
        assert set(changed) == expect, changed


def test_apply_params_scales_only_the_documented_fields():
    flat = mjcf.load_compiled(mjcf.COMPILED_MOCAP)
    base = flatten.reduce_model(flat)
    p = np.arange(1, flatten.NPARAM + 1, dtype=np.float64) * 0.5
    d = flatten.apply_params(base, p)
    assert d.mass[12] == base.mass[12] * p[0] and d.mass[11] == base.mass[11]
    assert [d.geom_friction[g][0] for g in range(5)] == [base.geom_friction[g][0] * p[1 + g] for g in range(5)]
    assert d.geom_friction[4][1] == base.geom_friction[4][1]
    assert d.nu == 1 and d.act_gain[0] == base.act_gain[0] * p[6] and d.act_bias[0][0] == base.act_bias[0][0]
    assert [d.damping[j] for j in range(6)] == [base.damping[j] * p[13] for j in range(6)]
    assert [d.damping[j] for j in range(6, 18)] == [base.damping[j] for j in range(6, 18)]
    nominal = flatten.apply_params(base, np.ones(flatten.NPARAM))
    assert ctypes.string_at(ctypes.byref(nominal), ctypes.sizeof(nominal)) == ctypes.string_at(ctypes.byref(base), ctypes.sizeof(base))
    flat_copy = flatten.apply_params_flat(flat, p)
    assert flat_copy["body_mass"] is not flat["body_mass"] and not np.array_equal(flat_copy["body_mass"], flat["body_mass"])


def test_param_bounds_expand_groups():
    lo, hi = flatten.param_bounds({"cube_mass": (0.5, 2.0), "friction": (0.7, 1.3), "gain": (0.8, 1.2), "arm_damping": (0.5, 2)})
    assert lo.shape == hi.shape == (flatten.NPARAM,)
    assert lo[0] == 0.5 and hi[0] == 2.0 and lo[13] == 0.5 and hi[13] == 2.0
    assert np.all(lo[1:6] == 0.7) and np.all(hi[1:6] == 1.3) and np.all(lo[6:13] == 0.8) and np.all(hi[6:13] == 1.2)
    lo, hi = flatten.param_bounds({"friction_cube": (0.9, 1.1)})
    assert lo[5] == 0.9 and hi[5] == 1.1 and np.all(np.delete(lo, 5) == 1) and np.all(np.delete(hi, 5) == 1)
    lo, hi = flatten.param_bounds({})
    assert np.all(lo == 1) and np.all(hi == 1)
    assert flatten.PARAM_NAMES[flatten.P_GAIN] == "gain_0" and flatten.PARAM_NAMES[flatten.P_ARM_DAMPING] == "arm_damping"


@pytest.mark.parametrize("ranges", [
    {"mass": (0.5, 2.0)},                       # unknown name
    {"cube_mass": (2.0, 0.5)},                  # lo > hi
    {"cube_mass": (0.0, 1.0)},                  # <= 0
    {"gain": (-1.0, 1.0)},
    {"friction": (float("nan"), 1.0)},
    {"friction": (1.0, float("inf"))},
    {"friction": (0.5, 1.0), "friction_cube": (0.9, 1.1)},   # a slot given twice
    {"cube_mass": 1.0},                         # not a pair
])
def test_param_bounds_reject_malformed_input(ranges):
    with pytest.raises(ValueError):
        flatten.param_bounds(ranges)


def test_param_bounds_reject_mesh_collision():
    with pytest.raises(ValueError, match="mesh_collision"):
        flatten.param_bounds({"cube_mass": (0.5, 2.0)}, mesh_collision=True)
