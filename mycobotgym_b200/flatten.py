"""FlatModel (mjModel-like table) -> `mcb_model_desc` (include/mycobot_b200.h).

Second half of north-star subsystem (1): the compiled model is reduced to its 13 jointed
bodies -- bodies without joints (flange, camera frames, gripper_base, gripper_tcp, finger
layers; mycobot280_main.xml:157-175,194-200,221-226) are merged into their jointed ancestor
(composite mass / centre of mass / inertia, composed fixed transforms) -- and laid out as the
fixed-size structure-of-arrays the CUDA kernels read.  The merge is exact rigid-body algebra;
the oracle works on the unmerged 25-body table, so GPU-vs-oracle parity also checks the merge.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import mjcf
from .mjcf import quat2mat, quat_mul

NB, NV, NQ, NU, NHINGE, NGEOM, MAXPAIR = 13, 18, 19, 7, 12, 5, 12
MAXHULL, MAXHPAIR = 16, 192
CUBE_BODY = 12
# the jointed bodies of the reduced model in mcb_model_desc order (the rows of xfrc_applied): fixed bodies are merged into these
BODY_NAMES = ("link1", "link2", "link3", "link4", "link5", "link6", "right_gear_link", "right_finger_link", "left_gear_link",
              "left_finger_link", "right_hinge_link", "left_hinge_link", "object0")
# the primitive geoms in mcb_model_desc order: the geom ids of the contact output (MyCobotVectorEnv.contacts)
GEOM_NAMES = ("floor", "table", "right_finger_layer", "left_finger_layer", "object0")
MAXCON, CONTACT_DOUBLES = 24, 19     # MCB_MAXCON contact slots per env, MCB_CONTACT_DOUBLES per slot: dist, pos3, frame9, force6

_d = C.c_double
_i = C.c_int32


class ModelDesc(C.Structure):
    _fields_ = [
        ("parent", _i * NB), ("level", _i * NB), ("subtree_size", _i * NB), ("dof_body", _i * NV),
        ("ancmask", C.c_uint32 * NB),
        ("Tpos", _d * 3 * NB), ("Tmat", _d * 9 * NB), ("axis", _d * 3 * NB),
        ("mass", _d * NB), ("ipos", _d * 3 * NB), ("inertia", _d * 6 * NB),
        ("armature", _d * NV), ("damping", _d * NV), ("dof_invweight0", _d * NV),
        ("ref_robot", _d * 3), ("qpos0", _d * NQ),
        ("jnt_limited", _i * NHINGE), ("jnt_range", _d * 2 * NHINGE), ("jnt_solref", _d * 2 * NHINGE),
        ("jnt_solimp", _d * 5 * NHINGE),
        ("con_body1", _i * 2), ("con_body2", _i * 2), ("con_anchor1", _d * 3 * 2), ("con_anchor2", _d * 3 * 2),
        ("con_diag", _d * 2), ("con_solref", _d * 2 * 2), ("con_solimp", _d * 5 * 2),
        ("jeq_dof1", _i), ("jeq_dof2", _i), ("jeq_polycoef", _d * 5), ("jeq_diag", _d), ("jeq_solref", _d * 2),
        ("jeq_solimp", _d * 5),
        ("geom_type", _i * NGEOM), ("geom_body", _i * NGEOM), ("geom_condim", _i * NGEOM),
        ("geom_pos", _d * 3 * NGEOM), ("geom_mat", _d * 9 * NGEOM), ("geom_size", _d * 3 * NGEOM),
        ("geom_rbound", _d * NGEOM), ("geom_friction", _d * 3 * NGEOM), ("geom_solref", _d * 2 * NGEOM),
        ("geom_solimp", _d * 5 * NGEOM), ("geom_solmix", _d * NGEOM), ("geom_invweight", _d * 2 * NGEOM),
        ("npair", _i), ("pair_g1", _i * MAXPAIR), ("pair_g2", _i * MAXPAIR),
        ("eef_body", _i), ("eef_pos", _d * 3), ("obj_body", _i),
        ("geom_finger_r", _i), ("geom_finger_l", _i), ("geom_object", _i), ("target0_pos", _d * 3),
        ("act_moment", _d * NV * NU), ("act_gain", _d * NU), ("act_bias", _d * 3 * NU),
        ("act_ctrlrange", _d * 2 * NU), ("act_forcerange", _d * 2 * NU), ("act_ctrllimited", _i * NU),
        ("act_forcelimited", _i * NU),
        ("timestep", _d), ("gravity", _d * 3), ("tolerance", _d), ("ls_tolerance", _d), ("meaninertia", _d),
        ("impratio", _d), ("iterations", _i), ("ls_iterations", _i),
        ("initial_gripper_xpos", _d * 3), ("height_offset", _d), ("init_qpos", _d * NQ), ("init_ctrl", _d * NU),
        ("key_initial_gripper_xpos", _d * 3), ("key_height_offset", _d), ("key_qpos", _d * NQ), ("key_ctrl", _d * NU),
        ("nu", _i), ("has_weld", _i), ("weld_body2", _i), ("reserved0_", _i),
        ("Tquat", _d * 4 * NB), ("weld_anchor1", _d * 3), ("weld_anchor2", _d * 3), ("weld_relquat", _d * 4),
        ("weld_torquescale", _d), ("weld_diag", _d * 2), ("weld_solref", _d * 2), ("weld_solimp", _d * 5),
        ("mocap_pos0", _d * 3), ("mocap_quat0", _d * 4), ("key_mocap_pos", _d * 3), ("key_mocap_quat", _d * 4),
    ]


class TaskCfg(C.Structure):
    _fields_ = [
        ("has_object", _i), ("block_gripper", _i), ("target_in_the_air", _i), ("reward_type", _i),
        ("max_episode_steps", _i), ("frame_skip", _i), ("auto_reset", _i), ("nefc_max", _i),
        ("controller_type", _i), ("fetch_env", _i), ("control_steps", _i), ("mesh_collision", _i), ("reserved1_", _i),
        ("lockstep_warps", _i),
        ("distance_threshold", _d),
    ]


class HullDesc(C.Structure):
    """mcb_hull_desc (include/mycobot_b200.h): convex hulls of the mesh geoms in the frames of the REDUCED model's bodies."""
    _fields_ = [
        ("nhull", _i), ("npair", _i), ("nvert", _i), ("reserved_", _i),
        ("body", _i * MAXHULL), ("vadr", _i * MAXHULL), ("vnum", _i * MAXHULL), ("mult", _i * MAXHULL), ("condim", _i * MAXHULL),
        ("center", _d * 3 * MAXHULL), ("rbound", _d * MAXHULL), ("friction", _d * 3 * MAXHULL), ("solref", _d * 2 * MAXHULL),
        ("solimp", _d * 5 * MAXHULL), ("solmix", _d * MAXHULL), ("invweight", _d * 2 * MAXHULL),
        ("pair_a", C.c_uint8 * MAXHPAIR), ("pair_b", C.c_uint8 * MAXHPAIR),
        ("vert", C.POINTER(_d)),
    ]


def _set(arr, value):
    a = np.ascontiguousarray(value)
    flat = np.ctypeslib.as_array(arr).reshape(-1)
    flat[:] = a.reshape(-1)


def _rel_pose(m, body, anc):
    """Pose of `body`'s frame in the frame of ancestor body `anc` (anc == 0: world), at q = 0 of the
    joints strictly between them (there are none by construction: only fixed bodies are crossed)."""
    pos = np.zeros(3)
    quat = np.array([1.0, 0, 0, 0])
    b = body
    while b != anc:
        pos = m["body_pos"][b] + quat2mat(m["body_quat"][b]) @ pos
        quat = quat_mul(m["body_quat"][b], quat)
        b = int(m["body_parentid"][b])
    return pos, quat


def reduce_model(m) -> ModelDesc:
    nbody = int(m["nbody"])
    assert int(m["nv"]) == NV and int(m["nq"]) == NQ and int(m["nu"]) in (1, NU) and int(m["njnt"]) == NB
    jointed = [b for b in range(nbody) if m["body_jntnum"][b] > 0]
    assert len(jointed) == NB
    jidx = {b: k for k, b in enumerate(jointed)}
    assert np.all(m["jnt_pos"] == 0), "reduced FK assumes joint anchors at the body origin"
    d = ModelDesc()

    def weld_jointed(b):
        w = int(m["body_weldid"][b])
        return jidx[w] if w != 0 else -1

    parent, level = [], []
    for k, b in enumerate(jointed):
        p = int(m["body_parentid"][b])
        pw = int(m["body_weldid"][p])
        pk = jidx[pw] if pw != 0 else -1
        parent.append(pk)
        level.append(0 if pk < 0 else level[pk] + 1)
        anc = pw if pw != 0 else 0
        pos, quat = _rel_pose(m, b, anc)
        if m["jnt_type"][m["body_jntadr"][b]] == mjcf.JNT_FREE:
            pos, quat = np.zeros(3), np.array([1.0, 0, 0, 0])
        _set(d.Tpos[k], pos)
        _set(d.Tmat[k], quat2mat(quat))
        _set(d.Tquat[k], quat)
        _set(d.axis[k], m["jnt_axis"][m["body_jntadr"][b]])
    _set(d.parent, parent)
    _set(d.level, level)
    sub = [1] * NB
    for k in range(NB - 1, -1, -1):
        if parent[k] >= 0:
            sub[parent[k]] += sub[k]
    for k in range(NB):  # DFS pre-order => subtree is the contiguous range [k, k+sub[k])
        for c in range(k + 1, k + sub[k]):
            a = c
            while a != k and a >= 0:
                a = parent[a]
            assert a == k
    _set(d.subtree_size, sub)
    _set(d.dof_body, [jidx[int(b)] for b in m["dof_bodyid"]])
    for k, b in enumerate(jointed):
        mask = 0
        dof = int(m["body_dofadr"][b] + m["body_dofnum"][b] - 1)
        while dof >= 0:
            mask |= 1 << dof
            dof = int(m["dof_parentid"][dof])
        d.ancmask[k] = mask

    # composite inertia of each jointed body with its merged fixed descendants
    for k, b in enumerate(jointed):
        parts = []
        for f in range(nbody):
            if int(m["body_weldid"][f]) != b or m["body_mass"][f] <= 0:
                continue
            pos, quat = _rel_pose(m, f, b)
            R = quat2mat(quat)
            Ri = R @ quat2mat(m["body_iquat"][f])
            parts.append((float(m["body_mass"][f]), pos + R @ m["body_ipos"][f], Ri @ np.diag(m["body_inertia"][f]) @ Ri.T))
        mt = sum(p[0] for p in parts)
        com = sum(p[0] * p[1] for p in parts) / mt
        I = np.zeros((3, 3))
        for ms, p, Ig in parts:
            dd = p - com
            I += Ig + ms * (dd @ dd * np.eye(3) - np.outer(dd, dd))
        d.mass[k] = mt
        _set(d.ipos[k], com)
        _set(d.inertia[k], [I[0, 0], I[1, 1], I[2, 2], I[0, 1], I[0, 2], I[1, 2]])
    _set(d.armature, m["dof_armature"])
    _set(d.damping, m["dof_damping"])
    _set(d.dof_invweight0, m["dof_invweight0"])
    _set(d.qpos0, m["qpos0"])

    fk = mjcf.fk_numpy(m, m["qpos0"])
    xpos, xquat, xmat, xipos = fk[0], fk[1], fk[2], fk[3]
    root = int(m["body_rootid"][jointed[0]])
    sel = [b for b in range(nbody) if m["body_rootid"][b] == root and m["body_mass"][b] > 0]
    mtot = sum(m["body_mass"][b] for b in sel)
    _set(d.ref_robot, sum(m["body_mass"][b] * xipos[b] for b in sel) / mtot)

    nh = 0
    for j in range(NB):
        if m["jnt_type"][j] != mjcf.JNT_HINGE:
            continue
        assert m["jnt_dofadr"][j] == nh and m["jnt_margin"][j] == 0
        d.jnt_limited[nh] = int(m["jnt_limited"][j])
        _set(d.jnt_range[nh], m["jnt_range"][j])
        _set(d.jnt_solref[nh], m["jnt_solref"][j])
        _set(d.jnt_solimp[nh], m["jnt_solimp"][j])
        nh += 1
    assert nh == NHINGE

    ci = 0
    d.has_weld = 0
    _set(d.mocap_quat0, [1, 0, 0, 0]); _set(d.key_mocap_quat, [1, 0, 0, 0]); _set(d.weld_relquat, [1, 0, 0, 0])
    for e in range(int(m["neq"])):
        if m["eq_type"][e] == mjcf.EQ_WELD:
            # the mocap variant's weld (mocap.xml:16-20): body1 = mocap body (static), body2 = gripper_tcp; it must be the first equality
            b1, b2 = int(m["eq_obj1id"][e]), int(m["eq_obj2id"][e])
            assert e == 0 and m["body_mocapid"][b1] == 0 and d.has_weld == 0
            w2 = int(m["body_weldid"][b2])
            p2, q2 = _rel_pose(m, b2, w2)
            assert abs(abs(q2[0]) - 1) < 1e-12, "gripper_tcp must share its jointed body's orientation"
            d.has_weld, d.weld_body2 = 1, jidx[w2]
            _set(d.weld_anchor1, m["eq_data"][e, 3:6])
            _set(d.weld_anchor2, p2 + quat2mat(q2) @ m["eq_data"][e, 0:3])
            _set(d.weld_relquat, m["eq_data"][e, 6:10])
            d.weld_torquescale = float(m["eq_data"][e, 10])
            _set(d.weld_diag, m["body_invweight0"][b1] + m["body_invweight0"][b2])
            _set(d.weld_solref, m["eq_solref"][e])
            _set(d.weld_solimp, m["eq_solimp"][e])
            _set(d.mocap_pos0, m["body_pos"][b1]); _set(d.mocap_quat0, m["body_quat"][b1])
            _set(d.key_mocap_pos, m["key_mpos"][0][:3]); _set(d.key_mocap_quat, m["key_mquat"][0][:4])
        elif m["eq_type"][e] == mjcf.EQ_CONNECT:
            b1, b2 = int(m["eq_obj1id"][e]), int(m["eq_obj2id"][e])
            assert b1 in jidx and b2 in jidx
            d.con_body1[ci], d.con_body2[ci] = jidx[b1], jidx[b2]
            _set(d.con_anchor1[ci], m["eq_data"][e, 0:3])
            _set(d.con_anchor2[ci], m["eq_data"][e, 3:6])
            d.con_diag[ci] = m["body_invweight0"][b1, 0] + m["body_invweight0"][b2, 0]
            _set(d.con_solref[ci], m["eq_solref"][e])
            _set(d.con_solimp[ci], m["eq_solimp"][e])
            ci += 1
        else:
            d1, d2 = int(m["jnt_dofadr"][m["eq_obj1id"][e]]), int(m["jnt_dofadr"][m["eq_obj2id"][e]])
            d.jeq_dof1, d.jeq_dof2 = d1, d2
            _set(d.jeq_polycoef, m["eq_data"][e, 0:5])
            d.jeq_diag = m["dof_invweight0"][d1] + m["dof_invweight0"][d2]
            _set(d.jeq_solref, m["eq_solref"][e])
            _set(d.jeq_solimp, m["eq_solimp"][e])
    assert ci == 2 and [t for t in m["eq_type"] if t != mjcf.EQ_WELD] == [mjcf.EQ_CONNECT, mjcf.EQ_CONNECT, mjcf.EQ_JOINT]

    assert int(m["ngeom"]) == NGEOM
    for g in range(NGEOM):
        gb = int(m["geom_bodyid"][g])
        w = int(m["body_weldid"][gb])
        pos, quat = _rel_pose(m, gb, w if w != 0 else 0)
        R = quat2mat(quat)
        d.geom_type[g] = int(m["geom_type"][g])
        d.geom_body[g] = weld_jointed(gb)
        d.geom_condim[g] = int(m["geom_condim"][g])
        _set(d.geom_pos[g], pos + R @ m["geom_pos"][g])
        _set(d.geom_mat[g], R @ quat2mat(m["geom_quat"][g]))
        _set(d.geom_size[g], m["geom_size"][g])
        d.geom_rbound[g] = m["geom_rbound"][g]
        _set(d.geom_friction[g], m["geom_friction"][g])
        _set(d.geom_solref[g], m["geom_solref"][g])
        _set(d.geom_solimp[g], m["geom_solimp"][g])
        d.geom_solmix[g] = m["geom_solmix"][g]
        _set(d.geom_invweight[g], m["body_invweight0"][gb])
        assert m["geom_margin"][g] == 0 and m["geom_gap"][g] == 0
    pairs = []
    excl = {tuple(e) for e in m["exclude"].tolist()}
    for g1 in range(NGEOM):
        for g2 in range(g1 + 1, NGEOM):
            a, b = (g1, g2) if m["geom_type"][g1] <= m["geom_type"][g2] else (g2, g1)
            b1, b2 = int(m["geom_bodyid"][a]), int(m["geom_bodyid"][b])
            w1, w2 = int(m["body_weldid"][b1]), int(m["body_weldid"][b2])
            if w1 == w2 or (min(b1, b2), max(b1, b2)) in excl:
                continue
            if w1 and w2 and (m["body_weldid"][m["body_parentid"][w1]] == w2 or m["body_weldid"][m["body_parentid"][w2]] == w1):
                continue
            if not ((m["geom_contype"][a] & m["geom_conaffinity"][b]) or (m["geom_contype"][b] & m["geom_conaffinity"][a])):
                continue
            pairs.append((a, b))
    assert len(pairs) <= MAXPAIR
    d.npair = len(pairs)
    for i, (a, b) in enumerate(pairs):
        d.pair_g1[i], d.pair_g2[i] = a, b

    s_eef = m["site_names"].index("EEF")
    s_obj = m["site_names"].index("object0")
    sb = int(m["site_bodyid"][s_eef])
    w = int(m["body_weldid"][sb])
    pos, quat = _rel_pose(m, sb, w)
    d.eef_body = jidx[w]
    assert abs(abs(quat[0]) - 1) < 1e-12 and np.all(m["site_quat"][s_eef] == [1, 0, 0, 0]), "EEF site must share its body's orientation"
    _set(d.eef_pos, pos + quat2mat(quat) @ m["site_pos"][s_eef])
    ob = int(m["site_bodyid"][s_obj])
    assert ob in jidx and np.all(m["site_pos"][s_obj] == 0)
    d.obj_body = jidx[ob]
    gn = m["geom_names"]
    d.geom_finger_r, d.geom_finger_l, d.geom_object = gn.index("right_finger_layer"), gn.index("left_finger_layer"), gn.index("object0")
    s_t = m["site_names"].index("target0")
    assert m["site_bodyid"][s_t] == 0
    _set(d.target0_pos, m["site_pos"][s_t])

    nu = int(m["nu"])
    d.nu = nu

    def padu(a, width=None):
        a = np.asarray(a, dtype=np.float64)
        out = np.zeros((NU,) + a.shape[1:])
        out[:nu] = a
        return out

    _set(d.act_moment, padu(m["actuator_moment"]))
    _set(d.act_gain, padu(m["actuator_gain"]))
    _set(d.act_bias, padu(m["actuator_biasprm"]))
    _set(d.act_ctrlrange, padu(m["actuator_ctrlrange"]))
    _set(d.act_forcerange, padu(m["actuator_forcerange"]))
    _set(d.act_ctrllimited, padu(m["actuator_ctrllimited"]).astype(np.int32))
    _set(d.act_forcelimited, padu(m["actuator_forcelimited"]).astype(np.int32))
    d.timestep, d.tolerance, d.ls_tolerance = float(m["timestep"]), float(m["tolerance"]), float(m["ls_tolerance"])
    _set(d.gravity, m["gravity"])
    d.meaninertia, d.impratio = float(m["stat_meaninertia"]), float(m["impratio"])
    d.iterations, d.ls_iterations = int(m["iterations"]), int(m["ls_iterations"])

    # _env_setup constants (mycobot.py:450-481), non-fetch: sites at qpos0
    seb = int(m["site_bodyid"][s_eef])
    _set(d.initial_gripper_xpos, xpos[seb] + xmat[seb] @ m["site_pos"][s_eef])
    d.height_offset = float((xpos[ob] + xmat[ob] @ m["site_pos"][s_obj])[2])
    _set(d.init_qpos, m["qpos0"])
    _set(d.init_ctrl, np.zeros(NU))
    if d.has_weld:
        pass  # fetch keyframe forward uses the keyframe's mocap pose; FK of the robot does not depend on it
    # fetch envs: mj_resetDataKeyframe(0) then forward (mycobot.py:451-472)
    kq = m["key_qpos"][0].copy()
    kq[15:19] /= np.linalg.norm(kq[15:19])
    fkk = mjcf.fk_numpy(m, kq)
    _set(d.key_initial_gripper_xpos, fkk[0][seb] + fkk[2][seb] @ m["site_pos"][s_eef])
    d.key_height_offset = float((fkk[0][ob] + fkk[2][ob] @ m["site_pos"][s_obj])[2])
    _set(d.key_qpos, m["key_qpos"][0])
    _set(d.key_ctrl, padu(m["key_ctrl"][0]))
    return d


# Per-env physics parameters (include/mycobot_b200.h, MCB_NPARAM): multipliers of model fields, nominal value 1.0.
PARAM_NAMES = ("cube_mass", "friction_floor", "friction_table", "friction_finger_r", "friction_finger_l", "friction_cube",
               "gain_0", "gain_1", "gain_2", "gain_3", "gain_4", "gain_5", "gain_6", "arm_damping")
NPARAM = len(PARAM_NAMES)
P_CUBE_MASS, P_FRICTION, P_GAIN, P_ARM_DAMPING = 0, 1, 6, 13
PARAM_GROUPS = {"friction": PARAM_NAMES[P_FRICTION:P_GAIN], "gain": PARAM_NAMES[P_GAIN:P_ARM_DAMPING]}


def param_bounds(param_ranges, mesh_collision=False):
    """`param_ranges` ({name: (lo, hi)}) -> (lo, hi), two float64 arrays of NPARAM.  Names are PARAM_NAMES or the groups
    'friction' / 'gain', which give the same range to each of their slots (each slot is still drawn on its own); unlisted slots
    get (1, 1).  Raises ValueError for unknown names, a slot named twice, bounds that are not finite or <= 0, lo > hi, and for
    mesh_collision=True (hull pairs keep the model's friction)."""
    if mesh_collision:
        raise ValueError("per-env parameters are not supported with mesh_collision=True")
    lo, hi = np.ones(NPARAM), np.ones(NPARAM)
    seen = set()
    for key, rng in dict(param_ranges).items():
        slots = PARAM_GROUPS.get(key, (key,))
        for name in slots:
            if name not in PARAM_NAMES:
                raise ValueError(f"unknown parameter {key!r}; known: {', '.join(PARAM_NAMES + tuple(PARAM_GROUPS))}")
            if name in seen:
                raise ValueError(f"parameter {name!r} is given twice")
            seen.add(name)
        try:
            a, b = (float(v) for v in rng)
        except (TypeError, ValueError):
            raise ValueError(f"{key!r}: a range is a pair (lo, hi), got {rng!r}") from None
        if not (np.isfinite(a) and np.isfinite(b) and a > 0 and b > 0):
            raise ValueError(f"{key!r}: bounds must be finite and > 0, got ({a}, {b})")
        if a > b:
            raise ValueError(f"{key!r}: lo > hi ({a} > {b})")
        for name in slots:
            k = PARAM_NAMES.index(name)
            lo[k], hi[k] = a, b
    return lo, hi


def latency_bounds(spec, frame_skip, mesh_collision=False):
    """Actuation latency in substeps, `None | d | (lo, hi)` -> None or (lo, hi), two ints with 0 <= lo <= hi <= frame_skip (an int d
    gives (d, d)).  Raises ValueError for non-integers (bool and float included), negative bounds, lo > hi, hi > frame_skip, and for
    mesh_collision=True (latency runs in the kernels of batches with per-env parameters, which hull collisions do not support)."""
    if spec is None:
        return None
    if mesh_collision:
        raise ValueError("actuation latency is not supported with mesh_collision=True")

    def as_int(v):
        if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, np.integer)):
            raise ValueError(f"actuation latency bounds are integers (substeps), got {v!r}")
        return int(v)

    if isinstance(spec, (tuple, list)):
        if len(spec) != 2:
            raise ValueError(f"actuation latency is an int or a pair (lo, hi), got {spec!r}")
        lo, hi = as_int(spec[0]), as_int(spec[1])
    else:
        lo = hi = as_int(spec)
    if lo < 0:
        raise ValueError(f"actuation latency must be >= 0, got ({lo}, {hi})")
    if lo > hi:
        raise ValueError(f"actuation latency: lo > hi ({lo} > {hi})")
    if hi > frame_skip:
        raise ValueError(f"actuation latency must be <= frame_skip ({frame_skip}), got ({lo}, {hi})")
    return lo, hi


def applied_forces(qfrc_applied, xfrc_applied, num_envs, mesh_collision=False):
    """Checks the arguments of `MyCobotVectorEnv.set_applied_forces` and returns them as contiguous float64 torch tensors (None
    stays None; input on the CPU stays there): qfrc_applied (N, NV) generalized forces, xfrc_applied (N, NB, 6) world-frame force
    and torque per body of BODY_NAMES.  Raises ValueError for another shape, a non-finite value, and for mesh_collision=True."""
    import torch

    if mesh_collision:
        raise ValueError("applied forces are not supported with mesh_collision=True")
    out = []
    for name, x, shape in (("qfrc_applied", qfrc_applied, (num_envs, NV)), ("xfrc_applied", xfrc_applied, (num_envs, NB, 6))):
        if x is None:
            out.append(None)
            continue
        t = x if torch.is_tensor(x) else torch.as_tensor(np.asarray(x))
        if t.dtype.is_complex or t.dtype == torch.bool:
            raise ValueError(f"{name} must be real, got {t.dtype}")
        if tuple(t.shape) != shape:
            raise ValueError(f"{name} must have shape {shape}, got {tuple(t.shape)}")
        t = t.to(dtype=torch.float64).contiguous()
        if not bool(torch.isfinite(t).all()):
            raise ValueError(f"{name} must be finite")
        out.append(t)
    return tuple(out)


def _check_params(p):
    p = np.asarray(p, dtype=np.float64)
    if p.shape != (NPARAM,):
        raise ValueError(f"expected {NPARAM} multipliers, got shape {p.shape}")
    return p


def apply_params(desc, p):
    """A copy of the reduced model `desc` with the NPARAM multipliers `p` baked into its fields -- the model a batch without per-env
    parameters would need to simulate what an env with parameters `p` simulates (the compiled constants stay, as on the device)."""
    p = _check_params(p)
    d = ModelDesc()
    C.memmove(C.byref(d), C.byref(desc), C.sizeof(ModelDesc))
    c = CUBE_BODY
    d.mass[c] = d.mass[c] * p[P_CUBE_MASS]
    for k in range(6):
        d.inertia[c][k] = d.inertia[c][k] * p[P_CUBE_MASS]
    for g in range(NGEOM):
        d.geom_friction[g][0] = d.geom_friction[g][0] * p[P_FRICTION + g]
    for u in range(int(d.nu)):
        d.act_gain[u] = d.act_gain[u] * p[P_GAIN + u]
        d.act_bias[u][1] = d.act_bias[u][1] * p[P_GAIN + u]
        d.act_bias[u][2] = d.act_bias[u][2] * p[P_GAIN + u]
    for j in range(6):
        d.damping[j] = d.damping[j] * p[P_ARM_DAMPING]
    return d


def apply_params_flat(m, p):
    """The same on the unmerged flat table (the oracle's model): body_mass / body_inertia of object0, geom_friction,
    actuator_gain, actuator_biasprm and dof_damping.  Returns a copy; `m` is left as it was."""
    p = _check_params(p)
    out = type(m)(m)
    obj = int(m["site_bodyid"][m["site_names"].index("object0")])
    for key in ("body_mass", "body_inertia", "geom_friction", "actuator_gain", "actuator_biasprm", "dof_damping"):
        out[key] = np.array(m[key], dtype=np.float64, copy=True)
    out["body_mass"][obj] = out["body_mass"][obj] * p[P_CUBE_MASS]
    out["body_inertia"][obj] = out["body_inertia"][obj] * p[P_CUBE_MASS]
    out["geom_friction"][:, 0] = out["geom_friction"][:, 0] * p[P_FRICTION:P_FRICTION + NGEOM]
    nu = int(m["nu"])
    gains = p[P_GAIN:P_GAIN + nu]
    out["actuator_gain"] = out["actuator_gain"] * gains
    out["actuator_biasprm"][:, 1] = out["actuator_biasprm"][:, 1] * gains
    out["actuator_biasprm"][:, 2] = out["actuator_biasprm"][:, 2] * gains
    out["dof_damping"][:6] = out["dof_damping"][:6] * p[P_ARM_DAMPING]
    return out


def reduce_hulls(m):
    """Convex hulls of the mesh geoms -> `mcb_hull_desc`: vertices / interior points moved into the frame of the jointed body the
    mesh's body is welded to (flange and gripper_base ride on link6), candidate pairs after MuJoCo's static filters (same weld
    body, parent-child unless one side is welded to the world, <contact><exclude>; all contype / conaffinity are 1).  Returns
    (desc, vertex array) -- the array must stay alive until mcb_model_set_hulls has copied it."""
    nh = int(m.get("nhull", 0))
    d = HullDesc()
    assert nh <= MAXHULL
    jointed = [b for b in range(int(m["nbody"])) if m["body_jntnum"][b] > 0]
    jidx = {b: k for k, b in enumerate(jointed)}
    verts = np.zeros((int(m["hull_vertnum"].sum()) if nh else 0, 3))
    d.nhull, d.nvert = nh, len(verts)
    for h in range(nh):
        hb = int(m["hull_bodyid"][h])
        w = int(m["body_weldid"][hb])
        pos, quat = _rel_pose(m, hb, w if w != 0 else 0)
        R = quat2mat(quat)
        a, n = int(m["hull_vertadr"][h]), int(m["hull_vertnum"][h])
        verts[a:a + n] = m["hull_vert"][a:a + n] @ R.T + pos
        d.body[h] = jidx[w] if w != 0 else -1
        d.vadr[h], d.vnum[h], d.mult[h], d.condim[h] = a, n, int(m["hull_mult"][h]), int(m["hull_condim"][h])
        _set(d.center[h], R @ m["hull_center"][h] + pos)
        d.rbound[h] = float(m["hull_rbound"][h])
        _set(d.friction[h], m["hull_friction"][h]); _set(d.solref[h], m["hull_solref"][h]); _set(d.solimp[h], m["hull_solimp"][h])
        d.solmix[h] = float(m["hull_solmix"][h])
        _set(d.invweight[h], m["body_invweight0"][hb])
    excl = {tuple(e) for e in m["exclude"].tolist()}
    par, weld = m["body_parentid"], m["body_weldid"]

    def filtered(b1, b2):
        w1, w2 = int(weld[b1]), int(weld[b2])
        if w1 == w2 or (min(b1, b2), max(b1, b2)) in excl:
            return True
        return bool(w1 and w2 and (weld[par[w1]] == w2 or weld[par[w2]] == w1))

    pairs = []
    for h in range(nh):                       # the oracle's order: hull h against every primitive, then against the later hulls
        for g in range(int(m["ngeom"])):
            if not filtered(int(m["geom_bodyid"][g]), int(m["hull_bodyid"][h])):
                pairs.append((g, NGEOM + h))
        for h2 in range(h + 1, nh):
            if not filtered(int(m["hull_bodyid"][h]), int(m["hull_bodyid"][h2])):
                pairs.append((NGEOM + h, NGEOM + h2))
    assert len(pairs) <= MAXHPAIR, len(pairs)
    d.npair = len(pairs)
    for i, (a, b) in enumerate(pairs):
        d.pair_a[i], d.pair_b[i] = a, b
    verts = np.ascontiguousarray(verts)
    d.vert = verts.ctypes.data_as(C.POINTER(_d))
    return d, verts
