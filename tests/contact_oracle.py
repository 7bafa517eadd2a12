"""The oracle's restatement of the contact output (test support; not a test module).

`contact_forces(sim)` lists the contacts of an OracleSim after its last forward pass with MuJoCo's `mj_contactForce`: the contact's
pyramid forces `efc_force[efc_address : efc_address + 2 (dim - 1)]` decoded like `mju_decodePyramid` with the contact's mixed
friction (sliding, sliding, torsional: the maximum of the two geoms' `geom_friction`, mj_contactParam).  Contact rows come last, in
contact order, so a contact's efc_address is nefc minus the rows of it and of the contacts after it.  `slots` lays such a list out like
`MyCobotVectorEnv.contacts()`.  The oracle's geoms are the engine's: the compiled model has exactly the MCB_NGEOM primitive geoms."""
import numpy as np

from mycobotgym_b200 import flatten


def contact_forces(sim):
    """[dict(geom1, geom2, dim, dist, pos[3], frame[3, 3], force[6], friction[3])] for the contacts of `sim`'s last forward pass;
    force is in the contact frame (normal, tangent 1, tangent 2, torsional, 0, 0), acting on geom2."""
    fr = np.asarray(sim.flat["geom_friction"], dtype=np.float64).reshape(-1, 3)
    cons = sim.contacts()
    f = np.array(sim.efc("force"))
    adr = sim.nefc - sum(2 * (c["dim"] - 1) for c in cons)
    out = []
    for c in cons:
        g1, g2, dim = c["geom1"], c["geom2"], c["dim"]
        assert dim in (3, 4), dim
        mu = np.array([max(fr[g1, 0], fr[g2, 0]), max(fr[g1, 0], fr[g2, 0]), max(fr[g1, 1], fr[g2, 1])])
        p = f[adr:adr + 2 * (dim - 1)]
        force = np.zeros(6)
        for k in range(2 * (dim - 1)):
            force[0] += p[k]
        for i in range(dim - 1):
            force[i + 1] = (p[2 * i] - p[2 * i + 1]) * mu[i]
        adr += 2 * (dim - 1)
        out.append(dict(c, force=force, friction=mu))
    return out


def world_force(c):
    """The contact's force on geom2 in world coordinates: frame' force[:3]."""
    return c["frame"].T @ c["force"][:3]


def generalized_force(sim, contacts):
    """sum_c J_c' (world force, torsional torque) with J_c the difference of geom2's and geom1's body Jacobians at the contact point:
    the contacts' share of qfrc_constraint."""
    gb = np.asarray(sim.flat["geom_bodyid"])
    q = np.zeros(sim.nv)
    for c in contacts:
        F, T = world_force(c), c["frame"][0] * c["force"][3]
        for body, sign in ((int(gb[c["geom2"]]), 1.0), (int(gb[c["geom1"]]), -1.0)):
            jp, jr = sim.jac(body, c["pos"])
            q += sign * (jp.T @ F + jr.T @ T)
    return q


def slots(contacts):
    """`contacts` in the layout of MyCobotVectorEnv.contacts() for one env (numpy): empty slots zero, geom ids -1."""
    K = flatten.MAXCON
    assert len(contacts) <= K
    out = dict(ncon=len(contacts), geom=np.full((K, 2), -1, np.int32), dim=np.zeros(K, np.int32), dist=np.zeros(K),
               pos=np.zeros((K, 3)), frame=np.zeros((K, 3, 3)), force=np.zeros((K, 6)))
    for i, c in enumerate(contacts):
        out["geom"][i] = (c["geom1"], c["geom2"])
        out["dim"][i] = c["dim"]
        out["dist"][i] = c["dist"]
        out["pos"][i] = c["pos"]
        out["frame"][i] = c["frame"]
        out["force"][i] = c["force"]
    return out
