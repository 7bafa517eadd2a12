"""The oracle's restatement of applied forces (test support; not a test module).

`AppliedOracleSim` runs OracleSim's forward stages one by one and adds MuJoCo's applied forces where mj_fwdAcceleration does: the
generalized forces `qfrc_applied` [nv] and, for every body with a nonzero row of `xfrc_applied` [nbody, 6] (world force 0:3, torque
3:6), J' xfrc with the body's Jacobian at its application point `xpos + xmat @ xfrc_point[body]` (mj_xfrcAccumulate; the point
defaults to the body's ipos, MuJoCo's xipos).  The sum joins qfrc_actuator right before o_fwd_acceleration forms qfrc_smooth, so the
unconstrained acceleration, the constraint solve and Euler all see it.  With `applied` False the sim is OracleSim itself; with zero
forces the stage-by-stage path reproduces it bit for bit (tests/test_applied_forces.py).

A reduced body k of the engine is the oracle's k-th jointed body with application point `desc.ipos[k]`, the merged body's centre of
mass in that body's frame (the reduced body keeps its jointed body's frame)."""
import ctypes as C

import numpy as np

from oracle.oracle import OracleEnv, OracleSim

_STAGES = ("o_kinematics", "o_compos", "o_crb", "o_factorM", "o_collision", "o_make_constraint", "o_fwd_velocity", "o_fwd_actuation")


class AppliedOracleSim(OracleSim):
    @classmethod
    def attach(cls, sim):
        """Turns an OracleSim (e.g. an OracleEnv's) into an AppliedOracleSim in place, with zero forces and `applied` False."""
        sim.__class__ = cls
        nb = int(sim.flat["nbody"])
        sim.qfrc_applied = np.zeros(sim.nv)
        sim.xfrc_applied = np.zeros((nb, 6))
        sim.xfrc_point = np.array(sim.flat["body_ipos"], dtype=np.float64).reshape(nb, 3).copy()
        sim.applied = False
        return sim

    def applied_qfrc(self):
        """qfrc_applied + J' xfrc_applied at the current frames (kinematics must be current)."""
        q = np.array(self.qfrc_applied, dtype=np.float64)
        xpos, xmat = self.xpos, self.xmat
        for b in np.flatnonzero(np.any(self.xfrc_applied != 0, axis=1)):
            p = xpos[b] + xmat[b] @ self.xfrc_point[b]
            jp, jr = self.jac(int(b), p)
            q += jp.T @ self.xfrc_applied[b, :3] + jr.T @ self.xfrc_applied[b, 3:]
        return q

    def forward(self):
        if not self.applied:
            return OracleSim.forward(self)
        m = C.byref(self.om)
        for name in _STAGES:
            getattr(self.L, name)(m, self.d)
        self.qfrc_actuator[:] += self.applied_qfrc()
        self.L.o_fwd_acceleration(m, self.d)
        self.L.o_fwd_constraint(m, self.d)

    def step(self, nstep=1):
        if not self.applied:
            return OracleSim.step(self, nstep)
        for _ in range(int(nstep)):
            self.forward()
            self.L.o_euler(C.byref(self.om), self.d)


def applied_oracle_env(flat, **kw):
    """An OracleEnv whose sim is an AppliedOracleSim."""
    oe = OracleEnv(flat, **kw)
    AppliedOracleSim.attach(oe.sim)
    return oe


def set_engine_forces(sim, desc, qfrc, xfrc):
    """The engine's forces of one env (qfrc [18], xfrc [13, 6] over the reduced bodies) on the oracle's unreduced model."""
    jointed = [b for b in range(int(sim.flat["nbody"])) if sim.flat["body_jntnum"][b] > 0]
    sim.qfrc_applied[:] = qfrc
    sim.xfrc_applied[:] = 0
    for k, b in enumerate(jointed):
        sim.xfrc_applied[b] = xfrc[k]
        sim.xfrc_point[b] = np.array(desc.ipos[k][:])
    sim.applied = True
