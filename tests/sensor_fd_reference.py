"""Reference sensor Jacobians of mjd_transitionFD (C = d sensordata / dx, D = d sensordata / du) on the CPU oracle.

Every rollout is one oracle mj_step from the saved state, exactly the rollouts of the oracle's (A, B): position columns
perturbed in the tangent space (mj_integratePos), velocity columns on qvel, control columns by the ctrlrange rules of B
(centred, one-sided against the nominal rollout at a bound, zero when neither side is inside the range).  A rollout's
reading is the sensordata its mj_step leaves (the forward pass at the perturbed input state; RK4: the first stage only),
differenced by plain subtraction, quaternion components included, as upstream mjd_stepFD does.
"""
from __future__ import annotations

import numpy as np


def transition_fd_sensors(model, od, eps: float, centered: bool):
    """(C, D) row-major (nsensordata x 2nv), (nsensordata x nu) at the oracle data ``od``'s state; the state (and
    sensordata) are restored on return."""
    nv, nu, ns = model.nv, model.nu, model.nsensordata
    saved = [a.copy() for a in (od.qpos, od.qvel, od.ctrl, od.qacc_warmstart, od.sensordata)]
    t0 = od.time

    def restore():
        for dst, src in zip((od.qpos, od.qvel, od.ctrl, od.qacc_warmstart, od.sensordata), saved):
            dst[...] = src
        od.time = t0

    def reading(perturb=None):
        restore()
        if perturb is not None:
            perturb()
        od.step()
        s = od.sensordata.copy()
        restore()
        return s

    def quotient(plus, minus, nominal, fwd, back):
        if fwd and back:
            return (plus() - minus()) * (1.0 / (2 * eps))
        if fwd:
            return (plus() - nominal) * (1.0 / eps)
        if back:
            return (nominal - minus()) * (1.0 / eps)
        return np.zeros(ns)

    nominal = reading()
    C = np.zeros((ns, 2 * nv))
    D = np.zeros((ns, nu))
    q0, v0, u0 = saved[0], saved[1], saved[2]
    for i in range(nv):
        dp = np.zeros(nv)
        dp[i] = 1.0

        def pos(sign, dp=dp):
            return lambda: reading(lambda: od.qpos.__setitem__(Ellipsis, od.integrate_pos(q0, dp, sign * eps)))

        C[:, i] = quotient(pos(1), pos(-1), nominal, True, centered)

        def vel(sign, i=i):
            return lambda: reading(lambda: od.qvel.__setitem__(i, v0[i] + sign * eps))

        C[:, nv + i] = quotient(vel(1), vel(-1), nominal, True, centered)
    for a in range(nu):
        u, lo, hi = u0[a], *model.actuator_ctrlrange[a]
        limited = bool(model.actuator_ctrllimited[a])
        fwd = not limited or (lo <= u <= hi and lo <= u + eps <= hi)
        back = (centered or not fwd) and (not limited or (lo <= u - eps <= hi and lo <= u <= hi))

        def ctl(sign, a=a):
            return lambda: reading(lambda: od.ctrl.__setitem__(a, u0[a] + sign * eps))

        D[:, a] = quotient(ctl(1), ctl(-1), nominal, fwd, back)
    restore()
    return C, D
