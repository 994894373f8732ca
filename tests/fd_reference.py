"""Plain reference of mjd_transitionFD on the CPU oracle: (A, B, C, D) and the difference rule of every control column.

Every rollout is one oracle mj_step from the restored state (qpos, qvel, ctrl, qacc_warmstart, time):
  * position columns perturbed in the tangent space (mj_integratePos of a unit vector), velocity columns on qvel;
  * control columns by ``control_rule`` (upstream mjd_stepFD's nudge_fwd / nudge_back): centred, forward or backward
    against the nominal rollout, or a zero column when neither side is inside ctrlrange;
  * next states differenced in the tangent space (mj_differentiatePos over the step h = eps or 2 eps), velocities and
    sensordata by plain subtraction times 1 / h, as the oracle's stateDiff and upstream's sensor differences do.
``centered`` false makes every state column a forward difference, as upstream.
"""
from __future__ import annotations

import numpy as np

def _in_range(x1: float, x2: float, lo: float, hi: float) -> bool:
    return lo <= x1 <= hi and lo <= x2 <= hi


def control_rule(u: float, lo: float, hi: float, limited: bool, eps: float, centered: bool) -> str:
    """Which difference upstream mjd_stepFD takes for a control at ``u``:
    nudge_fwd = !limited || inRange(u, u + eps); nudge_back = (centered || !nudge_fwd) && (!limited || inRange(u - eps, u))."""
    fwd = not limited or _in_range(u, u + eps, lo, hi)
    back = (centered or not fwd) and (not limited or _in_range(u - eps, u, lo, hi))
    if fwd and back:
        return "centered"
    return "forward" if fwd else ("backward" if back else "zero")


def transition_fd(model, od, eps: float, centered: bool, sensors: bool = True, rules=None):
    """(A, B, C, D, rules) at the oracle data ``od``'s state: A (2nv, 2nv), B (2nv, nu), C (nsensordata, 2nv),
    D (nsensordata, nu) row-major, rules the ``control_rule`` of each actuator.  The state (and sensordata) are restored on
    return.  ``sensors`` false leaves C and D empty.  ``rules`` (one per actuator) replaces control_rule: the columns a
    kernel that chose another difference would produce."""
    nq, nv, nu = model.nq, model.nv, model.nu
    ns = model.nsensordata if sensors else 0
    keep = (od.qpos, od.qvel, od.ctrl, od.qacc_warmstart, od.sensordata)
    saved = [a.copy() for a in keep]
    t0 = od.time

    def restore():
        for dst, src in zip(keep, saved):
            dst[...] = src
        od.time = t0

    def rollout(perturb=None):
        """(next state [qpos; qvel], sensordata) of one mj_step from the restored state after ``perturb``."""
        restore()
        if perturb is not None:
            perturb()
        od.step()
        out = np.concatenate([od.qpos, od.qvel]), od.sensordata[:ns].copy()
        restore()
        return out

    def diff(s1, s2, h):
        x1, y1 = s1
        x2, y2 = s2
        d = np.concatenate([od.differentiate_pos(h, x1[:nq], x2[:nq]), (x2[nq:] - x1[nq:]) * (1.0 / h)])
        return d, (y2 - y1) * (1.0 / h)

    def quotient(plus, minus, nominal, rule):
        if rule == "centered":
            return diff(minus(), plus(), 2 * eps)
        if rule == "forward":
            return diff(nominal, plus(), eps)
        if rule == "backward":
            return diff(minus(), nominal, eps)
        return np.zeros(2 * nv), np.zeros(ns)

    nominal = rollout()
    q0, v0, u0 = saved[0], saved[1], saved[2]
    A = np.zeros((2 * nv, 2 * nv))
    B = np.zeros((2 * nv, nu))
    C = np.zeros((ns, 2 * nv))
    D = np.zeros((ns, nu))
    state_rule = "centered" if centered else "forward"
    for i in range(nv):
        dp = np.zeros(nv)
        dp[i] = 1.0

        def pos(sign, dp=dp):
            return lambda: rollout(lambda: od.qpos.__setitem__(Ellipsis, od.integrate_pos(q0, dp, sign * eps)))

        A[:, i], C[:, i] = quotient(pos(1), pos(-1), nominal, state_rule)

        def vel(sign, i=i):
            return lambda: rollout(lambda: od.qvel.__setitem__(i, v0[i] + sign * eps))

        A[:, nv + i], C[:, nv + i] = quotient(vel(1), vel(-1), nominal, state_rule)
    if rules is None:
        rules = [control_rule(float(u0[a]), float(model.actuator_ctrlrange[a][0]), float(model.actuator_ctrlrange[a][1]),
                              bool(model.actuator_ctrllimited[a]), eps, centered) for a in range(nu)]
    for a, rule in enumerate(rules):

        def ctl(sign, a=a):
            return lambda: rollout(lambda: od.ctrl.__setitem__(a, u0[a] + sign * eps))

        B[:, a], D[:, a] = quotient(ctl(1), ctl(-1), nominal, rule)
    restore()
    return A, B, C, D, rules
