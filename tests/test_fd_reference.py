"""tests/fd_reference.py on the CPU: its control-column rule written out by hand at every ctrlrange edge, and its
(A, B, C, D) against the oracle's own mjd_transitionFD and the sensor reference, for centred and one-sided differences."""
import warnings

import numpy as np
import pytest

from conftest import load_model, oracle_for
from fd_reference import control_rule, transition_fd
from sensor_fd_reference import transition_fd_sensors
from test_gpu_rollout import _states
from test_oracle_analytic import SENSOR_XML

# A power-of-two FD step at which forward and centred quotients of the smooth models are clearly different (their
# difference, eps |f''| / 2, is ~1e-3 of an entry), and with which every edge control below and u +- eps are exact in
# FP32 and FP64.
EPS = 2.0 ** -7
# Offsets of the edge controls from (lo, lo, lo, lo, -, hi, hi, hi, hi) in units of eps / 2; None: an interior value.
EDGES = ((0, -1), (0, 0), (0, 1), (0, 2), None, (1, -2), (1, -1), (1, 0), (1, 1))


def mixed_rig(integrator: str = "Euler"):
    """test_sensor_fd's sensor rig with a ctrlrange on its second motor only: one unlimited and one limited actuator."""
    from mujoco_template import _mj as mj

    xml = SENSOR_XML.format(dt=0.002).replace('<motor name="m1" joint="twist"/>',
                                              '<motor name="m1" joint="twist" ctrllimited="true" ctrlrange="-0.5 0.75"/>')
    if integrator == "RK4":
        xml = xml.replace("<option ", '<option integrator="RK4" ')
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return mj.MjModel.from_xml_string(xml)


def case_model(case):
    """(model, state family) of a case name: a model name, or rig-euler / rig-rk4 for the mixed rig."""
    if case.startswith("rig"):
        return mixed_rig("RK4" if "rk4" in case else "Euler"), "rig"
    name = case.split("-")[0]
    return load_model(name), name


def edge_value(model, a, edge, eps, rng):
    """Control of actuator ``a`` at an entry of EDGES: bound + k eps / 2, or an interior multiple of eps / 2 at least
    2 eps from either bound.  Unlimited actuators: the pendulum's force clamp (+-3) stands in for the range, the rig's
    motor takes +-1."""
    if model.actuator_ctrllimited[a]:
        lo, hi = (float(x) for x in model.actuator_ctrlrange[a])
    else:
        lo, hi = (-3.0, 3.0) if model.nq == 1 else (-1.0, 1.0)
    if edge is None:
        return lo + 4 * eps + np.floor(rng.uniform(0, hi - lo - 8 * eps) / (eps / 2)) * (eps / 2)
    return (lo, hi)[edge[0]] + edge[1] * eps / 2


def edge_states(model, name, n, eps, seed):
    """(qpos, qvel, ctrl, warm) of n envs: env j puts actuator (7 j) mod nu on EDGES[j mod 9] and every other actuator on
    an interior value, so that one-sided columns of every kind meet centred ones of the same env."""
    qpos, qvel, _, warm = _states(model, name, n, seed)
    rng = np.random.default_rng(seed + 2)
    ctrl = np.array([[edge_value(model, a, None, eps, rng) for a in range(model.nu)] for _ in range(n)])
    for j in range(n):
        a = (7 * j) % model.nu
        ctrl[j, a] = edge_value(model, a, EDGES[j % len(EDGES)], eps, rng)
    return qpos, qvel, ctrl, warm


def _load(od, state, e):
    od.reset()
    for dst, src in zip((od.qpos, od.qvel, od.ctrl, od.qacc_warmstart), state):
        dst[:] = src[e]


# ---------------------------------------------------------------------------------------------------- the rule table
LO, HI, E = -1.5, 2.0, 2.0 ** -4
# (u, limited + centred, limited + one-sided); an unlimited actuator is centred / forward everywhere
TABLE = [
    (LO - E / 2, "zero", "zero"),
    (LO, "forward", "forward"),
    (LO + E / 2, "forward", "forward"),
    (LO + E, "centered", "forward"),
    (0.25, "centered", "forward"),
    (HI - E, "centered", "forward"),
    (HI - E / 2, "backward", "backward"),
    (HI, "backward", "backward"),
    (HI + E / 2, "zero", "zero"),
]


@pytest.mark.parametrize("u,centred,one_sided", TABLE)
def test_control_rule_table(u, centred, one_sided):
    assert control_rule(u, LO, HI, True, E, True) == centred
    assert control_rule(u, LO, HI, True, E, False) == one_sided
    assert control_rule(u, LO, HI, False, E, True) == "centered"
    assert control_rule(u, LO, HI, False, E, False) == "forward"


def test_control_rule_range_narrower_than_eps():
    """Neither u + eps nor u - eps is inside [0, eps / 2]: a zero column although u itself is inside the range."""
    for centered in (True, False):
        assert control_rule(E / 4, 0.0, E / 2, True, E, centered) == "zero"
        assert control_rule(E / 4, 0.0, E / 2, False, E, centered) == ("centered" if centered else "forward")


# -------------------------------------------------------------------------------------- the reference and the oracle
CASES = ["pendulum", "cartpole", "drone", "humanoid", "rig-euler", "rig-rk4"]


@pytest.mark.parametrize("case", CASES)
def test_reference_equals_oracle_transition_fd(case):
    """(A, B) against orc_transition_fd at the edge controls, both modes.  The two run the same oracle steps from the same
    restored state and difference them with the same mj_differentiatePos and reciprocal step, so they agree bit for bit
    (measured: 0 in every case); the only allowance is for a different order of the same products, 1e-15 of the column."""
    model, name = case_model(case)
    n = len(EDGES) if name == "humanoid" else 2 * len(EDGES)
    state = edge_states(model, name, n, EPS, seed=5)
    om, od = oracle_for(model)
    seen, worst = set(), 0.0
    for centered in (True, False):
        for e in range(n):
            _load(od, state, e)
            A, B, _, _, rules = transition_fd(model, od, EPS, centered, sensors=False)
            seen.update(rules)
            Ao, Bo = od.transition_fd(EPS, centered)
            for m, mo in ((A, Ao), (B, Bo)):
                scale = np.maximum(np.max(np.abs(mo), axis=0), 1e-300)
                worst = max(worst, float(np.max(np.abs(m - mo) / scale)))
    print(f"{case}: reference vs orc_transition_fd, worst per-column relative difference {worst:.2e}; rules {sorted(seen)}")
    assert worst <= 1e-15
    if np.any(model.actuator_ctrllimited):  # the edge table reaches every rule
        assert seen == {"centered", "forward", "backward", "zero"}


@pytest.mark.parametrize("case", ["drone", "rig-euler", "rig-rk4"])
def test_reference_equals_sensor_reference(case):
    """(C, D) against sensor_fd_reference.transition_fd_sensors, both modes: the same rollouts, the same quotients."""
    model, name = case_model(case)
    n = 18
    state = edge_states(model, name, n, EPS, seed=7)
    om, od = oracle_for(model)
    worst = 0.0
    for centered in (True, False):
        for e in range(n):
            _load(od, state, e)
            _, _, C, D, _ = transition_fd(model, od, EPS, centered)
            Cs, Ds = transition_fd_sensors(model, od, EPS, centered)
            for m, ms in ((C, Cs), (D, Ds)):
                scale = np.maximum(np.max(np.abs(ms), axis=0), 1e-300)
                worst = max(worst, float(np.max(np.abs(m - ms) / scale)))
            # the state is restored, sensordata included
            assert np.array_equal(od.qpos, state[0][e]) and np.array_equal(od.ctrl, state[2][e])
    print(f"{case}: (C, D) vs transition_fd_sensors, worst per-column relative difference {worst:.2e}")
    assert worst <= 1e-15


def test_one_sided_columns_are_one_sided():
    """Forward and centred references differ where the FD step is visible, and agree on the columns whose rule the mode
    does not change (one-sided at a bound, zero outside the range)."""
    model, name = case_model("drone")
    state = edge_states(model, name, len(EDGES), EPS, seed=9)
    om, od = oracle_for(model)
    for e in range(len(EDGES)):
        _load(od, state, e)
        A1, B1, C1, D1, r1 = transition_fd(model, od, EPS, True)
        A0, B0, C0, D0, r0 = transition_fd(model, od, EPS, False)
        assert np.max(np.abs(A1 - A0)) > 1e-6 * np.max(np.abs(A1))
        for a in range(model.nu):
            if r1[a] == r0[a]:
                assert np.array_equal(B1[:, a], B0[:, a]) and np.array_equal(D1[:, a], D0[:, a]), (e, a, r1[a])
            if r1[a] == "zero":
                assert not np.any(B1[:, a]) and not np.any(D1[:, a])
