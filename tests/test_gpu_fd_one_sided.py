"""One-sided finite differences on the GPU: centered = 0, and control columns within eps of a ctrlrange bound, in every FD
linearisation path (b2_linearize, b2_linearize_sensors, b2_linearize_rollout, b2_control_tick and the single-env
mjd_transitionFD), column by column against the plain reference of the same rollouts (tests/fd_reference.py).

The FD step is a power of two and every edge control is bound + k eps / 2, so u +- eps is exact in FP32 and FP64 and the
kernels make the reference's boundary decisions.  At EPS = 2^-7 forward and centred quotients differ by ~eps |f''| / 2,
well above the tolerances: each test also asserts, on the reference side, that a kernel which ignored ``centered`` or
took the wrong side of a bound would be outside its bound."""
import os

import numpy as np
import pytest

from conftest import oracle_for
from fd_reference import transition_fd
from test_fd_reference import EDGES, EPS, case_model, edge_states, edge_value
from test_gpu_linearize_rollout import _compare
from test_gpu_rollout import _batch, _rel

pytestmark = pytest.mark.gpu

# Floor of a column's scale: a stepped state (or sensor reading) s is rounded to a few units in the last place, so a
# difference quotient of two of them carries ~ 2 k ulp |s| / eps of rounding whatever the column is.  k = 8 and |s| the
# largest entry of the nominal next state (or sensordata), at least 1: FP64 at eps = 2^-7, 16 * 2^-52 * 128 |s| = 4.5e-13 |s|.
# A column whose reference stays below the floor is FD rounding about a true zero (a sensor that does not see a
# translation of the free joint, say): there the two sides only have to agree within the floor (measured on a B200:
# 0.21 of it at worst).  Every other column is compared on its own scale against the bounds below.
FLOOR_ULPS = 16
# Worst per-column relative difference to the reference (max |gpu - ref| over a column / max |ref column|), per path and
# case, FP64 at eps = 2^-7, both modes; measured on a B200 (1000 W) and written after each bound, which is ~10x it.
# The humanoid's columns carry its constraint solver's tolerance (contacts, warm start), 1 / eps amplified.
TOL_LIN = {"pendulum": 8e-12,           # 7.7e-13
           "pendulum-generic": 8e-12,   # 7.7e-13
           "cartpole": 4e-11,           # 3.8e-12
           "cartpole-generic": 8e-11,   # 7.5e-12
           "drone": 1e-11,              # 1.0e-12
           "drone-generic": 1e-11,      # 1.0e-12
           "humanoid": 4e-8,            # 3.7e-9
           "humanoid-lane": 4e-8}       # 3.3e-9
TOL_SENS = {"drone": 1.5e-8,            # 1.3e-9 (C; mjd_transitionFD on one env: 4.8e-10)
            "drone-generic": 1.5e-8,    # 1.3e-9
            "rig-euler": 4e-9,          # 3.4e-10
            "rig-rk4": 4e-9}            # 3.9e-10
# rows t = 0, T / 2, T - 1 of the call; the cartpole's later rows meet its slider limit and contacts (solver tolerance)
TOL_ROLL = {"cartpole": 1e-7,           # 9.9e-9
            "drone": 1.5e-8,            # 1.3e-9
            "rig-rk4": 4e-9,            # 3.9e-10
            "humanoid": 4e-8}           # 3.7e-9
TOL_TICK = {"cartpole": 4e-11,          # 3.9e-12
            "drone": 8e-12,             # 7.7e-13
            "humanoid": 2e-10}          # 1.9e-11
# fused tick against the three-launch sequence (measured: bit-identical in all three cases; the fused kernel evaluates
# the law itself, so the bound allows it to round a control differently)
TOL_FUSED = {"cartpole": 1e-9, "drone": 1e-9, "humanoid": 0.0}
# FP32 against FP64 at the same eps, relative to max(1, max |entry|) of the whole matrix: test_gpu_sensor_fd's bounds,
# 1e-3 for (A, B) and 5e-2 for (C, D) ...
FP32_AB, FP32_CD = 1e-3, 5e-2
# ... except where FP32 at eps = 2^-7 was measured above 1e-3 on a B200: the saturated cartpole tick (the law rounds
# the unsaturated controls differently) and the humanoid, whose one-sided columns difference against a nominal state
# that sits on its foot contacts (centred: 3.7e-5)
FP32_AB_CASE = {("tick", "cartpole"): 2e-2,          # 1.9e-3
                ("linearize", "humanoid"): 2e-2,     # 1.6e-3
                ("linearize", "humanoid-lane"): 2.5e-2,  # 2.5e-3
                ("rollout", "humanoid"): 2e-2,       # (its first step is b2_linearize's state)
                ("tick", "humanoid"): 1.3e-2}        # 1.3e-3 on the lane engine (B2_DISABLE_WARP=1), 8.9e-4 on the warp engine
T = 8  # steps of the linearize_rollout cases


def _n(name):
    return 18 if name == "humanoid" else 36


def _forced(var):
    return os.environ.get(var) == "1"  # the whole suite may run with either switch set


def _setup(monkeypatch, case):
    if "generic" in case:
        monkeypatch.setenv("B2_DISABLE_SPEC", "1")
    if "lane" in case:
        monkeypatch.setenv("B2_DISABLE_WARP", "1")
    return case_model(case)


def _variant(case, name):
    if name == "humanoid":
        return "generic" if "lane" in case or _forced("B2_DISABLE_WARP") else "generic-warp"
    if "generic" in case or name == "rig" or _forced("B2_DISABLE_SPEC"):
        return "generic"
    return name


def _host(t):
    """(rows, cols, N) device matrix -> (N, rows, cols) float64 host array"""
    return t.permute(2, 0, 1).cpu().numpy().astype(np.float64)


def _ref_env(model, od, q, v, u, w, eps, centered, alt=False):
    """Reference at one state: dict of A, B, C, D, rules and the floors of (A, B) and (C, D).  ``alt``: the control columns
    under the other choice (centred -> forward, forward <-> backward), as a kernel that chose wrongly would give them."""
    od.reset()
    od.qpos[:] = q; od.qvel[:] = v; od.ctrl[:] = u; od.qacc_warmstart[:] = w
    od.step()
    fx = FLOOR_ULPS * 2.0 ** -52 * max(1.0, float(np.max(np.abs(np.concatenate([od.qpos, od.qvel]))))) / eps
    fs = FLOOR_ULPS * 2.0 ** -52 * max(1.0, float(np.max(np.abs(od.sensordata)))) / eps if model.nsensordata else 0.0
    od.reset()
    od.qpos[:] = q; od.qvel[:] = v; od.ctrl[:] = u; od.qacc_warmstart[:] = w
    A, B, C, D, rules = transition_fd(model, od, eps, centered)
    if alt:
        flip = {"centered": "forward", "forward": "backward", "backward": "forward", "zero": "zero"}
        A, B, C, D, rules = transition_fd(model, od, eps, centered, rules=[flip[r] for r in rules])
    return dict(A=A, B=B, C=C, D=D, rules=rules, fx=fx, fs=fs)


def _ref_batch(model, state, eps, centered, alt=False):
    om, od = oracle_for(model)
    q, v, u, w = state
    return [_ref_env(model, od, q[e], v[e], u[e], w[e], eps, centered, alt) for e in range(q.shape[0])]


def _col_err(got, ref, floor):
    """per column: max |got - ref| / max(max |ref column|, floor), and whether the column is above the floor"""
    if ref.size == 0:
        return np.zeros(0), np.zeros(0, bool)
    top = np.max(np.abs(ref), axis=0)
    return np.max(np.abs(got - ref), axis=0) / np.maximum(top, floor), top > floor


def _check(label, got, refs, tol, mats="AB"):
    """got: {"A": (N, ...), ...}.  Every column above the floor within tol of the reference on its own scale, every
    column below it within the floor; the zero columns of the reference (controls with no side inside ctrlrange) exactly
    zero.  Returns the worst value of the columns above the floor."""
    worst, where, noise = 0.0, None, 0.0
    for e, ref in enumerate(refs):
        for k in mats:
            err, live = _col_err(got[k][e], ref[k], ref["fx" if k in "AB" else "fs"])
            if np.any(live) and float(np.max(err[live])) > worst:
                worst, where = float(np.max(err[live])), (k, e, int(np.flatnonzero(live)[np.argmax(err[live])]))
            if np.any(~live):
                noise = max(noise, float(np.max(err[~live])))
        for a, r in enumerate(ref["rules"]):
            if r == "zero":
                for k in [m for m in "BD" if m in mats]:
                    assert not np.any(got[k][e][:, a]), (label, k, e, a)
    print(f"{label}: worst per-column relative difference to the reference {worst:.2e} at (matrix, env, column) {where} "
          f"(bound {tol:.1e}); columns below the floor within {noise:.2f} of it")
    assert worst <= tol, (label, where, worst)
    assert noise <= 1.0, (label, noise)
    return worst


def _discriminates(label, model, refs, other, alt, tol, mats="AB"):
    """The reference of the other mode (``other``) and the wrong-side control columns (``alt``) differ from ``refs`` by
    at least 100 x tol in some position, some velocity and some control column: a kernel that ignored ``centered`` or
    took the wrong side of a bound fails the comparison.  (Inside the range the cartpole's and the drone's controls act
    linearly, so there the forward and centred control columns are the same; at a bound the wrong side is not.)"""
    nv = model.nv
    sep = {"position": 0.0, "velocity": 0.0, "control": 0.0}
    for r, o, a in zip(refs, other, alt):
        for k in [m for m in "AC" if m in mats]:
            err, _ = _col_err(o[k], r[k], r["fx" if k == "A" else "fs"])
            if err.size:
                sep["position"] = max(sep["position"], float(np.max(err[:nv])))
                sep["velocity"] = max(sep["velocity"], float(np.max(err[nv:])))
        for k in [m for m in "BD" if m in mats]:
            f = r["fx" if k == "B" else "fs"]
            for x in (o, a):
                err, _ = _col_err(x[k], r[k], f)
                live = [i for i, rule in enumerate(r["rules"]) if rule != "zero"]
                if err.size and live:
                    sep["control"] = max(sep["control"], float(np.max(err[live])))
    print(f"{label}: forward vs centred / wrong side, largest per-column separation " +
          ", ".join(f"{k} {v:.2e}" for k, v in sep.items()) + f" (needed {100 * tol:.1e})")
    for k, v in sep.items():
        assert v >= 100 * tol, (label, k, v)


_REFS = {}


def _refs(case, model, name, state, centered):
    """(reference, other mode, wrong side) of a case's edge states, computed once per session"""
    key = (case.replace("-generic", "").replace("-lane", ""), centered)
    if key not in _REFS:
        _REFS[key] = tuple(_ref_batch(model, state, EPS, c, alt) for c, alt in ((centered, False), (not centered, False), (centered, True)))
    return _REFS[key]


def _edge_case(monkeypatch, case):
    model, name = _setup(monkeypatch, case)
    return model, name, edge_states(model, name, _n(name), EPS, seed=11)


# ----------------------------------------------------------------------------------------------------------- b2_linearize
LIN_CASES = ["pendulum", "pendulum-generic", "cartpole", "cartpole-generic", "drone", "drone-generic", "humanoid", "humanoid-lane"]


@pytest.mark.parametrize("centered", [False, True])
@pytest.mark.parametrize("case", LIN_CASES)
def test_linearize(monkeypatch, case, centered):
    model, name, state = _edge_case(monkeypatch, case)
    data = _batch(model, state[0].shape[0], 64, state)
    assert data.backend.batch.kernel_variant == _variant(case, name)
    A, B = (_host(t) for t in data.backend.linearize(EPS, centered))
    refs, other, alt = _refs(case, model, name, state, centered)
    label = f"b2_linearize {case} centered={int(centered)} ({data.backend.batch.kernel_variant})"
    _check(label, {"A": A, "B": B}, refs, TOL_LIN[case])
    _discriminates(label, model, refs, other, alt, TOL_LIN[case])
    if np.any(model.actuator_ctrllimited):
        seen = {r for ref in refs for r in ref["rules"]}
        assert seen == ({"centered", "forward", "backward", "zero"} if centered else {"forward", "backward", "zero"})


# --------------------------------------------------------------------------------------------------- b2_linearize_sensors
SENS_CASES = ["drone", "drone-generic", "rig-euler", "rig-rk4"]


@pytest.mark.parametrize("centered", [False, True])
@pytest.mark.parametrize("case", SENS_CASES)
def test_linearize_sensors(monkeypatch, case, centered):
    model, name, state = _edge_case(monkeypatch, case)
    data = _batch(model, state[0].shape[0], 64, state)
    assert data.backend.batch.kernel_variant == _variant(case, name)
    A, B, C, D = (_host(t) for t in data.backend.linearize_sensors(EPS, centered))
    refs, other, alt = _refs(case, model, name, state, centered)
    label = f"b2_linearize_sensors {case} centered={int(centered)} ({data.backend.batch.kernel_variant})"
    _check(label, dict(A=A, B=B, C=C, D=D), refs, TOL_SENS[case], mats="ABCD")
    _discriminates(label, model, refs, other, alt, TOL_SENS[case], mats="ABCD")


def test_single_env_transition_fd_one_sided():
    """_mj.mjd_transitionFD(model, data, eps, False, A, B, C, D) on one env (mapped host memory), drone edge states."""
    from mujoco_template import _mj as mj

    model, name = case_model("drone")
    q, v, u, w = edge_states(model, name, len(EDGES), EPS, seed=13)
    refs = _ref_batch(model, (q, v, u, w), EPS, False)
    d1 = mj.MjData(model)
    nx, ns = 2 * model.nv, model.nsensordata
    got = {k: [] for k in "ABCD"}
    for e in range(q.shape[0]):
        d1.qpos[:] = q[e]; d1.qvel[:] = v[e]; d1.ctrl[:] = u[e]; d1.qacc_warmstart[:] = w[e]
        mats = [np.full(s, np.nan) for s in ((nx, nx), (nx, model.nu), (ns, nx), (ns, model.nu))]
        mj.mjd_transitionFD(model, d1, EPS, False, *mats)
        for k, m in zip("ABCD", mats):
            got[k].append(m)
    _check("mjd_transitionFD drone centered=0", {k: np.stack(x) for k, x in got.items()}, refs, TOL_SENS["drone"], mats="ABCD")


# --------------------------------------------------------------------------------------------------- b2_linearize_rollout
ROLL_CASES = ["cartpole", "drone", "rig-rk4", "humanoid"]


def _edge_sequence(model, state, steps, eps, seed):
    """(steps, nu, n): env e keeps its interior controls and moves actuator (7 e) mod nu through the edge table."""
    rng = np.random.default_rng(seed)
    ctrl = state[2]
    n = ctrl.shape[0]
    U = np.repeat(ctrl.T[None], steps, axis=0)
    for e in range(n):
        a = (7 * e) % model.nu
        for t in range(steps):
            U[t, a, e] = edge_value(model, a, EDGES[(e + t) % len(EDGES)], eps, rng)
    return U


def _loop(model, n, prec, state, U, eps, centered, sensors):
    """The definition of b2_linearize_rollout: per step ctrl <- U[t]; b2_linearize_sensors (or b2_linearize); b2_step(1)."""
    import torch

    data = _batch(model, n, prec, state)
    be = data.backend
    rec = {k: [] for k in ("A", "B", "C", "D", "qpos", "qvel", "warm", "sensordata")}
    for t in range(U.shape[0]):
        rec["qpos"].append(data.qpos.cpu().numpy()); rec["qvel"].append(data.qvel.cpu().numpy())
        rec["warm"].append(data.qacc_warmstart.cpu().numpy())
        data.ctrl.copy_(torch.as_tensor(U[t], device=data.ctrl.device, dtype=data.ctrl.dtype))
        mats = be.linearize_sensors(eps, centered) if sensors else be.linearize(eps, centered)
        for k, m in zip("ABCD", mats):
            rec[k].append(m.cpu().numpy())
        be.step(1)
        rec["sensordata"].append(data.sensordata.cpu().numpy())
    rec["qpos"].append(data.qpos.cpu().numpy()); rec["qvel"].append(data.qvel.cpu().numpy())
    rec["warm"].append(data.qacc_warmstart.cpu().numpy())
    return {k: np.stack(v) for k, v in rec.items() if v}


def _rollout(model, n, prec, state, U, eps, centered, sensors):
    import torch

    data = _batch(model, n, prec, state)
    seq = torch.as_tensor(U, device=data.qpos.device, dtype=data.qpos.dtype)
    res = data.backend.linearize_rollout(seq, U.shape[0], eps, centered, sensors)
    out = {k: v.cpu().numpy() for k, v in zip(("A", "B", "C", "D", "qpos", "qvel", "warm", "sensordata"), res) if v is not None}
    return out, data.backend.batch.kernel_variant


@pytest.mark.parametrize("case", ROLL_CASES)
def test_linearize_rollout_one_sided(monkeypatch, case):
    model, name, state = _edge_case(monkeypatch, case)
    n = state[0].shape[0]
    sensors = model.nsensordata > 0
    U = _edge_sequence(model, state, T, EPS, seed=17)
    new, variant = _rollout(model, n, 64, state, U, EPS, False, sensors)
    assert variant == _variant(case, name)
    ref = _loop(model, n, 64, state, U, EPS, False, sensors)
    worst_row, worst_jac, same = _compare(model, 64, new, ref, variant == "generic-warp", sensors, exact=variant != "drone")
    print(f"linearize_rollout centered=0 vs loop {case} ({variant}): rows {worst_row:.2e}, Jacobians bit-identical at "
          f"{100 * same:.1f} % of (t, env), worst elsewhere {worst_jac:.2e}")
    mats = "ABCD" if sensors else "AB"
    om, od = oracle_for(model)
    refs, other, alt, got = [], [], [], {k: [] for k in mats}
    for t in (0, T // 2, T - 1):
        for e in range(n):
            x = (new["qpos"][t, :, e], new["qvel"][t, :, e], U[t, :, e], new["warm"][t, :, e])
            refs.append(_ref_env(model, od, *x, EPS, False))
            other.append(_ref_env(model, od, *x, EPS, True))
            alt.append(_ref_env(model, od, *x, EPS, False, alt=True))
            for k in mats:
                got[k].append(new[k][t, ..., e])
    label = f"linearize_rollout {case} centered=0 ({variant}) at t = 0, {T // 2}, {T - 1}"
    _check(label, {k: np.stack(x) for k, x in got.items()}, refs, TOL_ROLL[case], mats=mats)
    _discriminates(label, model, refs, other, alt, TOL_ROLL[case], mats=mats)
    seen = {r for ref in refs for r in ref["rules"]}
    assert {"forward", "backward", "zero"} <= seen


# ------------------------------------------------------------------------------------------------------- b2_control_tick
TICK_CASES = ["cartpole", "drone", "humanoid"]


def _gain(model, name, state, seed):
    """(K, qpos_ref, ctrl_ref) of a law u = clip(ctrl_ref - K x) that saturates a good share of the envs: K is scaled
    so that |K x| is 1.5 half-ranges for the median env."""
    om, od = oracle_for(model)
    qref = np.array(model.key_qpos[0]) if name == "drone" else np.array(model.qpos0)
    lo, hi = model.actuator_ctrlrange[:, 0], model.actuator_ctrlrange[:, 1]
    uref = (lo + hi) / 2
    x = np.stack([np.concatenate([od.differentiate_pos(1.0, qref, q), v]) for q, v in zip(state[0], state[1])])
    K0 = np.random.default_rng(seed).normal(size=(model.nu, 2 * model.nv))
    K = K0 * (1.5 * np.median((hi - lo) / 2) / np.median(np.abs(x @ K0.T)))
    return K, qref, uref, x


@pytest.mark.parametrize("case", TICK_CASES)
def test_control_tick_one_sided(monkeypatch, case):
    """b2_control_tick(eps, centered = 0) with the LQR law: the fused tick (Euler: the step rides in the FD launch;
    humanoid: law, warp FD and step) against b2_lqr_control, b2_linearize, b2_step, and both against the reference at
    the clipped controls.  Saturated envs sit exactly on a bound: their control columns are one-sided."""
    import torch

    model, name = _setup(monkeypatch, case)
    n = _n(name)
    state = edge_states(model, name, n, EPS, seed=19)
    K, qref, uref, x = _gain(model, name, state, seed=23)
    res = {}
    for fused in (True, False):
        data = _batch(model, n, 64, state)
        be = data.backend
        be.batch.lqr_set_gain(K, qref, uref)
        if fused:
            A, B = be.control_tick(EPS, False, True, derived=False)
        else:
            be.batch.lqr_control(be.state_struct(), torch.cuda.current_stream().cuda_stream)
            A, B = be.linearize(EPS, False)
            be.step(1)
        res[fused] = dict(A=_host(A), B=_host(B), qpos=data.qpos.cpu().numpy().T, qvel=data.qvel.cpu().numpy().T,
                          ctrl=data.ctrl.cpu().numpy().T)
        variant = be.batch.kernel_variant
    assert variant == _variant(case, name)
    worst = 0.0
    for k in ("A", "B"):
        for e in range(n):
            err = _rel(res[True][k][e], res[False][k][e])
            worst = max(worst, err)
            assert err <= TOL_FUSED[case], (k, e, err)
    assert _rel(res[True]["ctrl"], res[False]["ctrl"]) <= 1e-12  # test_gpu_parity's bound for the applied controls
    print(f"control tick {case} ({variant}): fused vs three-launch sequence, worst relative difference {worst:.2e}")
    # the clipped law on the host, and the saturated envs exactly on a bound
    lo, hi = model.actuator_ctrlrange[:, 0], model.actuator_ctrlrange[:, 1]
    u_law = uref - x @ K.T
    u = res[True]["ctrl"]
    sat = (u_law <= lo) | (u_law >= hi)
    assert np.array_equal(u[sat], np.clip(u_law, lo, hi)[sat])
    assert np.max(np.abs(u - np.clip(u_law, lo, hi))) <= 1e-12 * np.max(np.abs(hi))
    assert 0 < np.count_nonzero(sat) < sat.size, "the gain saturates no control, or every one"
    om, od = oracle_for(model)
    refs, other, alt = [], [], []
    for e in range(n):
        x = (state[0][e], state[1][e], u[e], state[3][e])
        refs.append(_ref_env(model, od, *x, EPS, False))
        other.append(_ref_env(model, od, *x, EPS, True))
        alt.append(_ref_env(model, od, *x, EPS, False, alt=True))
        od.reset()
        od.qpos[:] = state[0][e]; od.qvel[:] = state[1][e]; od.ctrl[:] = u[e]; od.qacc_warmstart[:] = state[3][e]
        od.step()
        assert _rel(res[True]["qpos"][e], od.qpos) <= 1e-9 and _rel(res[True]["qvel"][e], od.qvel) <= 1e-9, e
    label = f"control tick {case} centered=0 ({variant})"
    _check(label, res[True], refs, TOL_TICK[case])
    _discriminates(label, model, refs, other, alt, TOL_TICK[case])
    assert {"forward", "backward"} <= {r for ref in refs for r in ref["rules"]}


# --------------------------------------------------------------------------------------------------------- FP32 vs FP64
FP32_CASES = [("linearize", c) for c in ("pendulum", "cartpole", "cartpole-generic", "drone", "humanoid", "humanoid-lane")] + \
             [("sensors", c) for c in ("drone", "drone-generic", "rig-rk4")] + \
             [("rollout", c) for c in ("cartpole", "drone", "rig-rk4", "humanoid")] + \
             [("tick", c) for c in TICK_CASES]


def _zero_columns(m):
    return np.all(m == 0, axis=-2)  # (envs, columns)


@pytest.mark.parametrize("centered", [False, True])
@pytest.mark.parametrize("path,case", FP32_CASES)
def test_fp32_agrees_with_fp64(monkeypatch, path, case, centered):
    """FP32 against FP64 at the same eps = 2^-7: within test_gpu_sensor_fd's bounds (1e-3 of the largest entry for (A, B),
    5e-2 for (C, D)), and the same exactly-zero columns (the same boundary decisions)."""
    import torch

    if path == "tick" and centered:
        pytest.skip("BatchedEnv's control tick is centred and covered by test_gpu_parity; this is the one-sided one")
    model, name, state = _edge_case(monkeypatch, case)
    n = state[0].shape[0]
    out = {}
    for prec in (64, 32):
        data = _batch(model, n, prec, state)
        be = data.backend
        if path == "linearize":
            mats = be.linearize(EPS, centered)
        elif path == "sensors":
            mats = be.linearize_sensors(EPS, centered)
        elif path == "rollout":
            U = torch.as_tensor(_edge_sequence(model, state, T, EPS, seed=17), device="cuda", dtype=data.qpos.dtype)
            # the first step only: later rows of the two precisions are different states (at +-200 N the cartpole's
            # FP32 rows meet its slider limit and contacts at other steps than the FP64 ones)
            mats = [m[0] for m in be.linearize_rollout(U, T, EPS, centered, model.nsensordata > 0)[:4] if m is not None]
        else:
            K, qref, uref, _ = _gain(model, name, state, seed=23)
            be.batch.lqr_set_gain(K, qref, uref)
            mats = be.control_tick(EPS, centered, True, derived=False)
        out[prec] = [_host(m) for m in mats]
    worst = []
    for k, (m64, m32) in enumerate(zip(out[64], out[32])):
        err = max(_rel(m32[e], m64[e]) for e in range(m64.shape[0]))
        worst.append(err)
        assert err <= (FP32_AB_CASE.get((path, case), FP32_AB) if k < 2 else FP32_CD), ("ABCD"[k], err)
        if k in (1, 3):  # control columns: zero exactly where no side of the control is inside ctrlrange, in both
            assert np.array_equal(_zero_columns(m32), _zero_columns(m64)), "ABCD"[k]
    print(f"FP32 vs FP64 {path} {case} centered={int(centered)}: " + ", ".join(f"{'ABCD'[k]} {w:.2e}" for k, w in enumerate(worst)))
