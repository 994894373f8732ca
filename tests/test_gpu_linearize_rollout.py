"""b2_linearize_rollout on the GPU: (A, B, C, D) at every step of an open-loop control sequence, held to its definition --
the loop  ctrl <- U[t]; b2_linearize_sensors; b2_step(1)  on a copy of the state -- and to the CPU oracle."""
import itertools
import os

import numpy as np
import pytest

from conftest import load_model, oracle_for
from test_gpu_rollout import FP32_RTOL, LANE_RTOL, _batch, _controls, _model, _rel, _states

pytestmark = pytest.mark.gpu

T = 16
N = 64
EPS = {64: 1e-6, 32: 1e-3}  # FP32: a step well above the rounding of the stepped state
# Jacobians, relative to max(1, max |entry|), where they are not bit for bit the loop's:
#  - about the same nominal rows, on the specialised drone kernels: k_linearize_traj is another whole-kernel compilation of
#    the register-resident physics (instruction selection, FMA contraction), so a rollout's stepped state may move in the
#    last bits, amplified by 1 / eps in the quotient (measured on a B200: 1.8e-9 in C, 1.1e-10 in A; test_gpu_sensor_fd
#    sees the same between its two kernels)
#  - about nominal rows that differ from the loop's in the last bits (the specialised kernels): that difference carried
#    through the rollouts and amplified by 1 / eps (measured on a B200: 7.2e-6 FP64 and 5.3e-2 FP32 at eps = 1e-3, both on
#    the specialised cartpole; 1.4e-2 FP32 drone)
SAME_NOMINAL_RTOL = {64: 5e-9, 32: 2e-2}
JAC_RTOL = {64: 3e-5, 32: 1e-1}
ORACLE_RTOL = 1e-6  # test_gpu_parity's bound for b2_linearize against the oracle
ARRAYS = ("qpos", "qvel", "ctrl", "qacc_warmstart")


def _np(t):
    return None if t is None else t.cpu().numpy()


def _loop(model, n, prec, state, U, sensors, steps=T):
    """The definition, on a batch of its own: per step, linearize (b2_linearize_sensors with C / D) at the current state,
    then step(1).  Returns the recorded rows and the flags the loop leaves."""
    import torch

    data = _batch(model, n, prec, state)
    be = data.backend
    eps = EPS[prec]
    rec = {k: [] for k in ("A", "B", "C", "D", "qpos", "qvel", "warm", "sensordata")}
    for t in range(steps):
        rec["qpos"].append(_np(data.qpos)); rec["qvel"].append(_np(data.qvel)); rec["warm"].append(_np(data.qacc_warmstart))
        if U is not None and model.nu:
            data.ctrl.copy_(torch.as_tensor(U[t], device=data.ctrl.device, dtype=data.ctrl.dtype))
        mats = be.linearize_sensors(eps, True) if sensors else be.linearize(eps, True)
        for k, m in zip("ABCD", mats):
            rec[k].append(_np(m))
        be.step(1)
        rec["sensordata"].append(_np(data.sensordata))
    rec["qpos"].append(_np(data.qpos)); rec["qvel"].append(_np(data.qvel)); rec["warm"].append(_np(data.qacc_warmstart))
    out = {k: np.stack(v) for k, v in rec.items() if v}
    return out, _np(data.flags)


def _call(model, n, prec, state, U, sensors, steps=T):
    import torch

    data = _batch(model, n, prec, state)
    before = {k: _np(getattr(data, k)).copy() for k in ARRAYS}
    seq = None if U is None else torch.as_tensor(U, device=data.qpos.device, dtype=data.qpos.dtype)
    res = data.backend.linearize_rollout(seq, steps, EPS[prec], True, sensors)
    out = {k: _np(v) for k, v in zip(("A", "B", "C", "D", "qpos", "qvel", "warm", "sensordata"), res) if v is not None}
    # the state is left as it is
    for k in ARRAYS:
        assert np.array_equal(_np(getattr(data, k)), before[k], equal_nan=True), k
    return out, _np(data.flags), data


def _compare(model, prec, new, ref, warp, sensors, keep=None, exact=True):
    """Rows within test_gpu_rollout's bounds; Jacobians bit for bit where the nominal rows are bit for bit (within
    SAME_NOMINAL_RTOL when not ``exact``), else within JAC_RTOL.  Returns (worst row difference, worst Jacobian difference,
    fraction of (t, env) with identical Jacobians)."""
    tol = 0.0 if warp else (LANE_RTOL if prec == 64 else FP32_RTOL)
    keep = slice(None) if keep is None else keep
    worst_row = 0.0
    for k in ("qpos", "qvel", "warm") + (("sensordata",) if sensors and model.nsensordata else ()):
        assert new[k].shape == ref[k].shape, k
        for t in range(new[k].shape[0]):
            err = _rel(new[k][t][:, keep], ref[k][t][:, keep])
            worst_row = max(worst_row, err)
            assert err <= tol, (k, t, err)
    worst_jac, same, total = 0.0, 0, 0
    mats = "ABCD" if sensors and model.nsensordata else "AB"
    for t in range(new["A"].shape[0]):
        nominal_equal = np.all([np.all((new[k][t] == ref[k][t]) | (np.isnan(new[k][t]) & np.isnan(ref[k][t])), axis=0)
                                for k in ("qpos", "qvel", "warm")], axis=0)
        for e in np.arange(nominal_equal.size)[keep]:
            bits = all(np.array_equal(new[k][t][..., e], ref[k][t][..., e], equal_nan=True) for k in mats)
            same += bits
            total += 1
            if nominal_equal[e] and exact:
                assert bits, (t, e)
            elif not bits:
                bound = SAME_NOMINAL_RTOL[prec] if nominal_equal[e] else JAC_RTOL[prec]
                for k in mats:
                    err = _rel(new[k][t][..., e], ref[k][t][..., e])
                    worst_jac = max(worst_jac, err)
                    assert err <= bound, (k, t, e, bool(nominal_equal[e]), err)
    return worst_row, worst_jac, same / max(total, 1)


CASES = [("pendulum", 64), ("cartpole", 64), ("cartpole-generic", 64), ("drone", 64), ("drone-generic", 64), ("rig-euler", 64),
         ("rig-rk4", 64), ("humanoid", 64), ("humanoid-lane", 64),
         ("cartpole", 32), ("drone", 32), ("drone-generic", 32), ("rig-rk4", 32), ("humanoid", 32)]


@pytest.mark.parametrize("case,prec", CASES)
def test_linearize_rollout_equals_loop(monkeypatch, case, prec):
    model, name = _model(monkeypatch, case)
    sensors = model.nsensordata > 0
    state = _states(model, name, N, seed=21)
    U = _controls(model, N, T, seed=22)
    ref, ref_flags = _loop(model, N, prec, state, U, sensors)
    new, flags, data = _call(model, N, prec, state, U, sensors)
    variant = data.backend.batch.kernel_variant
    forced = lambda var: os.environ.get(var) == "1"  # noqa: E731  (the whole suite may run with either switch set)
    if name == "humanoid":
        assert variant == ("generic" if "lane" in case or forced("B2_DISABLE_WARP") else "generic-warp")
    elif "generic" in case or name == "rig" or forced("B2_DISABLE_SPEC"):
        assert variant == "generic"
    else:
        assert variant == name
    warp = variant == "generic-warp"
    assert new["qpos"].shape == (T + 1, model.nq, N) and new["A"].shape == (T, 2 * model.nv, 2 * model.nv, N)
    assert (("C" in new) == sensors) and (("sensordata" in new) == sensors)
    assert np.array_equal(flags, ref_flags)
    worst_row, worst_jac, same = _compare(model, prec, new, ref, warp, sensors, exact=variant != "drone")
    print(f"linearize_rollout vs loop {case} FP{prec} ({variant}): rows {worst_row:.2e}, Jacobians bit-identical at "
          f"{100 * same:.1f} % of (t, env), worst elsewhere {worst_jac:.2e}")


def test_single_step_equals_linearize_sensors_and_step():
    """T = 1: b2_linearize_sensors at the state, and row 1 is b2_step(1)."""
    import torch

    model = load_model("drone")
    state = _states(model, "drone", N, seed=31)
    U = _controls(model, N, 1, seed=32)
    data = _batch(model, N, 64, state)
    data.ctrl.copy_(torch.as_tensor(U[0], device="cuda"))
    mats = [_np(m) for m in data.backend.linearize_sensors(EPS[64], True)]
    data.backend.step(1)
    new, _, _ = _call(model, N, 64, state, U, True, steps=1)
    for k, m in zip("ABCD", mats):
        err = _rel(new[k][0], m)
        print(f"T = 1 {k}: relative to b2_linearize_sensors {err:.2e}{' (bit-identical)' if np.array_equal(new[k][0], m) else ''}")
        assert err <= JAC_RTOL[64], k
    assert np.array_equal(new["qpos"][0], state[0].T) and np.array_equal(new["qvel"][0], state[1].T)
    assert _rel(new["qpos"][1], _np(data.qpos)) <= LANE_RTOL and _rel(new["qvel"][1], _np(data.qvel)) <= LANE_RTOL
    assert _rel(new["warm"][1], _np(data.qacc_warmstart)) <= LANE_RTOL
    assert _rel(new["sensordata"][0], _np(data.sensordata)) <= LANE_RTOL


@pytest.mark.parametrize("case", ["cartpole", "rig-rk4"])
def test_held_controls(monkeypatch, case):
    model, name = _model(monkeypatch, case)
    sensors = model.nsensordata > 0
    state = _states(model, name, N, seed=41)
    ref, ref_flags = _loop(model, N, 64, state, None, sensors)
    new, flags, _ = _call(model, N, 64, state, None, sensors)
    assert np.array_equal(flags, ref_flags)
    _compare(model, 64, new, ref, False, sensors)


def test_without_a_warm_start():
    """state.qacc_warmstart = NULL: every step starts from zeros (b2_step's rule), and no warm rows are written."""
    import torch

    model = load_model("drone")
    state = _states(model, "drone", N, seed=45)
    U = torch.as_tensor(_controls(model, N, T, seed=46), device="cuda")
    nx = 2 * model.nv
    ref = _batch(model, N, 64, state)
    be = ref.backend
    st = be.state_struct()
    st.qacc_warmstart = None
    A0, q0 = [], []
    stream = torch.cuda.current_stream().cuda_stream
    for t in range(T):
        q0.append(ref.qpos.clone())
        ref.ctrl.copy_(U[t])
        A = torch.empty((nx, nx, N), device="cuda", dtype=torch.float64)
        be.batch.linearize(st, EPS[64], True, A.data_ptr(), None, stream)
        be.batch.step(st, 1, None, stream)
        A0.append(A)
    q0.append(ref.qpos.clone())
    data = _batch(model, N, 64, state)
    st = data.backend.state_struct()
    st.qacc_warmstart = None
    A1 = torch.empty((T, nx, nx, N), device="cuda", dtype=torch.float64)
    q1 = torch.empty((T + 1, model.nq, N), device="cuda", dtype=torch.float64)
    v1 = torch.empty((T + 1, model.nv, N), device="cuda", dtype=torch.float64)
    data.backend.batch.linearize_rollout(st, T, U.data_ptr(), EPS[64], True, A1.data_ptr(), None, None, None, q1.data_ptr(), v1.data_ptr(),
                                         None, None, stream)
    torch.cuda.synchronize()
    assert _rel(_np(q1), _np(torch.stack(q0))) <= LANE_RTOL
    assert _rel(_np(A1), _np(torch.stack(A0))) <= JAC_RTOL[64]


def test_every_null_combination():
    import torch
    from mujoco_template.exceptions import ConfigError, LinearizationError

    model = load_model("drone")
    n, steps = 40, 6
    state = _states(model, "drone", n, seed=51)
    U = torch.as_tensor(_controls(model, n, steps, seed=52), device="cuda")
    data = _batch(model, n, 64, state)
    be = data.backend
    full = [t.clone() for t in be.linearize_rollout(U, steps, EPS[64], True, True)]
    for mask in itertools.product((False, True), repeat=5):  # A, B, C, D, sensordata
        out = [torch.full_like(f, 7.0) if m else None for f, m in zip(full[:4], mask[:4])]
        out += [torch.full_like(f, 7.0) for f in full[4:7]] + [torch.full_like(full[7], 7.0) if mask[4] else None]
        if not any(mask[:4]):
            with pytest.raises(ConfigError):
                be.linearize_rollout(U, steps, EPS[64], True, True, out=out)
            continue
        be.linearize_rollout(U, steps, EPS[64], True, True, out=out)
        for o, f in zip(out, full):
            if o is not None:
                assert torch.equal(o, f), mask
    good = list(full)
    for k in (4, 5, 6):  # qpos / qvel trajectories, and the warm rows of a state with a warm start, are required
        bad = list(good)
        bad[k] = None
        with pytest.raises(ConfigError):
            be.linearize_rollout(U, steps, EPS[64], True, True, out=bad)
    with pytest.raises(LinearizationError):
        be.linearize_rollout(U, steps, 0.0, True, True, out=good)
    with pytest.raises(ConfigError):
        be.linearize_rollout(U, 0, EPS[64], True, True)


@pytest.mark.parametrize("case", ["drone", "rig-euler", "humanoid"])
def test_diverged_env_is_frozen(monkeypatch, case):
    model, name = _model(monkeypatch, case)
    sensors = model.nsensordata > 0
    n = 40
    state = _states(model, name, n, seed=61)
    U = _controls(model, n, T, seed=62)
    bad = 7
    state[1][bad, 0] = 5e9  # the forces this speed produces push the env past the divergence threshold (1e10)
    ref, ref_flags = _loop(model, n, 64, state, U, sensors)
    new, flags, data = _call(model, n, 64, state, U, sensors)
    assert flags[0, bad] & 3 and np.array_equal(flags, ref_flags)
    q, v = new["qpos"], new["qvel"]
    seen = [t for t in range(T + 1) if not np.all(np.abs(np.concatenate([q[t, :, bad], v[t, :, bad]])) <= 1e10)]
    assert seen and seen[0] < T, "the env did not diverge"
    t0 = seen[0]
    for t in range(t0, T + 1):
        for k in ("qpos", "qvel", "warm"):
            assert np.array_equal(new[k][t, :, bad], new[k][t0, :, bad], equal_nan=True), (k, t)
        if sensors and t0 < t < T:
            assert np.all(np.isnan(new["sensordata"][t, :, bad]))
    variant = data.backend.batch.kernel_variant
    keep = np.arange(n) != bad
    _compare(model, 64, new, ref, variant == "generic-warp", sensors, keep=keep, exact=variant != "drone")
    # the frozen env: its state rows and Jacobians are the loop's (the FD about its frozen state); the loop leaves stale
    # sensordata behind for it, the call NaN rows
    for k in ("qpos", "qvel", "warm") + tuple("ABCD" if sensors else "AB"):
        a, b = new[k][..., bad], ref[k][..., bad]
        if variant == "drone":  # the specialised kernels' last-bit differences, grown with the exploding state
            assert np.array_equal(np.isnan(a), np.isnan(b)), k
            if k in ("qpos", "qvel", "warm"):
                assert _rel(np.nan_to_num(a), np.nan_to_num(b)) <= LANE_RTOL, k
        else:
            assert np.array_equal(a, b, equal_nan=True), k


@pytest.mark.parametrize("case", ["cartpole", "drone", "rig-rk4"])
def test_matches_oracle(monkeypatch, case):
    """A_t, B_t at the first, middle and last step against the oracle's transition_fd at the recorded state."""
    model, name = _model(monkeypatch, case)
    n = 4
    state = _states(model, name, n, seed=71)
    U = _controls(model, n, T, seed=72)
    new, _, _ = _call(model, n, 64, state, U, False)
    om, od = oracle_for(model)
    worst = 0.0
    for t in (0, T // 2, T - 1):
        for e in range(n):
            od.reset()
            od.qpos[:] = new["qpos"][t, :, e]; od.qvel[:] = new["qvel"][t, :, e]; od.qacc_warmstart[:] = new["warm"][t, :, e]
            od.ctrl[:] = U[t, :, e]
            Ao, Bo = od.transition_fd(EPS[64], True)
            for a, b in ((new["A"][t, ..., e], Ao), (new["B"][t, ..., e], Bo)):
                err = _rel(a, np.asarray(b))
                worst = max(worst, err)
                assert err <= ORACLE_RTOL, (case, t, e, err)
    print(f"linearize_rollout vs oracle {case}: worst relative difference {worst:.2e}")


def test_two_launches_per_lane_engine_call():
    import torch
    from mujoco_template import _capi

    for name in ("cartpole", "drone"):
        model = load_model(name)
        data = _batch(model, N, 64, _states(model, name, N, seed=1))
        for steps in (1, 16, 200):
            U = torch.as_tensor(_controls(model, N, steps, seed=2), device="cuda")
            before = _capi.launch_count()
            data.backend.linearize_rollout(U, steps, EPS[64], True, name == "drone")
            assert _capi.launch_count() - before == 2, (name, steps)


def test_graph_capture_replays_the_eager_result():
    import torch

    model = load_model("drone")
    state = _states(model, "drone", 256, seed=81)
    data = _batch(model, 256, 64, state)
    be = data.backend
    U = torch.as_tensor(_controls(model, 256, 24, seed=82), device="cuda")
    eager = [t.clone() for t in be.linearize_rollout(U, 24, EPS[64], True, True)]
    out = [torch.empty_like(t) for t in eager]
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        be.linearize_rollout(U, 24, EPS[64], True, True, out=out)
    graph.replay()
    torch.cuda.synchronize()
    for o, e in zip(out, eager):
        assert torch.equal(o, e)


def test_jacobians_beyond_2_pow_31_elements():
    """64-bit offsets and index decode: a pendulum FP32 call whose A has 2.9e9 elements and whose FD launch has more than
    2^31 threads; the last step of the last envs against b2_linearize at the recorded state."""
    import torch
    from mujoco_template import _mj as mj

    model = load_model("pendulum")
    n, steps = 1 << 20, 700
    data = mj.BatchData(model, n, precision=32)
    e = torch.arange(n, device="cuda", dtype=torch.float32)
    data.qpos[0] = torch.sin(e * 0.001) * 3.0
    data.qvel[0] = torch.cos(e * 0.003)
    U = torch.empty((steps, 1, n), device="cuda", dtype=torch.float32)
    for t in range(steps):
        U[t, 0] = torch.sin(e * 0.01 + 0.05 * t) * 4.0
    A, B, _, _, q, v, w, _ = data.backend.linearize_rollout(U, steps, EPS[32], True, False)
    assert A.numel() > 2**31 and 3 * steps * n > 2**31
    pick = torch.tensor([0, 1, n - 2, n - 1], device="cuda")
    small = mj.BatchData(model, pick.numel(), precision=32)
    r = steps - 1
    small.qpos.copy_(q[r][:, pick]); small.qvel.copy_(v[r][:, pick]); small.qacc_warmstart.copy_(w[r][:, pick])
    small.ctrl.copy_(U[r][:, pick])
    As, Bs = small.backend.linearize(EPS[32], True)
    a, b = _np(A[r][:, :, pick]), _np(B[r][:, :, pick])
    print(f"beyond 2^31: last step vs b2_linearize, A {_rel(a, _np(As)):.2e}, B {_rel(b, _np(Bs)):.2e}")
    assert _rel(a, _np(As)) <= JAC_RTOL[32] and _rel(b, _np(Bs)) <= JAC_RTOL[32]
    # and the nominal trajectory of those envs is the one a small batch produces
    small2 = mj.BatchData(model, pick.numel(), precision=32)
    small2.qpos.copy_(q[0][:, pick]); small2.qvel.copy_(v[0][:, pick])
    qs, vs, _ = small2.backend.rollout(U[:, :, pick].contiguous(), steps, True)
    assert _rel(_np(q[steps][:, pick]), _np(qs[-1])) <= FP32_RTOL and _rel(_np(v[steps][:, pick]), _np(vs[-1])) <= FP32_RTOL


def test_batched_env_shapes_and_no_time_or_state_change():
    import torch

    import mujoco_template as mt
    from mujoco_template.exceptions import ConfigError

    model = load_model("drone")
    n, steps = 128, 12
    env = mt.BatchedEnv(model, n)
    qpos, qvel, ctrl, warm = _states(model, "drone", n, seed=91)
    for dst, src in zip((env.data.qpos, env.data.qvel, env.data.ctrl, env.data.qacc_warmstart), (qpos, qvel, ctrl, warm)):
        dst.copy_(torch.as_tensor(src.T.copy(), device="cuda"))
    start = {k: getattr(env.data, k).clone() for k in ARRAYS}
    t0, sub0 = env.data.time, env._substep
    U = torch.as_tensor(_controls(model, n, steps, seed=92), device="cuda").permute(2, 0, 1)  # (nenv, T, nu) view
    out = env.linearize_rollout(U, sensors=True, eps=1e-6)
    nx, nsd = 2 * model.nv, model.nsensordata
    assert out["qpos"].shape == (n, steps + 1, model.nq) and out["qvel"].shape == (n, steps + 1, model.nv)
    assert out["A"].shape == (n, steps, nx, nx) and out["B"].shape == (n, steps, nx, model.nu)
    assert out["C"].shape == (n, steps, nsd, nx) and out["D"].shape == (n, steps, nsd, model.nu)
    assert out["sensordata"].shape == (n, steps, nsd)
    assert env.data.time == t0 and env._substep == sub0
    for k, v in start.items():
        assert torch.equal(getattr(env.data, k), v), k
    assert torch.equal(out["qpos"][:, 0], start["qpos"].T)
    # the same as the backend call on the (T, nu, nenv) layout; without sensors only the four base entries
    ref = env.data.backend.linearize_rollout(U.permute(1, 2, 0).contiguous(), steps, 1e-6, True, True)
    for k, r in zip(("A", "B", "C", "D"), ref[:4]):
        assert torch.equal(out[k], r.permute(3, 0, 1, 2)), k
    plain = env.linearize_rollout(U, eps=1e-6)
    assert set(plain) == {"qpos", "qvel", "A", "B"} and torch.equal(plain["A"], out["A"])
    held = env.linearize_rollout(nsteps=3, eps=1e-6)
    assert held["A"].shape == (n, 3, nx, nx)
    for bad in (U.float(), U[:, :, :2], U.cpu()):
        with pytest.raises(ConfigError):
            env.linearize_rollout(bad)
    with pytest.raises(ConfigError):
        env.linearize_rollout(U, steps - 1)
