"""b2_rollout on the GPU: per-step controls and the recorded trajectory of every env in one call, held to its definition --
the loop  state.ctrl <- U[t]; b2_step(1)  -- and to the CPU oracle."""
import itertools

import numpy as np
import pytest

from conftest import load_model, oracle_for, random_states
from test_sensor_fd import sensor_rig

pytestmark = pytest.mark.gpu

# The lane kernel is a different compilation of the same physics as k_step: FP64 rows within 1e-10 relative over T = 64.
LANE_RTOL = 1e-10
# FP32: the largest 100-step bound of test_gpu_parity's FP32 divergence table for these models (FP32 against FP64)
FP32_RTOL = 5e-5
ORACLE_RTOL = 1e-9  # the parity suite's bound
T = 64


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b))))) if b.size else 0.0


def _model(monkeypatch, case):
    if "generic" in case:
        monkeypatch.setenv("B2_DISABLE_SPEC", "1")
    if "lane" in case:
        monkeypatch.setenv("B2_DISABLE_WARP", "1")
    if case.startswith("rig"):
        return sensor_rig("RK4" if "rk4" in case else "Euler"), "rig"
    name = case.split("-")[0]
    return load_model(name), name


def _states(model, name, n, seed):
    if name == "rig":
        rng = np.random.default_rng(seed)
        qpos = np.tile(model.qpos0, (n, 1))
        qpos[:, :3] = rng.uniform(-0.5, 0.5, (n, 3))
        q = rng.normal(size=(n, 4))
        qpos[:, 6:10] = q / np.linalg.norm(q, axis=1, keepdims=True)
        qvel = rng.normal(size=(n, model.nv))
        ctrl = rng.uniform(-1, 1, (n, model.nu))
    else:
        qpos, qvel, ctrl = random_states(model, name, n, seed=seed)
    warm = np.random.default_rng(seed + 1).normal(0, 0.1, (n, model.nv))
    return qpos, qvel, ctrl, warm


def _controls(model, n, steps, seed):
    """(steps, nu, n) per-env, per-step controls, a quarter of them outside ctrlrange."""
    rng = np.random.default_rng(seed)
    U = np.empty((steps, model.nu, n))
    for a in range(model.nu):
        lo, hi = (float(x) for x in model.actuator_ctrlrange[a])
        if not model.actuator_ctrllimited[a] or hi <= lo:
            lo, hi = -1.0, 1.0
        w = hi - lo
        U[:, a, :] = rng.uniform(lo - 0.15 * w, hi + 0.15 * w, (steps, n))
    return U


def _batch(model, n, prec, state):
    import torch
    from mujoco_template import _mj as mj

    data = mj.BatchData(model, n, precision=prec)
    dev, dt = data.qpos.device, data.qpos.dtype
    for dst, src in zip((data.qpos, data.qvel, data.ctrl, data.qacc_warmstart), state):
        dst.copy_(torch.as_tensor(src.T.copy(), device=dev, dtype=dt))
    return data


DERIVED = ("xpos", "xquat", "site_xpos", "subtree_com", "qacc", "qfrc_bias", "sensordata", "ncon", "nefc", "solver_iter")


def _snapshot(data):
    return {k: getattr(data, k).cpu().numpy().copy() for k in ("qpos", "qvel", "ctrl", "qacc_warmstart", "flags") + DERIVED}


def _loop(model, n, prec, state, U):
    """The definition: state.ctrl <- U[t]; b2_step(1) (derived arrays every step, for the sensor rows)."""
    import torch

    data = _batch(model, n, prec, state)
    q, v, s = [], [], []
    for t in range(U.shape[0]):
        if model.nu:
            data.ctrl.copy_(torch.as_tensor(U[t], device=data.ctrl.device, dtype=data.ctrl.dtype))
        data.backend.step(1)
        q.append(data.qpos.cpu().numpy().copy()); v.append(data.qvel.cpu().numpy().copy()); s.append(data.sensordata.cpu().numpy().copy())
    return np.stack(q), np.stack(v), np.stack(s), _snapshot(data)


def _rollout(model, n, prec, state, U):
    import torch

    data = _batch(model, n, prec, state)
    seq = None if U is None else torch.as_tensor(U, device=data.qpos.device, dtype=data.qpos.dtype)
    q, v, s = data.backend.rollout(seq, T if U is None else U.shape[0], True)
    return q.cpu().numpy(), v.cpu().numpy(), None if s is None else s.cpu().numpy(), _snapshot(data), data


CASES = [("pendulum", 64), ("pendulum-generic", 64), ("cartpole", 64), ("cartpole-generic", 64), ("drone", 64), ("drone-generic", 64),
         ("rig-euler", 64), ("rig-rk4", 64), ("humanoid", 64), ("humanoid-lane", 64),
         ("pendulum", 32), ("cartpole", 32), ("cartpole-generic", 32), ("drone", 32), ("drone-generic", 32), ("rig-rk4", 32), ("humanoid", 32)]


@pytest.mark.parametrize("case,prec", CASES)
def test_rollout_equals_loop_of_single_steps(monkeypatch, case, prec):
    model, name = _model(monkeypatch, case)
    n = 96 if name == "humanoid" else 200
    state = _states(model, name, n, seed=11)
    U = _controls(model, n, T, seed=12)
    q0, v0, s0, end0 = _loop(model, n, prec, state, U)
    q1, v1, s1, end1, data = _rollout(model, n, prec, state, U)
    variant = data.backend.batch.kernel_variant
    import os

    forced = lambda var: os.environ.get(var) == "1"  # noqa: E731  (the whole suite may run with either switch set)
    if name == "humanoid":
        assert variant == ("generic" if "lane" in case or forced("B2_DISABLE_WARP") else "generic-warp")
    elif "generic" in case or name == "rig" or forced("B2_DISABLE_SPEC"):
        assert variant == "generic"
    else:
        assert variant == name
    warp = variant == "generic-warp"
    tol = 0.0 if warp else (LANE_RTOL if prec == 64 else FP32_RTOL)
    worst = 0.0
    for t in range(T):
        for a, b in ((q1[t], q0[t]), (v1[t], v0[t])) + (((s1[t], s0[t]),) if model.nsensordata else ()):
            err = _rel(a, b)
            worst = max(worst, err)
            assert err <= tol, (case, prec, t, err)
    if not model.nsensordata:
        assert s1 is None
    for k in ("qpos", "qvel", "qacc_warmstart") + DERIVED:
        if k in ("ncon", "nefc", "solver_iter", "flags"):
            continue
        worst = max(worst, _rel(end1[k], end0[k]))
        assert _rel(end1[k], end0[k]) <= tol, (case, k)
    assert np.array_equal(end1["ctrl"], end0["ctrl"]) and np.array_equal(end1["ctrl"], U[-1].astype(end1["ctrl"].dtype))
    assert np.array_equal(end1["flags"], end0["flags"])
    if warp or prec == 64:
        for k in ("ncon", "nefc"):
            assert np.array_equal(end1[k], end0[k]), (case, k)
    if warp:
        assert np.array_equal(q1, q0) and np.array_equal(v1, v0)
    # the final state is the last recorded row
    assert np.array_equal(q1[-1], end1["qpos"]) and np.array_equal(v1[-1], end1["qvel"])
    print(f"rollout vs loop {case} FP{prec} ({variant}): worst relative row difference {worst:.2e}")


@pytest.mark.parametrize("name", ["cartpole", "drone", "rig-rk4"])
def test_rollout_matches_oracle(monkeypatch, name):
    model, mname = _model(monkeypatch, name)
    n = 6
    state = _states(model, mname, n, seed=5)
    U = _controls(model, n, T, seed=6)
    q, v, s, _, _ = _rollout(model, n, 64, state, U)
    om, od = oracle_for(model)
    worst = 0.0
    for e in range(n):
        od.reset()
        od.qpos[:] = state[0][e]; od.qvel[:] = state[1][e]; od.qacc_warmstart[:] = state[3][e]
        for t in range(T):
            od.ctrl[:] = U[t, :, e]
            od.step()
            rows = [(q[t, :, e], od.qpos), (v[t, :, e], od.qvel)] + ([(s[t, :, e], od.sensordata)] if model.nsensordata else [])
            for a, b in rows:
                err = _rel(a, np.asarray(b))
                worst = max(worst, err)
                assert err <= ORACLE_RTOL, (name, e, t, err)
    print(f"rollout vs oracle {name}: worst relative row difference {worst:.2e}")


def test_held_controls_and_single_step():
    import torch

    model = load_model("cartpole")
    n = 300
    state = _states(model, "cartpole", n, seed=3)
    ref = _batch(model, n, 64, state)
    ref.backend.step(T)
    q, v, s, end, data = _rollout(model, n, 64, state, None)
    assert (s is None) == (model.nsensordata == 0)
    assert np.array_equal(end["qpos"], q[-1]) and np.array_equal(end["qvel"], v[-1]) and np.array_equal(end["ctrl"], state[2].T)
    assert _rel(q[-1], ref.qpos.cpu().numpy()) <= LANE_RTOL and _rel(v[-1], ref.qvel.cpu().numpy()) <= LANE_RTOL  # b2_step(T)
    # T = 1
    U = _controls(model, n, 1, seed=4)
    q0, v0, _, end0 = _loop(model, n, 64, state, U)
    data = _batch(model, n, 64, state)
    q1, v1, _ = data.backend.rollout(torch.as_tensor(U, device="cuda"), 1, True)
    assert _rel(q1.cpu().numpy(), q0) <= LANE_RTOL and _rel(v1.cpu().numpy(), v0) <= LANE_RTOL
    assert np.array_equal(data.ctrl.cpu().numpy(), U[0])


def test_every_null_combination_of_the_outputs():
    import torch

    model = load_model("drone")
    n = 130
    state = _states(model, "drone", n, seed=8)
    U = torch.as_tensor(_controls(model, n, 20, seed=9), device="cuda")
    data = _batch(model, n, 64, state)
    full = data.backend.rollout(U, 20, True)
    full_end = _snapshot(data)
    for mask in itertools.product((False, True), repeat=3):
        data = _batch(model, n, 64, state)
        out = tuple(torch.full_like(f, 7.0) if m else None for f, m in zip(full, mask))
        data.backend.rollout(U, 20, True, out=out)
        for o, f in zip(out, full):
            if o is not None:
                assert torch.equal(o, f), mask
        end = _snapshot(data)
        for k in ("qpos", "qvel", "qacc_warmstart", "ctrl", "flags", "sensordata", "xpos"):
            assert np.array_equal(end[k], full_end[k]), (mask, k)
    # derived=False leaves the derived arrays alone
    data = _batch(model, n, 64, state)
    data.backend.buffers["xpos"].fill_(3.0)
    data.backend.rollout(U, 20, False, derived=False)
    assert bool((data.backend.buffers["xpos"] == 3.0).all())
    assert np.array_equal(data.qpos.cpu().numpy(), full_end["qpos"])


@pytest.mark.parametrize("case", ["drone", "rig-euler", "humanoid"])
def test_diverged_env_is_frozen(monkeypatch, case):
    """An env driven to a bad state mid-rollout: its rows repeat the frozen state, its sensor rows are NaN, its flags are
    set, and the other envs are as in the loop."""
    model, name = _model(monkeypatch, case)
    n = 40
    state = _states(model, name, n, seed=13)
    U = _controls(model, n, T, seed=14)
    bad = 7
    state[1][bad, 0] = 5e9  # below the divergence threshold (1e10): the forces this speed produces push the env over it
    q0, v0, s0, end0 = _loop(model, n, 64, state, U)
    q1, v1, s1, end1, data = _rollout(model, n, 64, state, U)
    assert end1["flags"][0, bad] & 3 and np.array_equal(end1["flags"], end0["flags"])
    warp = data.backend.batch.kernel_variant == "generic-warp"
    tol = 0.0 if warp else LANE_RTOL
    # the step that detected it: the first whose input state is bad
    seen = [t for t in range(T) if not np.all(np.abs(np.concatenate([q1[t, :, bad], v1[t, :, bad]])) <= 1e10)]
    assert seen, "the env did not diverge"
    t0 = seen[0]
    for t in range(t0, T):
        assert np.array_equal(q1[t, :, bad], q1[t0, :, bad], equal_nan=True) and np.array_equal(v1[t, :, bad], v1[t0, :, bad], equal_nan=True)
        if s1 is not None and t > t0:
            assert np.all(np.isnan(s1[t, :, bad]))
    assert np.array_equal(q1[-1, :, bad], end1["qpos"][:, bad], equal_nan=True)
    assert np.array_equal(end1["ctrl"], U[-1])
    assert np.array_equal(end1["qpos"][:, bad], end0["qpos"][:, bad], equal_nan=True)
    assert np.array_equal(end1["qvel"][:, bad], end0["qvel"][:, bad], equal_nan=True)
    keep = np.arange(n) != bad
    for t in range(T):
        assert _rel(q1[t][:, keep], q0[t][:, keep]) <= tol and _rel(v1[t][:, keep], v0[t][:, keep]) <= tol
        if s1 is not None:
            assert _rel(s1[t][:, keep], s0[t][:, keep]) <= tol


def test_one_launch_per_lane_engine_rollout():
    import torch
    from mujoco_template import _capi

    for name in ("cartpole", "drone"):
        model = load_model(name)
        n = 64
        data = _batch(model, n, 64, _states(model, name, n, seed=1))
        U = torch.as_tensor(_controls(model, n, 500, seed=2), device="cuda")
        before = _capi.launch_count()
        data.backend.rollout(U, 500, True)
        assert _capi.launch_count() - before == 1


def test_batched_env_rollout_shapes_time_and_graph_capture():
    import torch

    import mujoco_template as mt
    from mujoco_template.exceptions import ConfigError

    model = load_model("drone")
    n = 256
    env = mt.BatchedEnv(model, n)
    qpos, qvel, ctrl, warm = _states(model, "drone", n, seed=17)
    for dst, src in zip((env.data.qpos, env.data.qvel, env.data.ctrl, env.data.qacc_warmstart), (qpos, qvel, ctrl, warm)):
        dst.copy_(torch.as_tensor(src.T.copy(), device="cuda"))
    start = {k: getattr(env.data, k).clone() for k in ("qpos", "qvel", "ctrl", "qacc_warmstart")}
    U = torch.as_tensor(_controls(model, n, 30, seed=18), device="cuda").permute(2, 0, 1)  # (nenv, T, nu) view
    traj = env.rollout(controls=U, record=True)
    assert traj["qpos"].shape == (n, 30, model.nq) and traj["qvel"].shape == (n, 30, model.nv)
    assert traj["sensordata"].shape == (n, 30, model.nsensordata)
    assert torch.equal(traj["qpos"][:, -1].T, env.data.qpos) and torch.equal(env.data.ctrl, U[:, -1].T)
    h, t = float(model.opt.timestep), 0.0
    for _ in range(30):
        t += h
    assert env.data.time == t and env._substep == 30
    for bad in (U.float(), U[:, :, :2], U.cpu()):
        with pytest.raises(ConfigError):
            env.rollout(controls=bad)
    with pytest.raises(ConfigError):
        env.rollout(29, controls=U)
    # captured in a CUDA graph: the replay gives the eager result bit for bit
    eager = {k: v.clone() for k, v in traj.items()}
    for k, v in start.items():
        getattr(env.data, k).copy_(v)
    be = env.data.backend
    Uc = U.permute(1, 2, 0).contiguous()
    outs = tuple(torch.empty_like(x.permute(1, 2, 0)) for x in (eager["qpos"], eager["qvel"], eager["sensordata"]))
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        be.rollout(Uc, 30, True, out=outs)
    for k, v in start.items():
        getattr(env.data, k).copy_(v)
    graph.replay()
    torch.cuda.synchronize()
    for o, k in zip(outs, ("qpos", "qvel", "sensordata")):
        assert torch.equal(o.permute(2, 0, 1), eager[k]), k
    assert torch.equal(env.data.qpos, eager["qpos"][:, -1].T)


def test_trajectory_beyond_2_pow_31_elements():
    """Offsets into the (T, dim, N) arrays are 64-bit: a pendulum FP32 rollout with T * N > 2^31 against the same envs
    rolled out in a small batch."""
    import torch
    from mujoco_template import _mj as mj

    model = load_model("pendulum")
    n, steps = 1 << 21, 1100  # 2.3e9 elements per trajectory array
    data = mj.BatchData(model, n, precision=32)
    e = torch.arange(n, device="cuda", dtype=torch.float32)
    data.qpos[0] = torch.sin(e * 0.001) * 3.0
    data.qvel[0] = torch.cos(e * 0.003)
    U = torch.empty((steps, 1, n), device="cuda", dtype=torch.float32)  # beyond the +-3 force clamp in places
    for t in range(steps):
        U[t, 0] = torch.sin(e * 0.01 + 0.05 * t) * 4.0
    pick = torch.tensor([0, 1, 12345, n - 2, n - 1], device="cuda")
    small = mj.BatchData(model, pick.numel(), precision=32)
    small.qpos.copy_(data.qpos[:, pick]); small.qvel.copy_(data.qvel[:, pick])
    q, v, _ = data.backend.rollout(U, steps, True)
    qs, vs, _ = small.backend.rollout(U[:, :, pick].contiguous(), steps, True)
    for r in (steps - 2, steps - 1):
        assert torch.equal(q[r][:, pick], qs[r]) and torch.equal(v[r][:, pick], vs[r])
    assert torch.equal(data.qpos[:, pick], small.qpos)
