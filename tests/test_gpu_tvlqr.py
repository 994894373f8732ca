"""b2_tvlqr and b2_rollout_feedback on the GPU: the backward pass against the NumPy reference (tests/tvlqr_reference.py),
the closed-loop rollout against its definition (the loop  law; b2_step(1)) and against b2_rollout, and the three calls
together: tangent-space sign check, stabilisation and a batched iLQR swing-up.

Bounds are about 10x the worst values measured on a B200 at 1000 W (the tests print them, prefixed MEASURED)."""
import numpy as np
import pytest

import tvlqr_reference as ref
from conftest import load_model, random_states
from test_gpu_rollout import _controls, _model, _states

pytestmark = pytest.mark.gpu

# worst relative difference of K / k / P0 / dV against the FP64 reference; measured: FP64 4.2e-15 on random systems,
# 5.4e-13 on the humanoid's linearize_rollout output; FP32 1.2e-6 on random systems, 1.2e-5 on the humanoid's
TVLQR_RTOL = {64: 5e-12, 32: 1.5e-4}


def _rel(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b))))) if b.size else 0.0


def _dev(x, dtype):
    import torch

    return torch.as_tensor(np.ascontiguousarray(x), device="cuda", dtype=dtype)


def _env_fastest(x, dtype):
    """(N, ...) host array -> CUDA view of env-fastest storage, as linearize_rollout returns them."""
    import torch

    x = np.asarray(x)
    return _dev(np.moveaxis(x, 0, -1), dtype).permute(x.ndim - 1, *range(x.ndim - 1))


def _check_env(res, A, B, Q, R, Qf, q, r, reg, e, tol):
    K, k, P0, dV, status = (t.double().cpu().numpy() for t in res)
    Kr, kr, Pr, dVr, sr = ref.tvlqr(A[e], B[e], Q, R, Qf, None if q is None else q[e], None if r is None else r[e], reg)
    assert status[e] == sr == 0, (e, status[e], sr)
    errs = (_rel(K[e], Kr), _rel(k[e], kr), _rel(P0[e], Pr), _rel(dV[e], dVr))
    assert max(errs) <= tol, (e, errs)
    return max(errs)


SIZES = [(2, 1), (4, 1), (4, 2), (12, 4), (18, 2), (54, 21)]


@pytest.mark.parametrize("prec", [64, 32])
@pytest.mark.parametrize("linear", [False, True])
@pytest.mark.parametrize("nx,nu", SIZES)
def test_tvlqr_matches_reference_on_random_systems(nx, nu, linear, prec):
    import torch

    from mujoco_template.batched_controllers import batched_tvlqr

    dtype = torch.float64 if prec == 64 else torch.float32
    rng = np.random.default_rng(nx * 100 + nu)
    n, T = 37 if nx < 54 else 9, 16  # n not a multiple of the warp kernel's four envs per block
    sysm = [ref.random_system(rng, T, nx, nu, scale=0.1 / np.sqrt(nx)) for _ in range(n)]
    A, B = np.stack([s[0] for s in sysm]), np.stack([s[1] for s in sysm])
    Q, R, Qf = sysm[0][2], sysm[0][3], sysm[0][4]
    q = np.stack([s[5] for s in sysm]) if linear else None
    r = np.stack([s[6] for s in sysm]) if linear else None
    reg = 0.5 if linear else 0.0
    res = batched_tvlqr(_env_fastest(A, dtype), _env_fastest(B, dtype), Q, R, Qf, None if q is None else _env_fastest(q, dtype),
                        None if r is None else _env_fastest(r, dtype), reg)
    if prec == 32:  # the reference on the FP32 inputs
        A, B = A.astype(np.float32).astype(float), B.astype(np.float32).astype(float)
    worst = max(_check_env(res, A, B, Q, R, Qf, q, r, reg, e, TVLQR_RTOL[prec]) for e in range(n))
    print(f"MEASURED tvlqr random {nx}x{nu} linear={linear} fp{prec}: {worst:.2e}")


@pytest.mark.parametrize("prec", [64, 32])
@pytest.mark.parametrize("name", ["cartpole", "drone", "humanoid"])
def test_tvlqr_matches_reference_on_linearize_rollout(name, prec):
    import torch

    import mujoco_template as mt
    from mujoco_template.batched_controllers import batched_tvlqr

    model = load_model(name)
    n, T = (8, 8) if name == "humanoid" else (64, 24)
    env = mt.BatchedEnv(model, n, precision=prec)
    qpos, qvel, ctrl = random_states(model, name, n, seed=3)
    d = env.data
    d.qpos.copy_(_dev(qpos.T, d.qpos.dtype)); d.qvel.copy_(_dev(qvel.T, d.qpos.dtype))
    U = torch.as_tensor(np.repeat(ctrl[:, None, :], T, 1), device=d.qpos.device, dtype=d.qpos.dtype)
    lin = env.linearize_rollout(U, eps=1e-6 if prec == 64 else 1e-3)
    nx, nu = 2 * model.nv, model.nu
    rng = np.random.default_rng(4)
    Q, R = np.diag(rng.uniform(0.5, 2, nx)), np.diag(rng.uniform(0.05, 1, nu))
    q, r = rng.normal(size=(n, T + 1, nx)), rng.normal(size=(n, T, nu))
    res = batched_tvlqr(lin["A"], lin["B"], Q, R, 10 * Q, _env_fastest(q, d.qpos.dtype), _env_fastest(r, d.qpos.dtype), 1e-3)
    A, B = lin["A"].double().cpu().numpy(), lin["B"].double().cpu().numpy()
    worst = max(_check_env(res, A, B, Q, R, 10 * Q, q, r, 1e-3, e, TVLQR_RTOL[prec]) for e in range(n))
    print(f"MEASURED tvlqr linearize_rollout {name} fp{prec}: {worst:.2e}")


@pytest.mark.parametrize("nx,nu", [(4, 1), (4, 2), (12, 4)])
def test_long_horizon_constant_system_matches_dlqr(nx, nu):
    import torch

    from mujoco_template.batched_controllers import batched_dlqr_gain, batched_tvlqr

    rng = np.random.default_rng(7)
    n, T = 16, 800
    A0 = np.eye(nx) + 0.05 * rng.normal(size=(n, nx, nx))
    B0 = 0.1 * rng.normal(size=(n, nx, nu))
    Q, R = np.eye(nx), 0.5 * np.eye(nu)
    Kd, Pd = batched_dlqr_gain(_dev(A0, torch.float64), _dev(B0, torch.float64), Q, R)
    A = np.repeat(A0[:, None], T, 1)
    B = np.repeat(B0[:, None], T, 1)
    K, _, P0, _, status = batched_tvlqr(_env_fastest(A, torch.float64), _env_fastest(B, torch.float64), Q, R)
    assert int(status.abs().max()) == 0
    eK, eP = _rel(K[:, 0].cpu(), Kd.cpu()), _rel(P0.cpu(), Pd.cpu())
    print(f"MEASURED tvlqr vs dlqr {nx}x{nu}: K {eK:.2e} P {eP:.2e}")
    assert eK <= 2e-10 and eP <= 2e-10, (eK, eP)  # measured: 2.1e-11 (4 x 1 K after 800 steps), others <= 1.2e-12


@pytest.mark.parametrize("nx,nu", [(4, 2), (12, 4), (18, 2)])
def test_indefinite_R_gives_status_and_nan_rows_and_reg_removes_them(nx, nu):
    import torch

    from mujoco_template.batched_controllers import batched_tvlqr

    rng = np.random.default_rng(9)
    n, T = 6, 10
    sysm = [ref.random_system(rng, T, nx, nu, scale=0.05) for _ in range(n)]
    A, B = np.stack([s[0] for s in sysm]), np.stack([s[1] for s in sysm])
    Q, Qf = sysm[0][2], sysm[0][4]
    R = np.eye(nu)
    R[-1, -1] = -200.0
    K, k, P0, dV, status = (t.cpu().numpy() for t in batched_tvlqr(_env_fastest(A, torch.float64), _env_fastest(B, torch.float64), Q, R, Qf))
    for e in range(n):
        sr = ref.tvlqr(A[e], B[e], Q, R, Qf)[4]
        assert sr < 0 and status[e] == sr, (e, status[e], sr)
        t = -sr - 1
        assert np.all(np.isnan(K[e, : t + 1])) and np.all(np.isnan(k[e, : t + 1])), e
        assert np.all(np.isfinite(K[e, t + 1:])) and np.all(np.isfinite(k[e, t + 1:])), e
        assert np.all(np.isnan(P0[e])) and np.all(np.isnan(dV[e])), e
    K2, _, P2, dV2, status2 = batched_tvlqr(_env_fastest(A, torch.float64), _env_fastest(B, torch.float64), Q, R, Qf, reg=1e4)
    assert int(status2.abs().max()) == 0 and bool(torch.isfinite(K2).all()) and bool(torch.isfinite(P2).all()) and bool(torch.isfinite(dV2).all())


def test_tvlqr_one_launch_graph_replay_and_shape_checks():
    import torch

    from mujoco_template import _capi
    from mujoco_template.batched_controllers import batched_tvlqr
    from mujoco_template.exceptions import ConfigError

    rng = np.random.default_rng(1)
    for nx, nu in ((4, 1), (12, 4)):
        n, T = 40, 12
        A = _env_fastest(np.eye(nx) + 0.05 * rng.normal(size=(n, T, nx, nx)), torch.float64)
        B = _env_fastest(rng.normal(size=(n, T, nx, nu)), torch.float64)
        Q, R = np.eye(nx), np.eye(nu)
        eager = batched_tvlqr(A, B, Q, R)
        torch.cuda.synchronize()
        c0 = _capi.launch_count()
        batched_tvlqr(A, B, Q, R)
        assert _capi.launch_count() - c0 == 1
        # a captured call writes into buffers that exist before the capture (fixed addresses), as a user's graph would
        out = [torch.empty((T, nu, nx, n), dtype=A.dtype, device="cuda"), torch.empty((T, nu, n), dtype=A.dtype, device="cuda"),
               torch.empty((nx, nx, n), dtype=A.dtype, device="cuda"), torch.empty((2, n), dtype=A.dtype, device="cuda"),
               torch.empty(n, dtype=torch.int32, device="cuda")]
        As, Bs = A.permute(1, 2, 3, 0), B.permute(1, 2, 3, 0)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            _capi.tvlqr(0, 64, T, nx, nu, n, As.data_ptr(), Bs.data_ptr(), Q.reshape(-1), R.reshape(-1), Q.reshape(-1), None, None, 0.0,
                        *[t.data_ptr() for t in out], torch.cuda.current_stream().cuda_stream)
        g.replay()
        torch.cuda.synchronize()
        views = (out[0].permute(3, 0, 1, 2), out[1].permute(2, 0, 1), out[2].permute(2, 0, 1), out[3].permute(1, 0), out[4])
        for a, b in zip(eager, views):
            assert torch.equal(a, b)
    A, B = A.contiguous(), B.contiguous()
    for bad in (lambda: batched_tvlqr(A[..., :-1], B, Q, R), lambda: batched_tvlqr(A, B[:, :-1], Q, R), lambda: batched_tvlqr(A, B.float(), Q, R),
                lambda: batched_tvlqr(A, B, np.eye(3), R), lambda: batched_tvlqr(A, B, Q, R, q=torch.zeros(40, 12, 12, dtype=torch.float64, device="cuda")),
                lambda: batched_tvlqr(A, B, Q, R, r=torch.zeros(40, 12, 4, dtype=torch.float64)), lambda: batched_tvlqr(A[0], B[0], Q, R),
                lambda: batched_tvlqr(A, B, Q, R, reg=-1.0)):
        with pytest.raises(ConfigError):
            bad()


def test_tvlqr_K_beyond_2_31_elements():
    import torch

    from mujoco_template.batched_controllers import batched_tvlqr

    nx, nu, T = 2, 1, 4
    n = (1 << 28) + 96  # K: T nu nx n > 2^31 elements
    g = torch.Generator(device="cuda").manual_seed(0)
    A = torch.randn((T, nx, nx, n), device="cuda", dtype=torch.float32, generator=g).mul_(0.1)
    A[:, 0, 0] += 1; A[:, 1, 1] += 1
    B = torch.randn((T, nx, nu, n), device="cuda", dtype=torch.float32, generator=g)
    Q, R = np.eye(nx), np.eye(nu)
    K, k, P0, dV, status = batched_tvlqr(A.permute(3, 0, 1, 2), B.permute(3, 0, 1, 2), Q, R)
    assert T * nu * nx * n > 2 ** 31
    for e in (0, n // 2, n - 1):
        Kr, kr, Pr, _, _ = ref.tvlqr(A[..., e].double().cpu().numpy(), B[..., e].double().cpu().numpy(), Q, R)
        assert _rel(K[e].double().cpu(), Kr) <= TVLQR_RTOL[32] and _rel(P0[e].double().cpu(), Pr) <= TVLQR_RTOL[32], e
    assert int(status.abs().max()) == 0
    del A, B, K, k, P0, dV


# ---------------------------------------------------------------- b2_rollout_feedback

def _state_batch(model, n, prec, state):
    import torch
    from mujoco_template import _mj as mj

    data = mj.BatchData(model, n, precision=prec)
    for dst, src in zip((data.qpos, data.qvel, data.ctrl, data.qacc_warmstart), state):
        dst.copy_(torch.as_tensor(src.T.copy(), device=data.qpos.device, dtype=data.qpos.dtype))
    return data


def _nominal_rows(data, T):
    """(T, dim, n) rows that repeat the current state (a valid nominal for the tangent-space difference)."""
    return data.qpos[None].repeat(T, 1, 1).contiguous(), data.qvel[None].repeat(T, 1, 1).contiguous()


FB_CASES = [("pendulum", 64), ("pendulum-generic", 64), ("cartpole", 64), ("cartpole-generic", 64), ("drone", 64), ("drone-generic", 64),
            ("rig-euler", 64), ("rig-rk4", 64), ("humanoid", 64), ("humanoid-lane", 64),
            ("cartpole", 32), ("cartpole-generic", 32), ("drone", 32), ("drone-generic", 32), ("humanoid", 32)]


@pytest.mark.parametrize("case,prec", FB_CASES)
def test_zero_gain_is_rollout_of_nominal_and_of_nominal_plus_k(monkeypatch, case, prec):
    """Bit-identical on every kernel set, the specialised ones included (measured: no difference in any case)."""
    import torch

    model, name = _model(monkeypatch, case)
    n, T = (32, 16) if name == "humanoid" else (128, 32)
    state = _states(model, name, n, seed=21)
    U = _controls(model, n, T, seed=22)
    kk = 0.1 * np.random.default_rng(23).normal(size=U.shape)
    worst = 0.0
    for with_k in (False, True):
        d0 = _state_batch(model, n, prec, state)
        dev, dt = d0.qpos.device, d0.qpos.dtype
        seq = torch.as_tensor(U, device=dev, dtype=dt)
        kt = torch.as_tensor(kk, device=dev, dtype=dt)
        q0, v0, s0 = d0.backend.rollout(seq + kt if with_k else seq, T, True)
        d1 = _state_batch(model, n, prec, state)
        qn, vn = _nominal_rows(d1, T)
        K = torch.zeros((T, model.nu, 2 * model.nv, n), device=dev, dtype=dt)
        alpha = torch.ones(n, device=dev, dtype=dt) if with_k else None
        u1, q1, v1, s1 = d1.backend.rollout_feedback(seq, qn, vn, K, kt if with_k else None, alpha, T, True)
        variant = d1.backend.batch.kernel_variant
        tol = 0.0
        pairs = [(q1, q0), (v1, v0), (d1.qpos, d0.qpos), (d1.qvel, d0.qvel), (d1.qacc_warmstart, d0.qacc_warmstart), (d1.xpos, d0.xpos)]
        if s0 is not None:
            pairs.append((s1, s0))
        for a, b in pairs:
            err = _rel(a.double().cpu(), b.double().cpu())
            worst = max(worst, err)
            assert err <= tol, (case, prec, with_k, variant, err)
        # the applied controls: the nominal (plus k), clipped to ctrlrange where limited
        u = (seq + kt if with_k else seq).clone()
        for a in range(model.nu):
            if model.actuator_ctrllimited[a]:
                lo, hi = (float(x) for x in model.actuator_ctrlrange[a])
                u[:, a] = u[:, a].clamp(lo, hi)
        assert torch.equal(u1, u)
        assert torch.equal(d1.ctrl, u[-1])
        assert torch.equal(d1.flags, d0.flags)
    print(f"MEASURED zero-gain feedback vs rollout {case} fp{prec} ({variant}): {worst:.2e}")


def _gains(model, name, n, T, prec, state, U, seed):
    """(lin, K, k) from linearize_rollout + batched_tvlqr about the open-loop rollout of U from `state`."""
    import torch

    import mujoco_template as mt
    from mujoco_template.batched_controllers import batched_tvlqr

    data = _state_batch(model, n, prec, state)
    env = mt.BatchedEnv(model, n, data=data)
    seq = torch.as_tensor(U, device=data.qpos.device, dtype=data.qpos.dtype).permute(2, 0, 1)
    lin = env.linearize_rollout(seq, eps=1e-6 if prec == 64 else 1e-3)
    nx = 2 * model.nv
    rng = np.random.default_rng(seed)
    Q, R = np.diag(rng.uniform(0.5, 2, nx)), np.eye(model.nu)
    K, k, _, _, status = batched_tvlqr(lin["A"], lin["B"], Q, R, 10 * Q, reg=1e-6)
    assert int(status.abs().max()) == 0
    return env, seq, lin, K, k


@pytest.mark.parametrize("case,prec", [("cartpole", 64), ("cartpole-generic", 64), ("drone", 64), ("drone-generic", 64), ("rig-rk4", 64),
                                       ("humanoid", 64), ("humanoid-lane", 64), ("drone-generic", 32), ("humanoid", 32)])
def test_replaying_recorded_controls_reproduces_the_trajectory(monkeypatch, case, prec):
    import torch

    model, name = _model(monkeypatch, case)
    n, T = (16, 12) if name == "humanoid" else (64, 24)
    state = _states(model, name, n, seed=31)
    U = _controls(model, n, T, seed=32) * 0.5
    env, seq, lin, K, k = _gains(model, name, n, T, prec, state, U, 33)
    # start off the nominal: the law acts
    d1 = _state_batch(model, n, prec, state)
    d1.qvel.add_(0.05)
    env1 = type(env)(model, n, data=d1)
    alpha = torch.linspace(0.2, 1.0, n, device=d1.qpos.device, dtype=d1.qpos.dtype)
    rec = env1.rollout_feedback(seq, K, lin["qpos"], lin["qvel"], k=k, alpha=alpha, record=True)
    d0 = _state_batch(model, n, prec, state)
    d0.qvel.add_(0.05)
    q0, v0, _ = d0.backend.rollout(rec["ctrl"].permute(1, 2, 0).contiguous(), T, True)
    variant = d1.backend.batch.kernel_variant
    tol = 0.0  # bit-identical on every kernel set (measured)
    err = max(_rel(rec["qpos"].permute(1, 2, 0).double().cpu(), q0.double().cpu()), _rel(rec["qvel"].permute(1, 2, 0).double().cpu(), v0.double().cpu()),
              _rel(d1.qpos.double().cpu(), d0.qpos.double().cpu()))
    print(f"MEASURED replay of recorded controls {case} fp{prec} ({variant}): {err:.2e}")
    assert err <= tol, (case, variant, err)
    assert bool(torch.isfinite(rec["ctrl"]).all())


def _law_loop(data, model, seq, qn, vn, K, k, alpha, T):
    """The definition: u = clip(ubar + alpha k - K [q (-) qbar ; v - vbar]); b2_step(1), with the law in torch."""
    import torch

    b = data.backend
    nv = model.nv
    dq = torch.empty_like(data.qvel)
    lo = torch.as_tensor(model.actuator_ctrlrange[:, 0], device=dq.device, dtype=dq.dtype)[:, None]
    hi = torch.as_tensor(model.actuator_ctrlrange[:, 1], device=dq.device, dtype=dq.dtype)[:, None]
    lim = torch.as_tensor(np.asarray(model.actuator_ctrllimited, dtype=bool), device=dq.device)[:, None]
    qs = []
    for t in range(T):
        b._pre()
        b.batch.differentiate_pos(dq.data_ptr(), 1.0, qn[t].data_ptr(), data.qpos.data_ptr(), b.stream)
        x = torch.cat([dq, data.qvel - vn[t]], 0)  # (2nv, n)
        u = seq[t] + alpha[None] * k[t] - torch.einsum("ajn,jn->an", K[t], x)
        data.ctrl.copy_(torch.where(lim, torch.minimum(torch.maximum(u, lo), hi), u))
        b.step(1)
        qs.append(data.qpos.clone())
    return torch.stack(qs)


@pytest.mark.parametrize("case", ["cartpole-generic", "drone-generic", "rig-euler", "humanoid"])
def test_rollout_feedback_matches_the_law_step_loop(monkeypatch, case):
    import torch

    model, name = _model(monkeypatch, case)
    n, T = (16, 10) if name == "humanoid" else (64, 20)
    state = _states(model, name, n, seed=41)
    U = _controls(model, n, T, seed=42) * 0.5
    env, seq, lin, K, k = _gains(model, name, n, T, 64, state, U, 43)
    qn, vn = lin["qpos"].permute(1, 2, 0), lin["qvel"].permute(1, 2, 0)
    Ks, ks = K.permute(1, 2, 3, 0), k.permute(1, 2, 0)
    alpha = torch.full((n,), 0.7, device=qn.device, dtype=qn.dtype)
    d0 = _state_batch(model, n, 64, state); d0.qvel.add_(0.03)
    q0 = _law_loop(d0, model, seq.permute(1, 2, 0), qn, vn, Ks, ks, alpha, T)
    d1 = _state_batch(model, n, 64, state); d1.qvel.add_(0.03)
    _, q1, _, _ = d1.backend.rollout_feedback(seq.permute(1, 2, 0).contiguous(), qn, vn, Ks, ks, alpha, T, True)
    err = _rel(q1.cpu(), q0.cpu())
    print(f"MEASURED feedback vs torch law loop {case}: {err:.2e}")
    assert err <= 3e-13, (case, err)  # the law's sums in another order; measured worst 2.4e-14 (cartpole)


def _deviation(data, q, v, qbar, vbar):
    import torch

    b = data.backend
    dq = torch.empty_like(v)
    b._pre()
    b.batch.differentiate_pos(dq.data_ptr(), 1.0, qbar.data_ptr(), q.data_ptr(), b.stream)
    return torch.cat([dq, v - vbar], 0)


@pytest.mark.parametrize("case", ["cartpole", "drone", "rig-euler", "humanoid"])
def test_closed_loop_deviation_follows_the_linearisation_to_second_order(monkeypatch, case):
    """Start at x0 (+) delta: the closed-loop deviation follows prod (A_t - B_t K_t) delta up to O(|delta|^2), so halving
    delta quarters the residual.  Checks the sign of K and the tangent space of the law against those of A."""
    import torch

    model, name = _model(monkeypatch, case)
    n, T = 8, 8
    state = _states(model, name, n, seed=51)
    U = _controls(model, n, T, seed=52)
    for a in range(model.nu):  # controls well inside ctrlrange: no clipping
        lo, hi = (float(x) for x in model.actuator_ctrlrange[a])
        if model.actuator_ctrllimited[a]:
            U[:, a] = 0.5 * (lo + hi) + 0.2 * (hi - lo) * np.tanh(U[:, a])
    env, seq, lin, K, k = _gains(model, name, n, T, 64, state, U, 53)
    qn, vn = lin["qpos"].permute(1, 2, 0), lin["qvel"].permute(1, 2, 0)
    A, B = lin["A"].permute(1, 2, 3, 0), lin["B"].permute(1, 2, 3, 0)
    Ks = K.permute(1, 2, 3, 0)
    dirn = torch.as_tensor(np.random.default_rng(54).normal(size=(2 * model.nv, n)), device=qn.device, dtype=qn.dtype)
    res = []
    # the humanoid's contacts make its map smooth only piecewise: a perturbation of 1e-4 already changes the contact set
    for scale in ((1e-6, 5e-7) if name == "humanoid" else (1e-4, 5e-5)):
        d = _state_batch(model, n, 64, state)
        delta = scale * dirn
        d.backend._pre()
        d.backend.batch.integrate_pos(d.qpos.data_ptr(), delta[: model.nv].contiguous().data_ptr(), 1.0, d.backend.stream)
        d.qvel.add_(delta[model.nv:])
        x = _deviation(d, d.qpos, d.qvel, qn[0], vn[0])
        _, q1, v1, _ = d.backend.rollout_feedback(seq.permute(1, 2, 0).contiguous(), qn, vn, Ks, None, None, T, True)
        worst = 0.0
        for t in range(T):
            x = torch.einsum("ijn,jn->in", A[t] - torch.einsum("ian,ajn->ijn", B[t], Ks[t]), x)
            actual = _deviation(d, q1[t].contiguous(), v1[t].contiguous(), qn[t + 1].contiguous(), vn[t + 1])
            worst = max(worst, float((actual - x).abs().max()))
        res.append(worst)
    ratio = res[0] / res[1]
    print(f"MEASURED second-order residual {case}: {res[0]:.2e} -> {res[1]:.2e}, ratio {ratio:.2f}")
    assert 3.0 <= ratio <= 5.0, (case, res)


def test_cartpole_tvlqr_stabilises_the_upright_nominal():
    import torch

    import mujoco_template as mt
    from mujoco_template.batched_controllers import batched_tvlqr

    model = load_model("cartpole")
    n, T = 64, 500
    env = mt.BatchedEnv(model, n)
    d = env.data
    d.qpos.zero_(); d.qvel.zero_(); d.ctrl.zero_()
    U = torch.zeros((n, T, 1), device=d.qpos.device, dtype=d.qpos.dtype)
    lin = env.linearize_rollout(U)
    Q = np.diag([10.0, 10.0, 1.0, 1.0])
    K, k, _, _, status = batched_tvlqr(lin["A"], lin["B"], Q, np.eye(1) * 0.01, 100 * Q)
    assert int(status.abs().max()) == 0
    dq = torch.as_tensor(np.random.default_rng(61).uniform(-0.05, 0.05, (2, n)), device=d.qpos.device, dtype=d.qpos.dtype)

    def start():
        d.qpos.copy_(dq); d.qvel.zero_()

    start()
    closed = env.rollout_feedback(U, K, lin["qpos"], lin["qvel"], record=True)
    start()
    opened = env.rollout(controls=U, record=True)
    dev_c = float((closed["qpos"][:, -1] - lin["qpos"][:, T]).abs().max())
    dev_o = float((opened["qpos"][:, -1] - lin["qpos"][:, T]).abs().max())
    print(f"MEASURED cartpole stabilisation: closed {dev_c:.2e} open {dev_o:.2e}")
    assert dev_c * 100 <= dev_o, (dev_c, dev_o)


def test_ilqr_pendulum_swing_up():
    """iLQR from the three calls: linearize_rollout -> batched_tvlqr -> rollout_feedback with per-env backtracking."""
    import torch

    import mujoco_template as mt
    from mujoco_template.batched_controllers import batched_tvlqr

    model = load_model("pendulum")
    n, T, iters = 16, 150, 12
    env = mt.BatchedEnv(model, n)
    d = env.data
    dev, dt = d.qpos.device, d.qpos.dtype
    x0 = torch.as_tensor(np.random.default_rng(71).uniform(-0.3, 0.3, (1, n)), device=dev, dtype=dt)
    goal = np.pi
    Q, R, Qf = np.diag([1.0, 0.1]), np.eye(1) * 0.01, np.diag([100.0, 10.0])
    Qt, Qft, Rt = (torch.as_tensor(M, device=dev, dtype=dt) for M in (Q, Qf, R))

    def reset():
        d.qpos.copy_(x0); d.qvel.zero_()

    def traj_cost(qs, vs, us):  # qs, vs (n, T+1, 1); us (n, T, 1)
        x = torch.cat([qs - goal, vs], -1)
        run = 0.5 * torch.einsum("nti,ij,ntj->n", x[:, :T], Qt, x[:, :T]) + 0.5 * torch.einsum("nti,ij,ntj->n", us, Rt, us)
        return run + 0.5 * torch.einsum("ni,ij,nj->n", x[:, T], Qft, x[:, T])

    ubar = torch.zeros((n, T, 1), device=dev, dtype=dt)
    reset()
    lin = env.linearize_rollout(ubar)
    J = traj_cost(lin["qpos"], lin["qvel"], ubar)
    J0 = J.clone()
    for it in range(iters):
        x = torch.cat([lin["qpos"] - goal, lin["qvel"]], -1)
        q = torch.einsum("ij,ntj->nti", Qt, x)
        q[:, T] = torch.einsum("ij,nj->ni", Qft, x[:, T])
        r = torch.einsum("ij,ntj->nti", Rt, ubar)
        K, k, _, dV, status = batched_tvlqr(lin["A"], lin["B"], Q, R, Qf, q, r, reg=1e-6)
        assert int(status.abs().max()) == 0
        alpha = torch.ones(n, device=dev, dtype=dt)
        accepted = torch.zeros(n, dtype=torch.bool, device=dev)
        best = None
        for _ in range(10):
            reset()
            rec = env.rollout_feedback(ubar, K, lin["qpos"], lin["qvel"], k=k, alpha=alpha, record=True)
            qs = torch.cat([x0.T[:, None], rec["qpos"]], 1)
            vs = torch.cat([torch.zeros_like(x0.T[:, None]), rec["qvel"]], 1)
            Jn = traj_cost(qs, vs, rec["ctrl"])
            take = ~accepted & (Jn < J)
            best = rec["ctrl"].clone() if best is None else best
            best[take] = rec["ctrl"][take]
            J = torch.where(take, Jn, J)
            accepted |= take
            if bool(accepted.all()):
                break
            alpha = torch.where(accepted, alpha, alpha * 0.5)
        ubar = torch.where(accepted[:, None, None], best, ubar)
        reset()
        lin = env.linearize_rollout(ubar)
        Jc = traj_cost(lin["qpos"], lin["qvel"], ubar)
        assert bool((Jc <= J * (1 + 1e-9) + 1e-9).all())  # accepted steps never raise the cost
        J = Jc
    frac = float((J / J0).max())
    print(f"MEASURED iLQR pendulum: worst J_final / J_start after {iters} iterations {frac:.3e}")
    assert frac <= 0.45, frac  # measured 0.387


@pytest.mark.parametrize("case", ["cartpole", "cartpole-generic", "humanoid"])
def test_diverged_env_is_frozen_with_nan_control_rows(monkeypatch, case):
    import torch

    model, name = _model(monkeypatch, case)
    n, T = 8, 6
    state = list(_states(model, name, n, seed=81))
    d = _state_batch(model, n, 64, state)
    qn, vn = _nominal_rows(d, T)
    d.qvel[0, 3] = float("nan")
    u_before = d.ctrl[:, 3].clone()
    seq = torch.zeros((T, model.nu, n), device=d.qpos.device, dtype=d.qpos.dtype)
    K = torch.zeros((T, model.nu, 2 * model.nv, n), device=d.qpos.device, dtype=d.qpos.dtype)
    u, q, v, _ = d.backend.rollout_feedback(seq, qn, vn, K, None, None, T, True)
    assert bool(torch.isnan(u[:, :, 3]).all()) and bool(torch.isfinite(u[:, :, [0, 1, 2, 4, 5, 6, 7]]).all())
    assert torch.equal(d.ctrl[:, 3], u_before)
    assert int(d.flags[0, 3]) & 2 and int(d.flags[0, 0]) & 3 == 0
    assert torch.equal(q[:, :, 3], q[:1, :, 3].expand(T, -1)) and torch.equal(q[0, :, 3], qn[0, :, 3])


@pytest.mark.parametrize("case", ["drone", "drone-generic", "rig-rk4", "humanoid"])
def test_every_null_combination_and_one_launch_and_graph_replay(monkeypatch, case):
    import itertools

    import torch

    from mujoco_template import _capi

    model, name = _model(monkeypatch, case)
    n, T = 16, 5
    state = _states(model, name, n, seed=91)
    U = _controls(model, n, T, seed=92)
    env, seq, lin, K, k = _gains(model, name, n, T, 64, state, U, 93)
    seq = seq.permute(1, 2, 0).contiguous()
    qn, vn = lin["qpos"].permute(1, 2, 0), lin["qvel"].permute(1, 2, 0)
    Ks, ks = K.permute(1, 2, 3, 0), k.permute(1, 2, 0)
    alpha = torch.linspace(0.1, 1, n, device=qn.device, dtype=qn.dtype)
    ref_runs = {}
    for use_k, use_a in itertools.product((False, True), repeat=2):
        d = _state_batch(model, n, 64, state)
        ref_runs[use_k, use_a] = (d.backend.rollout_feedback(seq, qn, vn, Ks, ks if use_k else None, alpha if use_a else None, T, True), d)
    # k NULL = 0 and alpha NULL = 1
    (u_na, *_), _ = ref_runs[False, True]
    (u_nn, *_), _ = ref_runs[False, False]
    assert torch.equal(u_na, u_nn)
    full, dfull = ref_runs[True, True]
    for mask in itertools.product((False, True), repeat=4):
        d = _state_batch(model, n, 64, state)
        out = tuple(torch.empty_like(t) if (t is not None and m) else None for t, m in zip(full, mask))
        d.backend.rollout_feedback(seq, qn, vn, Ks, ks, alpha, T, False, out=out)
        for t, f in zip(out, full):
            if t is not None:
                assert torch.equal(t, f), mask
        assert torch.equal(d.qpos, dfull.qpos) and torch.equal(d.ctrl, dfull.ctrl)
    d = _state_batch(model, n, 64, state)
    bufs = tuple(None if t is None else torch.empty_like(t) for t in full)
    torch.cuda.synchronize()
    c0 = _capi.launch_count()
    d.backend.rollout_feedback(seq, qn, vn, Ks, ks, alpha, T, False, out=bufs)
    if d.backend.batch.kernel_variant != "generic-warp":
        assert _capi.launch_count() - c0 == 1
    # graph replay equals the eager result
    d = _state_batch(model, n, 64, state)
    d.backend.rollout_feedback(seq, qn, vn, Ks, ks, alpha, T, False, out=bufs)  # warm-up
    x0 = [t.clone() for t in (d.qpos, d.qvel, d.ctrl, d.qacc_warmstart)]
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        d.backend.rollout_feedback(seq, qn, vn, Ks, ks, alpha, T, False, out=bufs)
    s0 = _state_batch(model, n, 64, state)
    for dst, src in zip((d.qpos, d.qvel, d.ctrl, d.qacc_warmstart), (s0.qpos, s0.qvel, s0.ctrl, s0.qacc_warmstart)):
        dst.copy_(src)
    d.flags.zero_()
    g.replay()
    torch.cuda.synchronize()
    for t, f in zip(bufs, full):
        if t is not None:
            assert torch.equal(t, f)
    assert torch.equal(d.qpos, dfull.qpos)
    del x0
