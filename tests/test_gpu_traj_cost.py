"""b2_traj_cost and batched_ilqr on the GPU: the kernel against the NumPy reference (tests/traj_cost_reference.py) on every
size class and both engines, its gradient against central differences through b2_integrate_pos, the four iLQR calls
against each other (first-order consistency of J(alpha) with dV), and the iLQR driver on a pendulum swing-up and a drone
reaching a yawed goal pose.

Bounds are about 10x the worst values measured on a B200 at 1000 W (the tests print them, prefixed MEASURED)."""
import ctypes as C
import warnings

import numpy as np
import pytest

import traj_cost_reference as ref
from conftest import load_model, random_states

pytestmark = pytest.mark.gpu

# worst error of J / q / r against the FP64 reference, relative to the largest reference value of the env; measured:
# FP64 4.9e-16 (drone), FP32 2.3e-7 (drone)
COST_RTOL = {64: 5e-15, 32: 3e-6}


def _rel(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b))))) if b.size else 0.0


def _model(monkeypatch, case):
    if "lane" in case:
        monkeypatch.setenv("B2_DISABLE_WARP", "1")
    if "generic" in case:
        monkeypatch.setenv("B2_DISABLE_SPEC", "1")
    name = case.split("-")[0]
    return load_model(name), name


def _problem(model, name, n, T, seed, max_angle=2.5):
    """Random trajectories (n, T+1, nq) ..., references with rotation errors up to max_angle, non-diagonal SPD weights
    whose rotation blocks are anisotropic."""
    rng = np.random.default_rng(seed)
    jnts, nq, nv, nu = ref.joints(model), model.nq, model.nv, model.nu
    qs = random_states(model, name, n * (T + 1), seed=seed)[0].reshape(n, T + 1, nq)
    qr = np.array(qs)
    for typ, pa, _ in jnts:
        if typ == ref.JNT_FREE:
            qs[:, :, pa:pa + 3] += rng.normal(0, 0.5, (n, T + 1, 3))
            for e in range(n):
                qr[e] = ref.random_rotation_errors(rng, jnts, qs[e], max_angle)
        else:
            qs[:, :, pa] += rng.normal(0, 0.3, (n, T + 1))
    vs, vr = rng.normal(size=(n, T + 1, nv)), rng.normal(size=(n, T + 1, nv))
    us, ur = rng.normal(size=(n, T, nu)), rng.normal(size=(n, T, nu))
    Q, R, Qf = ref.random_spd(rng, 2 * nv), ref.random_spd(rng, nu), ref.random_spd(rng, 2 * nv, 30.0)
    return jnts, (qs, vs, us, qr, vr, ur), (Q, R, Qf)


def _dev(x, dtype):
    import torch

    return torch.as_tensor(np.ascontiguousarray(x), device="cuda", dtype=dtype)


def _env_fastest(x, dtype):
    """(N, ...) host array -> CUDA view of env-fastest storage, as linearize_rollout returns them."""
    x = np.asarray(x)
    return _dev(np.moveaxis(x, 0, -1), dtype).permute(x.ndim - 1, *range(x.ndim - 1))


def _reference(jnts, nv, traj, W, e, exact=True, cast=None):
    parts = [None if t is None else (t[e] if cast is None else t[e].astype(cast).astype(float)) for t in traj]
    return ref.traj_cost(jnts, nv, *parts, *W, exact=exact)


CASES = [("pendulum", 64), ("cartpole", 64), ("drone", 64), ("humanoid", 64), ("humanoid-lane", 64),
         ("pendulum", 32), ("cartpole", 32), ("drone", 32), ("humanoid", 32)]


@pytest.mark.parametrize("case,prec", CASES)
def test_traj_cost_matches_reference(monkeypatch, case, prec):
    import torch

    import mujoco_template as mt

    model, name = _model(monkeypatch, case)
    n, T = (6, 5) if name == "humanoid" else (37, 9)  # n not a multiple of a block's 32 envs
    env = mt.BatchedEnv(model, n, precision=prec)
    dtype = env.data.qpos.dtype
    jnts, traj, W = _problem(model, name, n, T, seed=11)
    qs, vs, us, qr, vr, ur = traj
    J, q, r = env.traj_cost(_env_fastest(qs, dtype), _env_fastest(vs, dtype), _env_fastest(us, dtype), *W, qpos_ref=_env_fastest(qr, dtype),
                            qvel_ref=_env_fastest(vr, dtype), ctrl_ref=_env_fastest(ur, dtype), grad=True)
    J, q, r = (t.double().cpu().numpy() for t in (J, q, r))
    cast = np.float32 if prec == 32 else None
    worst = worst_naive = 0.0
    for e in range(n):
        Jr, qr_, rr = _reference(jnts, model.nv, traj, W, e, cast=cast)
        err = max(abs(J[e] - Jr) / max(1.0, abs(Jr)), _rel(q[e], qr_), _rel(r[e], rr))
        assert err <= COST_RTOL[prec], (case, prec, e, err)
        worst = max(worst, err)
        worst_naive = max(worst_naive, _rel(q[e], _reference(jnts, model.nv, traj, W, e, exact=False, cast=cast)[1]))
    variant = env.data.backend.batch.kernel_variant
    print(f"MEASURED traj_cost vs reference {case} fp{prec} ({variant}): {worst:.2e}; with G = I: {worst_naive:.2e}")
    if name in ("drone", "humanoid"):  # a kernel without Jr^-1 would fail by far
        assert worst_naive > 100 * COST_RTOL[prec], (case, worst_naive)


@pytest.mark.parametrize("case", ["drone", "humanoid"])
def test_every_null_combination_of_references_and_outputs(monkeypatch, case):
    import itertools

    import torch

    import mujoco_template as mt

    model, name = _model(monkeypatch, case)
    n, T = 40, 6
    env = mt.BatchedEnv(model, n)
    b = env.data.backend
    jnts, traj, W = _problem(model, name, n, T, seed=12)
    qs, vs, us, qr, vr, ur = (_dev(np.moveaxis(t, 0, -1), torch.float64) for t in traj)
    Wf = [M.reshape(-1) for M in W]
    zero_v, zero_u = torch.zeros_like(vr), torch.zeros_like(ur)
    full = b.traj_cost(qs, vs, us, qr, vr, ur, *Wf, T, True)
    for use_v, use_u in itertools.product((False, True), repeat=2):
        got = b.traj_cost(qs, vs, us, qr, vr if use_v else None, ur if use_u else None, *Wf, T, True)
        want = b.traj_cost(qs, vs, us, qr, vr if use_v else zero_v, ur if use_u else zero_u, *Wf, T, True)
        for g, w in zip(got, want):
            assert torch.equal(g, w), (use_v, use_u)
    for mask in itertools.product((False, True), repeat=3):
        if not any(mask):
            continue
        out = tuple(torch.full_like(t, 7.0) if m else None for t, m in zip(full, mask))
        b.traj_cost(qs, vs, us, qr, vr, ur, *Wf, T, True, out=out)
        for t, f in zip(out, full):
            if t is not None:
                assert torch.equal(t, f), mask


def test_batch_dependent_rejections():
    import torch

    from mujoco_template import _capi
    from mujoco_template import _mj as mj

    model = load_model("cartpole")
    data = mj.BatchData(model, 4)
    b = data.backend
    T = 3
    q = torch.zeros((T + 1, 2, 4), dtype=torch.float64, device="cuda")
    u = torch.zeros((T, 1, 4), dtype=torch.float64, device="cuda")
    Q = np.eye(4)
    Q[0, 1] = 1e-3  # not symmetric
    for Qb, Rb, Qfb, msg in ((Q, np.eye(1), np.eye(4), "Q is not"), (np.eye(4), np.eye(1), Q, "Qf is not")):
        with pytest.raises(_capi.TemplateError, match=msg):
            b.traj_cost(q, q, u, q, None, None, Qb.reshape(-1), Rb.reshape(-1), Qfb.reshape(-1), T, False)
    R2 = np.array([[1.0, 0.5], [0.4, 1.0]])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        two = mj.MjModel.from_xml_string(
            '<mujoco><worldbody><body><joint name="a" type="hinge" axis="0 1 0"/><joint name="b" type="hinge" axis="1 0 0"/>'
            '<geom type="sphere" size="0.1" mass="1"/></body></worldbody><actuator><motor joint="a"/><motor joint="b"/></actuator></mujoco>')
        bare = mj.MjModel.from_xml_string('<mujoco><worldbody><body><joint type="hinge" axis="0 1 0"/><geom type="sphere" size="0.1" mass="1"/>'
                                          '</body></worldbody></mujoco>')
    d2 = mj.BatchData(two, 4)
    q2, u2 = torch.zeros((T + 1, 2, 4), dtype=torch.float64, device="cuda"), torch.zeros((T, 2, 4), dtype=torch.float64, device="cuda")
    with pytest.raises(_capi.TemplateError, match="R is not"):
        d2.backend.traj_cost(q2, q2, u2, q2, None, None, np.eye(4).reshape(-1), R2.reshape(-1), np.eye(4).reshape(-1), T, False)
    d0 = mj.BatchData(bare, 4)
    lib = _capi.lib()
    p = q.data_ptr()
    W = (C.c_double * 16)(*np.eye(4).reshape(-1))
    rc = lib.b2_traj_cost(d0.backend.batch.handle, T, p, p, p, p, None, None, W, W, W, p, None, None, None)
    assert rc == -1 and b"no actuators" in lib.b2_last_error()


@pytest.mark.parametrize("case", ["drone", "humanoid"])
def test_gradient_matches_central_differences_through_integrate_pos(monkeypatch, case):
    """J(xbar (+) h d, u + h du), with (+) b2_integrate_pos on the device: halving h quarters the residual of the central
    difference against sum q'd + r'du, so q is the gradient in the tangent space of A and rollout_feedback."""
    import torch

    import mujoco_template as mt

    model, name = _model(monkeypatch, case)
    n, T = 32, 8
    env = mt.BatchedEnv(model, n)
    b = env.data.backend
    jnts, traj, W = _problem(model, name, n, T, seed=13, max_angle=2.0)
    qs, vs, us, qr, vr, ur = (_dev(np.moveaxis(t, 0, -1), torch.float64) for t in traj)
    Wf = [M.reshape(-1) for M in W]
    rng = np.random.default_rng(14)
    d = _dev(rng.normal(size=(T + 1, 2 * model.nv, n)), torch.float64)
    du = _dev(rng.normal(size=(T, model.nu, n)), torch.float64)
    J0, q, r = b.traj_cost(qs, vs, us, qr, vr, ur, *Wf, T, True)
    analytic = (q * d).sum((0, 1)) + (r * du).sum((0, 1))

    def J_at(h):
        qp = qs.clone()
        for t in range(T + 1):
            dq = d[t, : model.nv].contiguous()
            b._pre()
            b.batch.integrate_pos(qp[t].data_ptr(), dq.data_ptr(), h, b.stream)
        return b.traj_cost(qp, vs + h * d[:, model.nv:], us + h * du, qr, vr, ur, *Wf, T, False)[0]

    res = []
    for h in (1e-3, 5e-4):
        fd = (J_at(h) - J_at(-h)) / (2 * h)
        res.append(float(((fd - analytic).abs() / analytic.abs().clamp(min=1.0)).max()))
    ratio = res[0] / res[1]
    print(f"MEASURED central-difference residual {case}: {res[0]:.2e} -> {res[1]:.2e}, ratio {ratio:.2f}")
    assert 3.5 <= ratio <= 4.5, res


@pytest.mark.parametrize("case", ["cartpole", "humanoid"])
def test_nan_rows_reach_only_their_env(monkeypatch, case):
    import torch

    import mujoco_template as mt

    model, name = _model(monkeypatch, case)
    n, T = 40, 5
    env = mt.BatchedEnv(model, n)
    b = env.data.backend
    jnts, traj, W = _problem(model, name, n, T, seed=15)
    qs, vs, us, qr, vr, ur = (_dev(np.moveaxis(t, 0, -1), torch.float64) for t in traj)
    Wf = [M.reshape(-1) for M in W]
    clean = b.traj_cost(qs, vs, us, qr, vr, ur, *Wf, T, True)
    qs[2, 0, 3] = float("nan")    # a state row of env 3
    us[T - 1, 0, 5] = float("nan")  # the last control row of env 5 (a frozen env of rollout_feedback)
    J, q, r = b.traj_cost(qs, vs, us, qr, vr, ur, *Wf, T, True)
    assert bool(torch.isnan(J[3])) and bool(torch.isnan(J[5]))
    assert bool(torch.isnan(q[2, :, 3]).any()) and bool(torch.isnan(r[T - 1, :, 5]).all())
    others = [e for e in range(n) if e not in (3, 5)]
    assert torch.equal(J[others], clean[0][others]) and torch.equal(q[..., others], clean[1][..., others])
    assert torch.equal(r[..., others], clean[2][..., others])
    assert bool(torch.isfinite(q[:, :, 5]).all())  # env 5's states are clean


@pytest.mark.parametrize("case", ["drone", "humanoid"])
def test_one_launch_graph_replay_and_repeatability(monkeypatch, case):
    import torch

    import mujoco_template as mt
    from mujoco_template import _capi

    model, name = _model(monkeypatch, case)
    n, T = 64, 7
    env = mt.BatchedEnv(model, n)
    b = env.data.backend
    jnts, traj, W = _problem(model, name, n, T, seed=16)
    qs, vs, us, qr, vr, ur = (_dev(np.moveaxis(t, 0, -1), torch.float64) for t in traj)
    Wf = [M.reshape(-1) for M in W]
    eager = b.traj_cost(qs, vs, us, qr, vr, ur, *Wf, T, True)
    torch.cuda.synchronize()
    c0 = _capi.launch_count()
    again = b.traj_cost(qs, vs, us, qr, vr, ur, *Wf, T, True)
    assert _capi.launch_count() - c0 == 1, b.batch.kernel_variant
    for a, e in zip(again, eager):
        assert torch.equal(a, e)  # J bit-identical from run to run
    out = tuple(torch.empty_like(t) for t in eager)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        b.traj_cost(qs, vs, us, qr, vr, ur, *Wf, T, True, out=out)
    g.replay()
    torch.cuda.synchronize()
    for a, e in zip(out, eager):
        assert torch.equal(a, e)


def test_outputs_beyond_2_31_elements():
    import torch

    from mujoco_template import _mj as mj

    model = load_model("pendulum")
    n, T = (1 << 24) + 96, 64  # q: (T+1) 2nv n > 2^31 elements
    data = mj.BatchData(model, n, precision=32)
    b = data.backend
    g = torch.Generator(device="cuda").manual_seed(0)
    mk = lambda *s: torch.randn(s, device="cuda", dtype=torch.float32, generator=g)  # noqa: E731
    qs, vs, qr, us = mk(T + 1, 1, n), mk(T + 1, 1, n), mk(T + 1, 1, n), mk(T, 1, n)
    Q, R, Qf = np.array([[2.0, 0.3], [0.3, 1.0]]), np.eye(1) * 0.5, np.array([[5.0, 1.0], [1.0, 3.0]])
    J, q, r = b.traj_cost(qs, vs, us, qr, None, None, Q.reshape(-1), R.reshape(-1), Qf.reshape(-1), T, True)
    assert q.numel() > 2 ** 31
    jnts = ref.joints(model)
    worst = 0.0
    for e in (0, n // 2, n - 1):
        host = [t[..., e].double().cpu().numpy() for t in (qs, vs, us, qr)]
        Jr, qr_, rr = ref.traj_cost(jnts, 1, host[0], host[1], host[2], host[3], None, None, Q, R, Qf)
        err = max(abs(float(J[e]) - Jr) / max(1.0, abs(Jr)), _rel(q[..., e].double().cpu(), qr_), _rel(r[..., e].double().cpu(), rr))
        worst = max(worst, err)
    print(f"MEASURED traj_cost beyond 2^31 elements: {worst:.2e}")
    assert worst <= COST_RTOL[32], worst
    del qs, vs, qr, us, J, q, r


# ---------------------------------------------------------------- the four iLQR calls together

def _drone_hover(model):
    """Per-rotor thrust that holds the drone's weight."""
    return float(np.sum(model.body_mass) * 9.81 / model.nu)


def _setup(name, n, prec=64, seed=0):
    import torch

    import mujoco_template as mt

    model = load_model(name)
    env = mt.BatchedEnv(model, n, precision=prec)
    d = env.data
    dev, dt = d.qpos.device, d.qpos.dtype
    rng = np.random.default_rng(seed)
    if name == "pendulum":
        d.qpos.copy_(torch.as_tensor(rng.uniform(-0.3, 0.3, (1, n)), device=dev, dtype=dt)); d.qvel.zero_()
        W = (np.diag([1.0, 0.1]), np.eye(1) * 0.01, np.diag([100.0, 10.0]))
        refs = dict(qpos_ref=torch.tensor([np.pi], device=dev, dtype=dt))
    else:  # the drone in free flight, well above the floor, towards a pose yawed by 90 degrees
        q0 = np.tile(model.key_qpos[0], (n, 1))
        q0[:, 2] = 2.0
        q0[:, :2] += rng.uniform(-0.1, 0.1, (n, 2))
        d.qpos.copy_(torch.as_tensor(q0.T.copy(), device=dev, dtype=dt)); d.qvel.zero_()
        goal = np.array([0.3, -0.2, 2.3, np.cos(np.pi / 4), 0.0, 0.0, np.sin(np.pi / 4)])
        W = (np.diag([10.0, 10.0, 10.0, 2.0, 3.0, 5.0, 1.0, 1.0, 1.0, 0.5, 0.5, 0.5]), np.eye(4) * 0.01,
             np.diag([100.0, 100.0, 100.0, 20.0, 30.0, 50.0, 10.0, 10.0, 10.0, 5.0, 5.0, 5.0]))
        refs = dict(qpos_ref=torch.as_tensor(goal, device=dev, dtype=dt))
    return model, env, W, refs


@pytest.mark.parametrize("name", ["pendulum", "drone"])
def test_first_order_consistency_of_the_four_calls(name):
    """linearize_rollout -> traj_cost -> batched_tvlqr -> rollout_feedback: (J(alpha) - J) / (alpha dV[0]) -> 1 with an
    error that halves with alpha (nominal controls away from ctrlrange bounds, where the clip is smooth)."""
    import torch

    from mujoco_template.batched_controllers import batched_tvlqr

    n, T = 16, 40
    model, env, (Q, R, Qf), refs = _setup(name, n, seed=1)
    d = env.data
    rng = np.random.default_rng(2)
    base = _drone_hover(model) if name == "drone" else 0.0
    U = torch.as_tensor(base + 0.2 * rng.normal(size=(n, T, model.nu)), device=d.qpos.device, dtype=d.qpos.dtype)
    x0 = d.qpos.clone(), d.qvel.clone()
    lin = env.linearize_rollout(U)
    J, q, r = env.traj_cost(lin["qpos"], lin["qvel"], U, Q, R, Qf, grad=True, **refs)
    K, k, _, dV, status = batched_tvlqr(lin["A"], lin["B"], Q, R, Qf, q, r, reg=1e-6)
    assert int(status.abs().max()) == 0
    errs = []
    for a in (1e-2, 5e-3, 2.5e-3):
        d.qpos.copy_(x0[0]); d.qvel.copy_(x0[1])
        rec = env.rollout_feedback(U, K, lin["qpos"], lin["qvel"], k=k, alpha=a, record=True)
        qs = torch.cat([x0[0].T[:, None], rec["qpos"]], 1)
        vs = torch.cat([x0[1].T[:, None], rec["qvel"]], 1)
        Ja = env.traj_cost(qs, vs, rec["ctrl"], Q, R, Qf, **refs)
        errs.append(float(((Ja - J) / (a * dV[:, 0]) - 1).abs().max()))
    r1, r2 = errs[0] / errs[1], errs[1] / errs[2]
    print(f"MEASURED first-order consistency {name}: {errs[0]:.2e} {errs[1]:.2e} {errs[2]:.2e} (ratios {r1:.2f}, {r2:.2f})")
    assert errs[0] <= 0.05 and 1.6 <= r1 <= 2.5 and 1.6 <= r2 <= 2.5, errs


def _state(env):
    d, b = env.data, env.data.backend
    return [b.buffers[k].clone() for k in ("qpos", "qvel", "ctrl", "qacc_warmstart", "flags")] + [d.time, env._substep]


def _same_state(a, b):
    for x, y in zip(a[:5], b[:5]):
        assert torch_equal(x, y)
    assert a[5:] == b[5:]


def torch_equal(x, y):
    import torch

    return torch.equal(x, y)


@pytest.mark.parametrize("name,prec", [("pendulum", 64), ("drone", 64), ("drone", 32)])
def test_batched_ilqr(name, prec):
    import torch

    from mujoco_template.batched_controllers import batched_ilqr

    n = 16 if name == "pendulum" else 8
    T, iters = (150, 12) if name == "pendulum" else (200, 20)  # the drone: 2 s
    model, env, (Q, R, Qf), refs = _setup(name, n, prec, seed=71)
    if name == "pendulum":  # the start of tests/test_gpu_tvlqr.py::test_ilqr_pendulum_swing_up
        env.data.qpos.copy_(torch.as_tensor(np.random.default_rng(71).uniform(-0.3, 0.3, (1, n)), device="cuda", dtype=env.data.qpos.dtype))
    base = _drone_hover(model) if name == "drone" else 0.0
    U0 = torch.full((n, T, model.nu), base, device="cuda", dtype=env.data.qpos.dtype)
    env.data.ctrl.fill_(0.5)
    before = _state(env)
    out = batched_ilqr(env, U0, Q, R, Qf, iters=iters, eps=None if prec == 64 else 1e-3, **refs)
    _same_state(_state(env), before)
    H = out["J_history"]
    assert bool((H[1:] <= H[:-1]).all()), H  # an env's J never increases
    assert torch.equal(out["J"], H[-1])
    frac = float((out["J"] / H[0]).max())
    # the returned trajectory is that of the returned controls, and its cost is J, up to the last bits in which the
    # closed-loop rollout and the open-loop replay of its controls may differ
    lin = env.linearize_rollout(out["ctrl"], eps=None if prec == 64 else 1e-3)
    Jc = env.traj_cost(lin["qpos"], lin["qvel"], out["ctrl"], Q, R, Qf, **refs)
    replay = max(_rel(lin["qpos"].double().cpu(), out["qpos"].double().cpu()), _rel(lin["qvel"].double().cpu(), out["qvel"].double().cpu()),
                 float(((Jc - out["J"]).abs() / out["J"].abs()).max()))
    msg = f"MEASURED batched_ilqr {name} fp{prec}: worst J_final / J_0 {frac:.3e} after {H.shape[0] - 1} iterations, replay {replay:.1e}"
    pose = None
    if name == "drone":
        goal = refs["qpos_ref"].double().cpu().numpy()
        qT = out["qpos"][:, -1].double().cpu().numpy()
        err = np.array([ref.differentiate_pos(ref.joints(model), model.nv, goal, qT[e]) for e in range(n)])
        pose = float(np.abs(err[:, :3]).max()), float(np.abs(err[:, 3:]).max())
        msg += f"; final pose error {pose[0]:.3f} m, {pose[1]:.3f} rad"
    print(msg)
    assert replay <= (1e-13 if prec == 64 else 3e-5), replay  # measured 5.6e-15 / 2.5e-6 (the drone)
    assert frac <= (0.45 if name == "pendulum" else 0.3), frac  # measured 0.387 (the bound of test_gpu_tvlqr.py) and 0.213
    assert pose is None or (pose[0] <= 0.05 and pose[1] <= 0.05), pose  # measured 0.013 m, 0.009 rad
    assert int(out["status"].abs().max()) == 0
