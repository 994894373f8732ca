"""The NumPy reference of b2_tvlqr's backward pass (tests/tvlqr_reference.py) pinned on the CPU: against scipy's DARE, the
dense least-squares minimiser and the exact cost change; plus the argument checks of b2_tvlqr / b2_rollout_feedback in
the C-ABI and of their Python front ends, none of which needs a GPU."""
import ctypes as C

import numpy as np
import pytest
import scipy.linalg
import torch

import tvlqr_reference as ref
from conftest import load_model

ERR_ARG = -1


@pytest.mark.parametrize("nx,nu", [(2, 1), (4, 1), (4, 2), (12, 4)])
def test_constant_system_long_horizon_is_the_dare(nx, nu):
    rng = np.random.default_rng(nx * 10 + nu)
    A0 = np.eye(nx) + 0.1 * rng.normal(size=(nx, nx))
    B0 = rng.normal(size=(nx, nu))
    Q, R = np.eye(nx), np.eye(nu)
    T = 600
    K, _, P0, _, status = ref.tvlqr(np.repeat(A0[None], T, 0), np.repeat(B0[None], T, 0), Q, R)
    P = scipy.linalg.solve_discrete_are(A0, B0, Q, R)
    Kd = np.linalg.solve(R + B0.T @ P @ B0, B0.T @ P @ A0)
    assert status == 0
    assert np.max(np.abs(P0 - P)) <= 1e-9 * np.max(np.abs(P))
    assert np.max(np.abs(K[0] - Kd)) <= 1e-9 * max(1.0, np.max(np.abs(Kd)))


@pytest.mark.parametrize("nx,nu,T", [(2, 1, 5), (4, 2, 12), (6, 3, 20)])
def test_feedback_policy_is_the_dense_least_squares_minimiser(nx, nu, T):
    rng = np.random.default_rng(T)
    A, B, Q, R, Qf, q, r = ref.random_system(rng, T, nx, nu)
    x0 = rng.normal(size=nx)
    K, k, P0, dV, status = ref.tvlqr(A, B, Q, R, Qf, q, r)
    assert status == 0
    xs, us = ref.rollout_linear(A, B, x0, K, k)
    u_star = ref.dense_minimiser(A, B, x0, Q, R, Qf, q, r)
    assert np.max(np.abs(us - u_star)) <= 1e-10 * max(1.0, np.max(np.abs(u_star)))
    # the optimal cost is the value function at x0: 1/2 x0'P0 x0 + s0'x0 + dV0 + dV1 (s0 not returned: use J itself)
    J = ref.cost(xs, us, Q, R, Qf, q, r)
    assert J <= ref.cost(*ref.rollout_linear(A, B, x0, K, k, 0.9), Q, R, Qf, q, r)


@pytest.mark.parametrize("alpha", [0.0, 0.25, 0.5, 1.0, 1.7])
def test_expected_cost_change_is_exact_for_a_linear_system(alpha):
    rng = np.random.default_rng(3)
    A, B, Q, R, Qf, q, r = ref.random_system(rng, 15, 5, 2)
    # exact for reg = 0: then K'Quu k = Qux'k, and the cost-to-go of the policy is linear-quadratic in alpha
    K, k, _, dV, _ = ref.tvlqr(A, B, Q, R, Qf, q, r)
    xs, us = ref.rollout_linear(A, B, np.zeros(5), K, k, alpha)
    J = ref.cost(xs, us, Q, R, Qf, q, r)  # the nominal (zero deviation) costs 0
    expect = alpha * dV[0] + alpha ** 2 * dV[1]
    assert abs(J - expect) <= 1e-10 * max(1.0, abs(expect))
    assert dV[0] < 0 and dV[1] > 0


def test_indefinite_R_gives_status_and_nan_rows():
    rng = np.random.default_rng(5)
    A, B, Q, _, Qf, q, r = ref.random_system(rng, 6, 4, 2)
    R = np.diag([1.0, -50.0])
    K, k, P0, dV, status = ref.tvlqr(A, B, Q, R, Qf, q, r)
    assert status < 0
    t = -status - 1
    assert np.all(np.isnan(K[: t + 1])) and np.all(np.isnan(k[: t + 1])) and np.all(np.isnan(P0)) and np.all(np.isnan(dV))
    assert np.all(np.isfinite(K[t + 1:]))
    K2, _, _, _, status2 = ref.tvlqr(A, B, Q, R, Qf, q, r, reg=1e4)
    assert status2 == 0 and np.all(np.isfinite(K2))


def test_b2_tvlqr_rejects_bad_arguments():
    from mujoco_template import _capi

    lib = _capi.lib()
    buf = (C.c_double * 16)()
    p = C.cast(buf, C.c_void_p).value
    w = (C.c_double * 16)(*([1.0] * 16))

    def call(nsteps=2, nx=2, nu=1, nenv=4, precision=64, A=p, B=p, Q=w, R=w, Qf=w, K=p, reg=0.0):
        return lib.b2_tvlqr(0, precision, nsteps, nx, nu, nenv, A, B, Q, R, Qf, None, None, reg, K, None, None, None, None, None)

    cases = [dict(nsteps=0), dict(nx=0), dict(nu=0), dict(nenv=0), dict(nsteps=-3), dict(reg=-1e-9), dict(reg=float("nan")),
             dict(precision=16), dict(A=None), dict(B=None), dict(Q=None), dict(R=None), dict(Qf=None), dict(K=None)]
    for kw in cases:
        assert call(**kw) == ERR_ARG, kw
        assert b"b2_tvlqr" in lib.b2_last_error(), kw


def test_b2_rollout_feedback_rejects_bad_arguments():
    from mujoco_template import _capi

    lib = _capi.lib()
    buf = (C.c_double * 8)()
    p = C.cast(buf, C.c_void_p).value
    st = _capi.State(p, p, p, None, None)

    def call(nsteps=4, u=p, q=p, v=p, K=p):
        return lib.b2_rollout_feedback(None, C.byref(st), nsteps, u, q, v, K, None, None, None, None, None, None, None, None)

    for kw, msg in ((dict(nsteps=0), b"nsteps"), (dict(nsteps=-1), b"nsteps"), (dict(u=None), b"required"), (dict(q=None), b"required"),
                    (dict(v=None), b"required"), (dict(K=None), b"required"), ({}, b"null batch")):
        assert call(**kw) == ERR_ARG, kw
        err = lib.b2_last_error()
        assert b"b2_rollout_feedback" in err and msg in err, (kw, err)


def test_batched_tvlqr_rejects_host_tensors_and_non_tensors():
    from mujoco_template.batched_controllers import batched_tvlqr
    from mujoco_template.exceptions import ConfigError, TemplateError

    A, B = torch.zeros(3, 5, 4, 4, dtype=torch.float64), torch.zeros(3, 5, 4, 1, dtype=torch.float64)
    with pytest.raises(TemplateError):
        batched_tvlqr(A, B, np.eye(4), np.eye(1))
    with pytest.raises(ConfigError):
        batched_tvlqr(A.numpy(), B, np.eye(4), np.eye(1))


class _Backend:
    """Stands in for NativeBackend: records what BatchedEnv.rollout_feedback hands to the library."""

    def __init__(self, model, nenv):
        self.calls = []
        self.model, self.nenv = model, nenv

    def rollout_feedback(self, seq, qpos, qvel, K, k, alpha, nsteps, record):
        self.calls.append(dict(seq=seq, qpos=qpos, qvel=qvel, K=K, k=k, alpha=alpha, nsteps=nsteps, record=record))
        m, n = self.model, self.nenv
        mk = lambda dim: torch.zeros((nsteps, dim, n), dtype=torch.float64)  # noqa: E731
        return (mk(m.nu), mk(m.nq), mk(m.nv), mk(m.nsensordata) if m.nsensordata else None) if record else None


class _Data:
    def __init__(self, model, nenv):
        self.nenv, self.time = nenv, 0.0
        self.qpos = torch.zeros((model.nq, nenv), dtype=torch.float64)
        self.backend = _Backend(model, nenv)


def test_batched_rollout_feedback_validates_inputs_and_lays_out_arrays():
    import mujoco_template as mt
    from mujoco_template.exceptions import ConfigError

    model = load_model("cartpole")
    n, T, nx = 5, 7, 2 * model.nv
    env = mt.BatchedEnv(model, n, data=_Data(model, n))
    be = env.data.backend
    U = torch.randn(n, T, model.nu, dtype=torch.float64)
    # linearize_rollout's views: permuted (T+1, dim, n) buffers
    qbuf, vbuf = torch.randn(T + 1, model.nq, n, dtype=torch.float64), torch.randn(T + 1, model.nv, n, dtype=torch.float64)
    Kbuf, kbuf = torch.randn(T, model.nu, nx, n, dtype=torch.float64), torch.randn(T, model.nu, n, dtype=torch.float64)
    q, v, K, k = qbuf.permute(2, 0, 1), vbuf.permute(2, 0, 1), Kbuf.permute(3, 0, 1, 2), kbuf.permute(2, 0, 1)
    out = env.rollout_feedback(U, K, q, v, k=k, alpha=0.5, record=True)
    c = be.calls[-1]
    assert c["nsteps"] == T and c["record"]
    for name, buf in (("qpos", qbuf), ("qvel", vbuf), ("K", Kbuf), ("k", kbuf)):
        assert c[name].data_ptr() == buf.data_ptr(), name  # handed over without a copy
    assert torch.equal(c["seq"], U.permute(1, 2, 0))
    assert torch.equal(c["alpha"], torch.full((n,), 0.5, dtype=torch.float64))
    assert set(out) == {"qpos", "qvel", "ctrl"} and out["ctrl"].shape == (n, T, model.nu) and out["qpos"].shape == (n, T, model.nq)
    assert env.data.time == pytest.approx(T * model.opt.timestep) and env._substep == T
    # T rows of the nominal states work too; alpha None and a tensor; k None
    assert env.rollout_feedback(U, K, q[:, :T], v[:, :T]) is None
    assert be.calls[-1]["alpha"] is None and be.calls[-1]["k"] is None
    a = torch.rand(n, dtype=torch.float64)
    env.rollout_feedback(U, K, q, v, alpha=a)
    assert torch.equal(be.calls[-1]["alpha"], a)
    bad = [
        dict(controls=None), dict(controls=U[:, :, :0]), dict(controls=U.float()),
        dict(K=K[:, :T - 1]), dict(K=K.float()), dict(K=K[..., :nx - 1]), dict(K=K.numpy()),
        dict(qpos=q[:, :T - 1]), dict(qpos=q[:, :, :1]), dict(qvel=torch.cat([v, v], 1)), dict(qvel=v.float()),
        dict(k=k[:, :, :0]), dict(k=k.float()),
        dict(alpha=torch.ones(n + 1, dtype=torch.float64)), dict(alpha=torch.ones(n, dtype=torch.float32)),
    ]
    ncalls = len(be.calls)
    for kw in bad:
        args = dict(controls=U, K=K, qpos=q, qvel=v)
        args.update(kw)
        with pytest.raises(ConfigError):
            env.rollout_feedback(args.pop("controls"), args.pop("K"), args.pop("qpos"), args.pop("qvel"), **args)
    assert len(be.calls) == ncalls
