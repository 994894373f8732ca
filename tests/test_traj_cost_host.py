"""b2_traj_cost / BatchedEnv.traj_cost without a GPU: the C-ABI rejects bad arguments before it needs a device, and
BatchedEnv.traj_cost validates its inputs, lays out trajectories and references env fastest and moves neither time nor
state.  (The rejections that need a batch -- a model without actuators, a weight that is not symmetric -- are in
tests/test_gpu_traj_cost.py.)"""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import load_model

ERR_ARG = -1


def test_b2_traj_cost_rejects_bad_arguments():
    from mujoco_template import _capi

    lib = _capi.lib()
    buf = (C.c_double * 64)()
    p = C.cast(buf, C.c_void_p).value
    W = C.cast(buf, C.POINTER(C.c_double))

    def call(nsteps=4, qpos=p, qvel=p, ctrl=p, qref=p, Q=W, R=W, Qf=W, J=p, q=p, r=p):
        return lib.b2_traj_cost(None, nsteps, qpos, qvel, ctrl, qref, None, None, Q, R, Qf, J, q, r, None)

    cases = [
        (dict(nsteps=0), b"nsteps"),
        (dict(nsteps=-3), b"nsteps"),
        (dict(qpos=None), b"required"),
        (dict(qvel=None), b"required"),
        (dict(ctrl=None), b"required"),
        (dict(qref=None), b"required"),
        (dict(Q=None), b"required"),
        (dict(R=None), b"required"),
        (dict(Qf=None), b"required"),
        (dict(J=None, q=None, r=None), b"all NULL"),
        (dict(), b"null batch"),  # valid arguments, no batch
        (dict(J=None, q=None), b"null batch"),  # one output is enough
    ]
    for kw, msg in cases:
        assert call(**kw) == ERR_ARG, kw
        err = lib.b2_last_error()
        assert b"b2_traj_cost" in err and msg in err, (kw, err)


class _Backend:
    """Stands in for NativeBackend: records what BatchedEnv.traj_cost hands to the library."""

    def __init__(self, model, nenv):
        self.calls = []
        self.model, self.nenv = model, nenv

    def traj_cost(self, qpos, qvel, ctrl, qref, vref, uref, Q, R, Qf, nsteps, grad):
        self.calls.append(dict(qpos=qpos, qvel=qvel, ctrl=ctrl, qref=qref, vref=vref, uref=uref, Q=Q, R=R, Qf=Qf, nsteps=nsteps, grad=grad))
        m, n, T = self.model, self.nenv, nsteps
        J = torch.arange(n, dtype=torch.float64)
        if not grad:
            return J, None, None
        return J, torch.zeros((T + 1, 2 * m.nv, n), dtype=torch.float64), torch.zeros((T, m.nu, n), dtype=torch.float64)


class _Data:
    def __init__(self, model, nenv):
        self.nenv, self.time = nenv, 0.0
        self.qpos = torch.zeros((model.nq, nenv), dtype=torch.float64)
        self.backend = _Backend(model, nenv)


def _env(name, nenv=5):
    import mujoco_template as mt

    model = load_model(name)
    return mt.BatchedEnv(model, nenv, data=_Data(model, nenv)), model


def _traj(model, n, T):
    """linearize_rollout-style views of env-fastest storage, and a (nenv, T, nu) control tensor."""
    q = torch.randn(T + 1, model.nq, n, dtype=torch.float64)
    v = torch.randn(T + 1, model.nv, n, dtype=torch.float64)
    u = torch.randn(T, model.nu, n, dtype=torch.float64)
    return q, v, u, q.permute(2, 0, 1), v.permute(2, 0, 1), u.permute(2, 0, 1)


def test_batched_traj_cost_hands_over_trajectories_without_a_copy_and_moves_nothing():
    env, model = _env("drone")
    be = env.data.backend
    n, T, nx = 5, 6, 2 * model.nv
    q, v, u, qv, vv, uv = _traj(model, n, T)
    Q, R = np.diag(np.arange(1.0, nx + 1)), np.eye(model.nu)
    qref = torch.randn(n, T + 1, model.nq, dtype=torch.float64)
    J = env.traj_cost(qv, vv, uv, Q, R, qpos_ref=qref)
    c = be.calls[-1]
    assert c["qpos"].data_ptr() == q.data_ptr() and c["qvel"].data_ptr() == v.data_ptr() and c["ctrl"].data_ptr() == u.data_ptr()
    assert torch.equal(c["qref"], qref.permute(1, 2, 0)) and c["vref"] is None and c["uref"] is None
    assert c["nsteps"] == T and c["grad"] is False and J.shape == (n,)
    assert np.array_equal(c["Q"], Q.reshape(-1)) and np.array_equal(c["Qf"], Q.reshape(-1)) and np.array_equal(c["R"], R.reshape(-1))
    J, gq, gr = env.traj_cost(qv, vv, uv, Q, R, 2 * Q, qpos_ref=qref, grad=True)
    assert be.calls[-1]["grad"] is True and np.array_equal(be.calls[-1]["Qf"], 2 * Q.reshape(-1))
    assert gq.shape == (n, T + 1, nx) and gr.shape == (n, T, model.nu)
    assert env.data.time == 0.0 and env._substep == 0


def test_batched_traj_cost_broadcasts_references_env_fastest():
    env, model = _env("cartpole", 4)
    be = env.data.backend
    n, T = 4, 3
    _, _, _, qv, vv, uv = _traj(model, n, T)
    Q, R = np.eye(4), np.eye(1)
    per_step = torch.randn(T + 1, model.nq, dtype=torch.float64)
    const_v = torch.randn(model.nv, dtype=torch.float64)
    per_env_u = torch.randn(n, T, model.nu, dtype=torch.float64)
    env.traj_cost(qv, vv, uv, Q, R, qpos_ref=per_step, qvel_ref=const_v, ctrl_ref=per_env_u)
    c = be.calls[-1]
    assert c["qref"].shape == (T + 1, model.nq, n) and c["qref"].is_contiguous()
    assert torch.equal(c["qref"], per_step[:, :, None].expand(T + 1, model.nq, n))
    assert c["vref"].shape == (T + 1, model.nv, n) and c["vref"].is_contiguous()
    assert torch.equal(c["vref"], const_v[None, :, None].expand(T + 1, model.nv, n))
    assert torch.equal(c["uref"], per_env_u.permute(1, 2, 0))
    env.traj_cost(qv, vv, uv, Q, R, qpos_ref=torch.zeros(model.nq, dtype=torch.float64), ctrl_ref=torch.ones(T, model.nu, dtype=torch.float64))
    assert torch.equal(be.calls[-1]["uref"], torch.ones(T, model.nu, n, dtype=torch.float64))


def test_batched_traj_cost_validates_inputs():
    from mujoco_template.exceptions import ConfigError

    env, model = _env("cartpole", 4)
    be = env.data.backend
    n, T = 4, 3
    _, _, _, qv, vv, uv = _traj(model, n, T)
    Q, R = np.eye(4), np.eye(1)
    qref = torch.zeros(model.nq, dtype=torch.float64)
    bad = [
        dict(qpos=qv[:, :T]), dict(qvel=vv[:3]), dict(ctrl=uv[..., :0].expand(n, T, 0)), dict(ctrl=uv.float()), dict(ctrl=uv.numpy()),
        dict(ctrl=uv[:, :0]), dict(qpos=qv.float()), dict(Q=np.eye(3)), dict(R=np.eye(2)), dict(Qf=np.eye(5)),
        dict(qpos_ref=None), dict(qpos_ref=torch.zeros(T, model.nq, dtype=torch.float64)), dict(qpos_ref=qref.float()),
        dict(qvel_ref=torch.zeros(n, T, model.nv, dtype=torch.float64)), dict(ctrl_ref=torch.zeros(T + 1, model.nu, dtype=torch.float64)),
        dict(ctrl_ref=torch.zeros(3, dtype=torch.float64)),
    ]
    for kw in bad:
        args = dict(qpos=qv, qvel=vv, ctrl=uv, Q=Q, R=R, Qf=None, qpos_ref=qref)
        args.update(kw)
        with pytest.raises(ConfigError, match="traj_cost"):
            env.traj_cost(args.pop("qpos"), args.pop("qvel"), args.pop("ctrl"), args.pop("Q"), args.pop("R"), args.pop("Qf"), **args)
    assert be.calls == []


def test_batched_traj_cost_rejects_a_model_without_actuators():
    from mujoco_template.exceptions import ConfigError

    env, model = _env("cartpole", 2)
    env.model = type("M", (), {"nu": 0, "nq": model.nq, "nv": model.nv})()
    with pytest.raises(ConfigError, match="no actuators"):
        env.traj_cost(None, None, None, np.eye(4), np.eye(1), qpos_ref=None)
