"""b2_linearize_rollout / BatchedEnv.linearize_rollout without a GPU: the C-ABI rejects bad arguments, and
BatchedEnv.linearize_rollout validates its inputs, lays out the controls and moves neither time nor state."""
import ctypes as C

import pytest
import torch

from conftest import load_model

ERR_ARG, ERR_LINEARIZE = -1, -5


def test_b2_linearize_rollout_rejects_bad_arguments():
    from mujoco_template import _capi

    lib = _capi.lib()
    buf = (C.c_double * 8)()
    p = C.cast(buf, C.c_void_p).value
    st = _capi.State(p, p, p, None, None)
    st_warm = _capi.State(p, p, p, p, None)
    call = lambda state, nsteps, eps, A, q, v, w=None: lib.b2_linearize_rollout(  # noqa: E731
        None, C.byref(state), nsteps, None, eps, 1, A, None, None, None, q, v, w, None, None)
    cases = [
        ((st, 0, 1e-6, p, p, p), ERR_ARG, b"nsteps"),
        ((st, -2, 1e-6, p, p, p), ERR_ARG, b"nsteps"),
        ((st, 4, 1e-6, p, None, p), ERR_ARG, b"qpos_traj"),
        ((st, 4, 1e-6, p, p, None), ERR_ARG, b"qvel_traj"),
        ((st_warm, 4, 1e-6, p, p, p), ERR_ARG, b"warm_traj"),
        ((st, 4, 1e-6, None, p, p), ERR_ARG, b"all NULL"),
        ((st, 4, 0.0, p, p, p), ERR_LINEARIZE, b"eps"),
        ((st, 4, -1e-6, p, p, p), ERR_LINEARIZE, b"eps"),
        ((st, 4, 1e-6, p, p, p), ERR_ARG, b"null batch"),  # valid arguments, no batch
        ((st_warm, 4, 1e-6, p, p, p, p), ERR_ARG, b"null batch"),
    ]
    for args, code, msg in cases:
        assert call(*args) == code, args
        err = lib.b2_last_error()
        assert b"b2_linearize_rollout" in err and msg in err, (args, err)


class _Backend:
    """Stands in for NativeBackend: records what BatchedEnv.linearize_rollout hands to the library."""

    def __init__(self, model, nenv):
        self.calls = []
        self.model, self.nenv = model, nenv

    def linearize_rollout(self, seq, nsteps, eps, centered, sensors):
        self.calls.append((seq, nsteps, eps, centered, sensors))
        m, n, T = self.model, self.nenv, nsteps
        nx, ns = 2 * m.nv, m.nsensordata
        mk = lambda *shape: torch.zeros(shape + (n,), dtype=torch.float64)  # noqa: E731
        sens = sensors and ns > 0
        return (mk(T, nx, nx), mk(T, nx, m.nu), mk(T, ns, nx) if sens else None, mk(T, ns, m.nu) if sens else None,
                mk(T + 1, m.nq), mk(T + 1, m.nv), mk(T + 1, m.nv), mk(T, ns) if sens else None)


class _Data:
    def __init__(self, model, nenv):
        self.nenv, self.time = nenv, 0.0
        self.qpos = torch.zeros((model.nq, nenv), dtype=torch.float64)
        self.backend = _Backend(model, nenv)


def _env(name, nenv=5):
    import mujoco_template as mt

    model = load_model(name)
    return mt.BatchedEnv(model, nenv, data=_Data(model, nenv)), model


def test_batched_linearize_rollout_validates_inputs_and_lays_out_controls():
    from mujoco_template.exceptions import ConfigError

    env, model = _env("cartpole")
    be = env.data.backend
    T = 7
    U = torch.randn(5, T, model.nu, dtype=torch.float64)
    for bad in (torch.randn(4, T, 1, dtype=torch.float64), torch.randn(5, T, 2, dtype=torch.float64), torch.randn(5, T, dtype=torch.float64),
                U.float(), U.numpy(), torch.randn(5, 0, 1, dtype=torch.float64)):
        with pytest.raises(ConfigError, match="linearize_rollout|nsteps"):
            env.linearize_rollout(bad)
    with pytest.raises(ConfigError, match="disagrees"):
        env.linearize_rollout(U, T + 1)
    for n in (None, 0, -1):
        with pytest.raises(ConfigError):
            env.linearize_rollout(nsteps=n)
    assert be.calls == []
    # handed over as (T, nu, nenv) -- without a copy when the controls already are a view of such a buffer
    buf = torch.randn(T, model.nu, 5, dtype=torch.float64)
    out = env.linearize_rollout(buf.permute(2, 0, 1))
    seq, nsteps, eps, centered, sensors = be.calls[-1]
    assert seq.data_ptr() == buf.data_ptr() and torch.equal(seq, buf)
    assert (nsteps, eps, centered, sensors) == (T, env.lin_eps, True, False)
    env.linearize_rollout(U, T, eps=1e-4, centered=False)
    assert torch.equal(be.calls[-1][0], U.permute(1, 2, 0)) and be.calls[-1][1:4] == (T, 1e-4, False)
    nx = 2 * model.nv
    assert set(out) == {"qpos", "qvel", "A", "B"}
    assert out["qpos"].shape == (5, T + 1, model.nq) and out["qvel"].shape == (5, T + 1, model.nv)
    assert out["A"].shape == (5, T, nx, nx) and out["B"].shape == (5, T, nx, model.nu)
    # held controls
    env.linearize_rollout(nsteps=3)
    assert be.calls[-1][0] is None and be.calls[-1][1] == 3
    # neither time nor the control-decimation counter moves
    assert env.data.time == 0.0 and env._substep == 0


def test_batched_linearize_rollout_sensor_outputs():
    env, model = _env("drone", 3)
    out = env.linearize_rollout(nsteps=4, sensors=True)
    nx, ns = 2 * model.nv, model.nsensordata
    assert out["C"].shape == (3, 4, ns, nx) and out["D"].shape == (3, 4, ns, model.nu) and out["sensordata"].shape == (3, 4, ns)
    assert set(env.linearize_rollout(nsteps=4)) == {"qpos", "qvel", "A", "B"}
    env, model = _env("pendulum", 3)
    assert model.nsensordata == 0 and set(env.linearize_rollout(nsteps=2, sensors=True)) == {"qpos", "qvel", "A", "B"}
