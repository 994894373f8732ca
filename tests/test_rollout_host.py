"""b2_rollout / BatchedEnv.rollout without a GPU: the C-ABI rejects bad arguments and never falls back to the CPU, and
BatchedEnv.rollout validates its inputs before anything reaches the device."""
import ctypes as C

import pytest
import torch

from conftest import load_model


def test_b2_rollout_rejects_bad_arguments_and_fails_loudly_without_gpu():
    from mujoco_template import _capi

    lib = _capi.lib()
    st = _capi.State()
    for nsteps in (0, -3, 5):
        assert lib.b2_rollout(None, C.byref(st), nsteps, None, None, None, None, None, None) == -1  # B2_ERR_ARG
        assert b"b2_rollout" in lib.b2_last_error()
    if not torch.cuda.is_available():
        with pytest.raises(_capi.TemplateError, match="no CUDA device"):
            _capi.NativeBatch(_capi.NativeModel(load_model("cartpole").blob), 4)


class _Backend:
    """Stands in for NativeBackend: records what BatchedEnv.rollout hands to the library."""

    def __init__(self, model, nenv):
        self.calls = []
        self.model, self.nenv = model, nenv

    def step(self, nsteps, derived=True):
        self.calls.append(("step", nsteps))

    def rollout(self, seq, nsteps, record):
        self.calls.append(("rollout", seq, nsteps, record))
        m = self.model
        mk = lambda d: torch.zeros((nsteps, d, self.nenv), dtype=torch.float64)  # noqa: E731
        return (mk(m.nq), mk(m.nv), mk(m.nsensordata) if m.nsensordata else None) if record else None


class _Data:
    def __init__(self, model, nenv):
        self.nenv, self.time = nenv, 0.0
        self.qpos = torch.zeros((model.nq, nenv), dtype=torch.float64)
        self.backend = _Backend(model, nenv)


def _env(name, nenv=5):
    import mujoco_template as mt

    model = load_model(name)
    return mt.BatchedEnv(model, nenv, data=_Data(model, nenv)), model


def test_batched_rollout_validates_inputs_and_lays_out_controls():
    from mujoco_template.exceptions import ConfigError

    env, model = _env("cartpole")
    be = env.data.backend
    T = 7
    U = torch.randn(5, T, model.nu, dtype=torch.float64)
    for bad in (torch.randn(4, T, 1, dtype=torch.float64), torch.randn(5, T, 2, dtype=torch.float64), torch.randn(5, T, dtype=torch.float64),
                U.float(), U.numpy(), torch.randn(5, 0, 1, dtype=torch.float64)):
        with pytest.raises(ConfigError):
            env.rollout(controls=bad)
    with pytest.raises(ConfigError, match="disagrees"):
        env.rollout(T + 1, controls=U)
    for n in (None, 0, -1):
        with pytest.raises(ConfigError):
            env.rollout(n)
    assert be.calls == [] and env.data.time == 0.0
    # held controls without a record: the fused step of before
    assert env.rollout(3) is None
    assert be.calls == [("step", 3)] and env._substep == 3
    # per-step controls: handed over as (T, nu, nenv) -- without a copy when they already are a view of such a buffer
    buf = torch.randn(T, model.nu, 5, dtype=torch.float64)
    traj = env.rollout(controls=buf.permute(2, 0, 1), record=True)
    kind, seq, nsteps, record = be.calls[-1]
    assert (kind, nsteps, record) == ("rollout", T, True) and seq.data_ptr() == buf.data_ptr()
    assert torch.equal(seq, buf)
    env.rollout(T, controls=U)
    assert torch.equal(be.calls[-1][1], U.permute(1, 2, 0)) and be.calls[-1][3] is False
    assert traj["qpos"].shape == (5, T, model.nq) and traj["qvel"].shape == (5, T, model.nv) and "sensordata" not in traj
    assert env._substep == 3 + 2 * T
    h = float(model.opt.timestep)
    t = 0.0
    for _ in range(3 + 2 * T):
        t += h
    assert env.data.time == t  # repeated addition
    # a record of held controls
    env.rollout(2, record=True)
    assert be.calls[-1][1] is None and be.calls[-1][2] == 2


def test_batched_rollout_records_sensors_and_rejects_controls_without_actuators():
    from mujoco_template.exceptions import ConfigError

    env, model = _env("drone", 3)
    traj = env.rollout(4, record=True)
    assert traj["sensordata"].shape == (3, 4, model.nsensordata)
    env, model = _env("pendulum", 3)
    assert model.nsensordata == 0 and "sensordata" not in env.rollout(2, record=True)
    # a model without actuators takes no control sequence
    from types import SimpleNamespace

    env.model = SimpleNamespace(nu=0, nq=model.nq, nv=model.nv, nsensordata=0, opt=model.opt)
    with pytest.raises(ConfigError, match="no actuators"):
        env.rollout(controls=torch.zeros((3, 2, 0), dtype=torch.float64))
