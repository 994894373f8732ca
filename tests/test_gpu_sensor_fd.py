"""b2_linearize_sensors on the GPU: (A, B) and the sensor Jacobians C = d sensordata / dx, D = d sensordata / du of every
env from one FD launch, against the CPU reference of the same rollouts (tests/sensor_fd_reference.py)."""
import itertools

import numpy as np
import pytest

from conftest import load_model, oracle_for, random_states
from sensor_fd_reference import transition_fd_sensors
from test_sensor_fd import rows, sensor_rig

pytestmark = pytest.mark.gpu

AB_RTOL = 1e-6
# (A, B) of the sensor variant against b2_linearize's: a few units in the last place of a rollout's stepped state, divided
# by the FD step 2 eps = 2e-6, are ~1e-10 of an entry of A
AB_BITS = 1e-9
EPS = 1e-6


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b))))) if b.size else 0.0


def _batch(model, n, precision=64):
    import torch
    from mujoco_template import _mj as mj

    assert torch.cuda.is_available()
    return mj.BatchData(model, n, precision=precision)


def _upload(data, qpos, qvel, ctrl, warm):
    import torch

    dev, dt = data.qpos.device, data.qpos.dtype
    for dst, src in ((data.qpos, qpos), (data.qvel, qvel), (data.ctrl, ctrl), (data.qacc_warmstart, warm)):
        dst.copy_(torch.as_tensor(src.T.copy(), device=dev, dtype=dt))


def _host(t):
    return t.permute(2, 0, 1).cpu().numpy()


def _states(model, name, n, seed):
    if name == "drone":
        qpos, qvel, ctrl = random_states(model, "drone", n, seed=seed)
        ctrl[0, 0] = 0.0    # lower ctrlrange bound: forward one-sided column
        ctrl[1, 1] = 13.0   # upper bound: backward
        ctrl[2, 2] = 14.0   # outside the range: zero column
    else:
        rng = np.random.default_rng(seed)
        qpos = np.tile(model.qpos0, (n, 1))
        qpos[:, :3] = rng.uniform(-0.5, 0.5, (n, 3))
        q = rng.normal(size=(n, 4))
        qpos[:, 6:10] = q / np.linalg.norm(q, axis=1, keepdims=True)
        qvel = rng.normal(size=(n, model.nv))
        ctrl = rng.uniform(-1, 1, (n, model.nu))
    warm = np.random.default_rng(seed + 1).normal(0, 0.1, (n, model.nv))
    return qpos, qvel, ctrl, warm


CASES = [("drone", "drone"), ("drone-generic", "generic"), ("rig-euler", "generic"), ("rig-rk4", "generic")]


def _model(monkeypatch, case):
    if case.endswith("generic"):
        monkeypatch.setenv("B2_DISABLE_SPEC", "1")
    if case.startswith("rig"):
        return sensor_rig("RK4" if case.endswith("rk4") else "Euler"), "rig"
    return load_model("drone"), "drone"


@pytest.mark.parametrize("case,variant", CASES)
def test_sensor_jacobians_match_oracle(monkeypatch, case, variant):
    model, name = _model(monkeypatch, case)
    n = 24
    qpos, qvel, ctrl, warm = _states(model, name, n, seed=3)
    data = _batch(model, n)
    _upload(data, qpos, qvel, ctrl, warm)
    assert data.backend.batch.kernel_variant == variant
    A, B, C, D = (_host(t) for t in data.backend.linearize_sensors(EPS, True))
    # the state, warm start included, is untouched
    for arr, ref in ((data.qpos, qpos), (data.qvel, qvel), (data.ctrl, ctrl), (data.qacc_warmstart, warm)):
        assert np.array_equal(arr.cpu().numpy().T, ref)
    # (A, B) are b2_linearize's: the same rollouts in the same order.  Bit for bit on the generic kernels.  The specialised
    # drone kernel is register-resident and compiled as a whole: the sensor code changes the instruction selection of the
    # physics it shares (such as which products are contracted into FMAs), which may move the stepped states in the last
    # bits (measured on a B200: 2.2e-10 relative in A, see AB_BITS)
    A0, B0 = (_host(t) for t in data.backend.linearize(EPS, True))
    print(f"{case}: (A, B) of b2_linearize_sensors vs b2_linearize, relative {max(_rel(A, A0), _rel(B, B0)):.2e}")
    assert _rel(A, A0) <= AB_BITS and _rel(B, B0) <= AB_BITS
    if variant == "generic":
        assert np.array_equal(A, A0) and np.array_equal(B, B0)
    om, od = oracle_for(model)
    for e in range(n):
        od.reset()
        od.qpos[:] = qpos[e]; od.qvel[:] = qvel[e]; od.ctrl[:] = ctrl[e]; od.qacc_warmstart[:] = warm[e]
        Co, Do = transition_fd_sensors(model, od, EPS, True)
        Ao, Bo = od.transition_fd(EPS, True)
        assert _rel(A[e], Ao) <= AB_RTOL and _rel(B[e], Bo) <= AB_RTOL, (case, e)
        assert _rel(C[e], Co) <= AB_RTOL, (case, e, _rel(C[e], Co))
        assert _rel(D[e], Do) <= AB_RTOL, (case, e, _rel(D[e], Do))
    if name == "drone":
        assert np.all(D[2, :, 2] == 0)  # control outside its range


def test_every_null_combination(monkeypatch):
    from mujoco_template import _capi
    from mujoco_template.exceptions import ConfigError, LinearizationError

    model = load_model("drone")
    n = 40
    data = _batch(model, n)
    _upload(data, *_states(model, "drone", n, seed=7))
    full = [t.clone() for t in data.backend.linearize_sensors(EPS, True)]
    be = data.backend
    for mask in itertools.product((False, True), repeat=4):
        if not any(mask):
            continue
        bufs = [t.new_full(t.shape, float("nan")) if m else None for t, m in zip(full, mask)]
        be.batch.linearize_sensors(be.state_struct(), EPS, True, *[b.data_ptr() if b is not None else None for b in bufs])
        be.batch.synchronize()
        for b, ref in zip(bufs, full):
            if b is None:
                continue
            if any(mask[2:]):  # the sensor kernel: the very same values
                assert bool((b == ref).all()), mask
            else:  # neither C nor D: b2_linearize's kernel (see test_sensor_jacobians_match_oracle)
                assert _rel(b.cpu().numpy(), ref.cpu().numpy()) <= AB_BITS, mask
    with pytest.raises(ConfigError):
        be.batch.linearize_sensors(be.state_struct(), EPS, True, None, None, None, None)
    with pytest.raises(LinearizationError):
        be.batch.linearize_sensors(be.state_struct(), 0.0, True, *[t.data_ptr() for t in full])
    assert _capi.EXPORTED_SYMBOLS.count("b2_linearize_sensors") == 1


def test_model_without_sensors_is_b2_linearize():
    """humanoid (no sensors; its FD runs on the warp engine): exactly b2_linearize's (A, B), empty C / D."""
    model = load_model("humanoid")
    assert model.nsensordata == 0
    n = 6
    qpos, qvel, ctrl = random_states(model, "humanoid", n, seed=13)
    data = _batch(model, n)
    _upload(data, qpos, qvel, ctrl, np.zeros((n, model.nv)))
    assert data.backend.batch.kernel_variant == "generic-warp"
    A, B, C, D = data.backend.linearize_sensors(EPS, True)
    A0, B0 = data.backend.linearize(EPS, True)
    assert bool((A == A0).all()) and bool((B == B0).all())
    assert C.shape == (0, 2 * model.nv, n) and D.shape == (0, model.nu, n)


def test_framepos_rows_equal_the_device_jacobian():
    from mujoco_template import _capi

    model = sensor_rig()
    n = 16
    data = _batch(model, n)
    _upload(data, *_states(model, "rig", n, seed=5))
    _, _, C, _ = data.backend.linearize_sensors(EPS, True)
    jp, _ = data.backend.jacobian(_capi.JAC_SITE, 0, False)
    C, jp = _host(C), _host(jp)
    assert np.max(np.abs(C[:, rows(model, "p_site"), :model.nv] - jp)) <= 1e-7


def test_single_env_transitionFD_fills_C_and_D():
    from mujoco_template import _mj as mj

    model = load_model("drone")
    n = 8
    qpos, qvel, ctrl, warm = _states(model, "drone", n, seed=9)
    data = _batch(model, n)
    _upload(data, qpos, qvel, ctrl, warm)
    Ab, Bb, Cb, Db = (_host(t) for t in data.backend.linearize_sensors(EPS, True))
    d1 = mj.MjData(model)
    d1.qpos[:] = qpos[0]; d1.qvel[:] = qvel[0]; d1.ctrl[:] = ctrl[0]; d1.qacc_warmstart[:] = warm[0]
    nx, ns = 2 * model.nv, model.nsensordata
    A, B = np.zeros((nx, nx)), np.zeros((nx, model.nu))
    C, D = np.full((ns, nx), np.nan), np.full((ns, model.nu), np.nan)
    mj.mjd_transitionFD(model, d1, EPS, True, A, B, C, D)
    assert np.array_equal(A, Ab[0]) and np.array_equal(B, Bb[0])
    assert np.array_equal(C, Cb[0]) and np.array_equal(D, Db[0])


def test_batched_env_linearize_sensors_shapes():
    import mujoco_template as mt

    model = load_model("drone")
    n = 5
    env = mt.BatchedEnv(model, n)
    A, B = env.linearize()
    mats = env.linearize(sensors=True)
    nv, nu, ns = model.nv, model.nu, model.nsensordata
    assert [tuple(t.shape) for t in mats] == [(n, 2 * nv, 2 * nv), (n, 2 * nv, nu), (n, ns, 2 * nv), (n, ns, nu)]
    assert bool((mats[0] == A).all()) and bool((mats[1] == B).all())


def test_fp32_agrees_with_fp64():
    """FP32 batches at eps = 1e-3 (an FP32 FD step: rounding ~6e-8 |s| / 2e-3) against FP64 at the same eps.  (A, B) agree to
    1e-3 of the largest entry.  C / D are allowed 5e-2: their accelerometer rows are d qacc / dx themselves, where the
    velocity rows of A carry h d qacc / dx (h = 0.01 on the drone), so the same FP32 error in qacc weighs 1 / h more."""
    model = load_model("drone")
    n = 64
    qpos, qvel, ctrl, warm = _states(model, "drone", n, seed=17)
    out = {}
    for prec in (64, 32):
        data = _batch(model, n, precision=prec)
        _upload(data, qpos, qvel, ctrl, warm)
        out[prec] = [_host(t).astype(np.float64) for t in data.backend.linearize_sensors(1e-3, True)]
    for k, (m64, m32) in enumerate(zip(out[64], out[32])):
        err = float(np.max(np.abs(m32 - m64)) / max(1.0, float(np.max(np.abs(m64)))))
        print(f"matrix {'ABCD'[k]}: fp32 vs fp64 relative {err:.2e}")
        assert err <= (1e-3 if k < 2 else 5e-2), ("ABCD"[k], err)
