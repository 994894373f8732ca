"""GPU parity tests proper: CUDA path (through the C-ABI) vs the CPU oracle on seeded inputs.

Tolerances (BASELINE.json north_star): FP64 per-step relative error <= 1e-9 on qpos/qvel;
(A, B) relative error <= 1e-6.
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN, MODEL_NAMES, load_model, oracle_for, random_states

pytestmark = pytest.mark.gpu

STEP_RTOL = 1e-9
AB_RTOL = 1e-6


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b)))))


def _batch(model, n):
    import torch
    from mujoco_template import _mj as mj

    assert torch.cuda.is_available()
    return mj.BatchData(model, n)


def _upload(data, qpos, qvel, ctrl, warm=None):
    import torch

    data.qpos.copy_(torch.as_tensor(qpos.T.copy(), device=data.qpos.device))
    data.qvel.copy_(torch.as_tensor(qvel.T.copy(), device=data.qpos.device))
    data.ctrl.copy_(torch.as_tensor(ctrl.T.copy(), device=data.qpos.device))
    if warm is None:
        data.qacc_warmstart.zero_()
    else:
        data.qacc_warmstart.copy_(torch.as_tensor(warm.T.copy(), device=data.qpos.device))


N_ENVS = {"pendulum": 96, "cartpole": 96, "drone": 64, "humanoid": 24}


@pytest.mark.parametrize("name", MODEL_NAMES)
def test_step_parity_per_step(name):
    """Every step from a shared state: GPU step == oracle step to <= 1e-9 relative."""
    from mujoco_template import _mj as mj

    model = load_model(name)
    n = N_ENVS[name]
    qpos, qvel, ctrl = random_states(model, name, n, seed=1)
    warm = np.zeros((n, model.nv))
    data = _batch(model, n)
    om, od = oracle_for(model)
    nsteps = 40 if name != "humanoid" else 25
    worst = 0.0
    for s in range(nsteps):
        _upload(data, qpos, qvel, ctrl, warm)
        mj.mj_step(model, data)
        gq, gv, gw = data.qpos.cpu().numpy().T, data.qvel.cpu().numpy().T, data.qacc_warmstart.cpu().numpy().T
        for e in range(n):
            od.reset()
            od.qpos[:] = qpos[e]; od.qvel[:] = qvel[e]; od.ctrl[:] = ctrl[e]; od.qacc_warmstart[:] = warm[e]
            od.step()
            qpos[e] = od.qpos; qvel[e] = od.qvel; warm[e] = od.qacc_warmstart
        worst = max(worst, _rel(gq, qpos), _rel(gv, qvel))
        assert _rel(gq, qpos) <= STEP_RTOL, (name, s, _rel(gq, qpos))
        assert _rel(gv, qvel) <= STEP_RTOL, (name, s, _rel(gv, qvel))
        assert _rel(gw, warm) <= 1e-7, (name, s, _rel(gw, warm))
    assert int(data.flags.max().item()) == 0
    print(f"{name}: worst per-step rel err {worst:.3e}")


@pytest.mark.parametrize("name", ["pendulum", "cartpole", "drone"])
def test_free_running_trajectory(name):
    """Independent 200-step rollouts stay within 1e-7 (smooth dynamics, no chaos at this horizon)."""
    from mujoco_template import _mj as mj

    model = load_model(name)
    n = 32
    qpos, qvel, ctrl = random_states(model, name, n, seed=2)
    if name == "drone":  # near-hover thrust: no tumbling into the floor within 2 s
        ctrl = np.random.default_rng(7).uniform(2.9, 3.6, ctrl.shape)
    data = _batch(model, n)
    _upload(data, qpos, qvel, ctrl)
    mj.mj_step(model, data, 200)  # fused launch
    om, od = oracle_for(model)
    om.batch_rollout(qpos, qvel, ctrl, nsteps=200, nthreads=4)
    assert np.all(np.isfinite(qpos))
    assert _rel(data.qpos.cpu().numpy().T, qpos) <= 1e-7
    assert _rel(data.qvel.cpu().numpy().T, qvel) <= 1e-7
    assert abs(data.time - 200 * model.opt.timestep) < 1e-9


def test_drone_landing_contacts_per_step():
    """Plane-box and plane-ellipsoid contacts (drone dropped with tilt, motors off)."""
    from mujoco_template import _mj as mj

    model = load_model("drone")
    n = 16
    qpos, qvel, ctrl = random_states(model, "drone", n, seed=8)
    qpos[:, 2] = np.linspace(0.12, 0.4, n)
    ctrl[:] = 0.0
    warm = np.zeros((n, model.nv))
    data = _batch(model, n)
    om, od = oracle_for(model)
    seen = 0
    for s in range(120):
        _upload(data, qpos, qvel, ctrl, warm)
        mj.mj_step(model, data)
        ncon_gpu = data.ncon.cpu().numpy()[0]
        for e in range(n):
            od.reset(); od.qpos[:] = qpos[e]; od.qvel[:] = qvel[e]; od.ctrl[:] = ctrl[e]; od.qacc_warmstart[:] = warm[e]
            od.step()
            assert od.ncon == ncon_gpu[e], (s, e)
            seen = max(seen, od.ncon)
            qpos[e] = od.qpos; qvel[e] = od.qvel; warm[e] = od.qacc_warmstart
        assert _rel(data.qpos.cpu().numpy().T, qpos) <= STEP_RTOL, s
        assert _rel(data.qvel.cpu().numpy().T, qvel) <= 1e-8, s
    assert seen >= 4


def test_drone_landing_contacts_fused_launches():
    """The same landing with eight steps per launch: within a fused launch the drone's kernel hands the state -- the
    warm start included -- from step to step through the SoA arrays (state streaming), so every launch must land where
    eight oracle steps from the same state and warm start do."""
    from mujoco_template import _mj as mj

    model = load_model("drone")
    n = 16
    qpos, qvel, ctrl = random_states(model, "drone", n, seed=8)
    qpos[:, 2] = np.linspace(0.12, 0.4, n)
    ctrl[:] = 0.0
    warm = np.zeros((n, model.nv))
    data = _batch(model, n)
    om, od = oracle_for(model)
    seen = 0
    for s in range(15):
        _upload(data, qpos, qvel, ctrl, warm)
        mj.mj_step(model, data, 8)
        for e in range(n):
            od.reset(); od.qpos[:] = qpos[e]; od.qvel[:] = qvel[e]; od.ctrl[:] = ctrl[e]; od.qacc_warmstart[:] = warm[e]
            for _ in range(8):
                od.step()
                seen = max(seen, od.ncon)
            qpos[e] = od.qpos; qvel[e] = od.qvel; warm[e] = od.qacc_warmstart
        assert _rel(data.qpos.cpu().numpy().T, qpos) <= 1e-8, s
        assert _rel(data.qvel.cpu().numpy().T, qvel) <= 1e-7, s
        assert _rel(data.qacc_warmstart.cpu().numpy().T, warm) <= 1e-6, s
    assert seen >= 4
    assert int(data.flags.max().item()) == 0


def test_bad_state_is_flagged_not_reset():
    """Upstream silently resets mjData on NaN/huge values; we flag the env instead (DESIGN.md)."""
    from mujoco_template import _capi, _mj as mj

    model = load_model("drone")
    n = 4
    qpos, qvel, ctrl = random_states(model, "drone", n, seed=9)
    qvel[1, 0] = 1e12
    qpos[2, 1] = np.nan
    data = _batch(model, n)
    _upload(data, qpos, qvel, ctrl)
    mj.mj_step(model, data)
    flags = data.flags.cpu().numpy()[0]
    assert flags[0] == 0 and flags[3] == 0
    assert flags[1] & _capi.FLAG_BAD_QVEL and flags[2] & _capi.FLAG_BAD_QPOS
    # ... and frozen: a flagged env is left exactly as it was, its neighbours step normally
    q1, v1 = data.qpos.cpu().numpy().T, data.qvel.cpu().numpy().T
    assert np.array_equal(q1[1], qpos[1]) and np.array_equal(v1[1], qvel[1])
    assert np.array_equal(v1[2], qvel[2]) and np.array_equal(np.isnan(q1[2]), np.isnan(qpos[2]))
    assert not np.array_equal(q1[0], qpos[0]) and not np.array_equal(q1[3], qpos[3])


def test_bad_state_is_frozen_on_the_warp_engine():
    from mujoco_template import _capi, _mj as mj

    model = load_model("humanoid")
    n = 5  # odd: the last lock-step pair has one env only
    qpos, qvel, ctrl = random_states(model, "humanoid", n, seed=3)
    qvel[1, 4] = -3e11
    qpos[4, 9] = np.inf
    data = _batch(model, n)
    _upload(data, qpos, qvel, ctrl)
    mj.mj_step(model, data, 2)
    flags = data.flags.cpu().numpy()[0]
    assert flags[0] == 0 and flags[2] == 0 and flags[3] == 0
    assert flags[1] & _capi.FLAG_BAD_QVEL and flags[4] & _capi.FLAG_BAD_QPOS
    q1, v1 = data.qpos.cpu().numpy().T, data.qvel.cpu().numpy().T
    assert np.array_equal(q1[1], qpos[1]) and np.array_equal(v1[1], qvel[1])
    assert np.array_equal(q1[4], qpos[4]) and np.array_equal(v1[4], qvel[4])
    # the healthy envs match the oracle
    om, od = oracle_for(model)
    for e in (0, 2, 3):
        od.reset()
        od.qpos[:] = qpos[e]; od.qvel[:] = qvel[e]; od.ctrl[:] = ctrl[e]
        od.step(2)
        assert _rel(q1[e], od.qpos) <= STEP_RTOL and _rel(v1[e], od.qvel) <= 1e-8


@pytest.mark.parametrize("name", MODEL_NAMES)
def test_linearize_parity(name):
    model = load_model(name)
    n = 16 if name != "humanoid" else 4
    qpos, qvel, ctrl = random_states(model, name, n, seed=3)
    if name == "drone":
        ctrl[0, 0] = 0.0   # at the lower ctrlrange bound: forward one-sided difference
        ctrl[1, 1] = 13.0  # at the upper bound: backward difference
    if name == "humanoid":
        ctrl[0, 3] = 1.0    # upper bound: backward difference
        ctrl[1, 5] = -1.0   # lower bound: forward difference
        ctrl[2, 7] = 1.5    # outside the range: mjd_transitionFD leaves the column at zero
    data = _batch(model, n)
    _upload(data, qpos, qvel, ctrl)
    eps = 1e-6
    A, B = data.backend.linearize(eps, True)
    A = A.permute(2, 0, 1).cpu().numpy(); B = B.permute(2, 0, 1).cpu().numpy()
    # state untouched
    assert np.array_equal(data.qpos.cpu().numpy().T, qpos)
    om, od = oracle_for(model)
    for e in range(n):
        od.reset()
        od.qpos[:] = qpos[e]; od.qvel[:] = qvel[e]; od.ctrl[:] = ctrl[e]
        Ao, Bo = od.transition_fd(eps, True)
        assert _rel(A[e], Ao) <= AB_RTOL, (name, e, _rel(A[e], Ao))
        assert _rel(B[e], Bo) <= AB_RTOL, (name, e, _rel(B[e], Bo))


def test_warp_engine_fd_matches_lane_engine_fd(monkeypatch):
    """humanoid (A, B): k_warp_linearize (one warp per column rollout pair) vs the lane engine's k_linearize."""
    model = load_model("humanoid")
    n = 7  # odd: the last lock-step pair of the last column has one item only
    qpos, qvel, ctrl = random_states(model, "humanoid", n, seed=13)
    ctrl[3, 0] = -1.0
    out = {}
    for warp in ("1", "0"):
        monkeypatch.setenv("B2_DISABLE_WARP", "0" if warp == "1" else "1")  # the batch picks its engine when it is created
        data = _batch(model, n)
        _upload(data, qpos, qvel, ctrl)
        A, B = data.backend.linearize(1e-6, True)
        out[warp] = (A.cpu().numpy(), B.cpu().numpy(), data.qpos.cpu().numpy().T.copy())
    assert np.array_equal(out["1"][2], qpos) and np.array_equal(out["0"][2], qpos)
    # same algorithm, different summation orders inside a step: roundoff amplified by 1 / eps
    assert _rel(out["1"][0], out["0"][0]) <= 1e-7 and _rel(out["1"][1], out["0"][1]) <= 1e-7
    assert np.abs(out["1"][0]).max() > 0.5 and np.abs(out["1"][1]).max() > 1e-3


@pytest.mark.parametrize("name", MODEL_NAMES)
def test_forward_derived_and_jacobians(name):
    from mujoco_template import _capi, _mj as mj

    model = load_model(name)
    n = 8
    qpos, qvel, ctrl = random_states(model, name, n, seed=4)
    data = _batch(model, n)
    _upload(data, qpos, qvel, ctrl)
    mj.mj_forward(model, data)
    om, od = oracle_for(model)
    body = model.nbody - 1
    for e in range(n):
        od.reset()
        od.qpos[:] = qpos[e]; od.qvel[:] = qvel[e]; od.ctrl[:] = ctrl[e]
        od.forward()
        assert _rel(data.xpos[:, e].cpu().numpy().reshape(-1, 3), od.xpos) <= 1e-12
        assert _rel(data.xipos[:, e].cpu().numpy().reshape(-1, 3), od.xipos) <= 1e-12
        assert _rel(data.geom_xpos[:, e].cpu().numpy().reshape(-1, 3), od.geom_xpos) <= 1e-12
        assert _rel(data.subtree_com[:, e].cpu().numpy().reshape(-1, 3), od.subtree_com) <= 1e-12
        assert _rel(data.qacc[:, e].cpu().numpy(), od.qacc) <= 1e-8
        assert int(data.ncon[0, e]) == od.ncon and int(data.nefc[0, e]) == od.nefc
        if model.nsite:
            assert _rel(data.site_xpos[:, e].cpu().numpy().reshape(-1, 3), od.site_xpos) <= 1e-12
    kinds = [("body", _capi.JAC_BODY, body), ("bodycom", _capi.JAC_BODYCOM, body), ("subtreecom", _capi.JAC_SUBTREECOM, 1)]
    if model.nsite:
        kinds.append(("site", _capi.JAC_SITE, model.nsite - 1))
    for kname, code, idx in kinds:
        jp, jr = data.backend.jacobian(code, idx, code in (_capi.JAC_BODY, _capi.JAC_SITE))
        for e in range(n):
            od.reset(); od.qpos[:] = qpos[e]; od.forward()
            jpo, jro = od.jac(kname, idx)
            assert _rel(jp[:, :, e].cpu().numpy(), jpo) <= 1e-12, (name, kname)
            if jr is not None:
                assert _rel(jr[:, :, e].cpu().numpy(), jro) <= 1e-12


@pytest.mark.parametrize("name", ["drone", "humanoid", "cartpole"])
def test_integrate_differentiate_pos(name):
    import torch

    model = load_model(name)
    n = 8
    qpos, qvel, _ = random_states(model, name, n, seed=5)
    rng = np.random.default_rng(6)
    vel = rng.normal(0, 1.0, (n, model.nv))
    data = _batch(model, n)
    dev = data.qpos.device
    q = torch.as_tensor(qpos.T.copy(), device=dev)
    v = torch.as_tensor(vel.T.copy(), device=dev)
    q2 = q.clone()
    data.backend.batch.integrate_pos(q2.data_ptr(), v.data_ptr(), 0.37)
    out = torch.zeros_like(v)
    data.backend.batch.differentiate_pos(out.data_ptr(), 0.37, q.data_ptr(), q2.data_ptr())
    torch.cuda.synchronize()
    om, od = oracle_for(model)
    for e in range(n):
        qo = od.integrate_pos(qpos[e], vel[e], 0.37)
        assert _rel(q2[:, e].cpu().numpy(), qo) <= 1e-13
        assert _rel(out[:, e].cpu().numpy(), od.differentiate_pos(0.37, qpos[e], qo)) <= 1e-12
    # round trip: differentiate(integrate(q, v, dt)) == v
    assert _rel(out.cpu().numpy().T, vel) <= 1e-9


def test_humanoid_contacts_active_and_reported():
    from mujoco_template import _mj as mj

    model = load_model("humanoid")
    data = _batch(model, 8)
    mj.mj_resetDataKeyframe(model, data, 1)
    mj.mj_forward(model, data)
    assert int(data.ncon.min()) == 4 and int(data.nefc.min()) == 16
    mj.mj_step(model, data, 300)
    assert int(data.flags.max()) == 0
    assert float(data.qpos[2].min()) > 0.0  # nobody fell through the floor


def test_cartpole_limit_and_floor_contact():
    """Slider limit (|x| > 2) and pole-floor contact rows match the oracle."""
    from mujoco_template import _mj as mj

    model = load_model("cartpole")
    n = 4
    qpos = np.array([[2.05, 0.1], [-2.1, -0.3], [0.0, 1.75], [1.99, -1.8]])
    qvel = np.array([[1.0, 0.0], [-0.5, 0.2], [0.0, 1.0], [0.3, -1.0]])
    ctrl = np.array([[100.0], [-250.0], [0.0], [10.0]])
    data = _batch(model, n)
    om, od = oracle_for(model)
    warm = np.zeros((n, 2))
    for s in range(60):
        _upload(data, qpos, qvel, ctrl, warm)
        mj.mj_step(model, data)
        for e in range(n):
            od.reset(); od.qpos[:] = qpos[e]; od.qvel[:] = qvel[e]; od.ctrl[:] = ctrl[e]; od.qacc_warmstart[:] = warm[e]
            od.step()
            qpos[e] = od.qpos; qvel[e] = od.qvel; warm[e] = od.qacc_warmstart
        assert _rel(data.qpos.cpu().numpy().T, qpos) <= STEP_RTOL, s
        assert _rel(data.qvel.cpu().numpy().T, qvel) <= STEP_RTOL, s


def test_single_env_config1_pendulum_cli():
    """BASELINE config #1: pendulum, ZeroController, 300 steps from reset (stationary)."""
    import mujoco_template as mt
    from conftest import load_model

    model = load_model("pendulum")
    handle = mt.ModelHandle(model)
    env = mt.Env(handle, obs_spec=mt.ObservationSpec(include_time=True), controller=mt.ZeroController())
    env.reset()
    steps = sum(1 for _ in env.passive(max_steps=300))
    assert steps == 300
    assert env.data.qpos[0] == 0.0 and env.data.qvel[0] == 0.0
    t = 0.0
    for _ in range(300):
        t += 0.005
    assert env.data.time == t


def test_single_env_linearize_and_info():
    import mujoco_template as mt

    class Lin:
        capabilities = mt.ControllerCapabilities(needs_linearization=True, needs_jacobians=("site:tip", "bodycom:pole"))
        def prepare(self, model, data): pass
        def __call__(self, model, data, t): data.ctrl[:] = 0.25

    model = load_model("cartpole")
    env = mt.Env(mt.ModelHandle(model), obs_spec=mt.ObservationSpec(sites_pos=("tip",), as_dict=False), controller=Lin())
    env.reset()
    env.data.qpos[:] = [0.1, 0.05]
    res = env.step()
    A, B = res.info["A"], res.info["B"]
    assert A.shape == (4, 4) and B.shape == (4, 1) and np.all(np.isfinite(A))
    assert res.info["jacobians"]["site:tip"]["jacp"].shape == (3, 2)
    assert res.obs.shape == (2 + 2 + 3,)
    res3 = env.step(3)
    assert isinstance(res3.info["A"], list) and len(res3.info["A"]) == 3
    om, od = oracle_for(model)
    A2, B2 = env.linearize()
    od.qpos[:] = env.data.qpos; od.qvel[:] = env.data.qvel; od.ctrl[:] = env.data.ctrl
    od.qacc_warmstart[:] = env.data.qacc_warmstart
    Ao, Bo = od.transition_fd(1e-6, True)
    assert _rel(A2, Ao) <= AB_RTOL and _rel(B2, Bo) <= AB_RTOL
    # python FD fallback path runs and agrees with native in the velocity rows
    A3, B3 = mt.linearize_discrete(env.model, env.data, use_native=False)
    assert _rel(A3[2:], A2[2:]) <= 1e-5 and _rel(A3[:2], -A2[:2]) <= 1e-5


def test_batched_env_lqr_graph_equals_eager_and_stabilises():
    """BatchedEnv + batched LQR: CUDA-graph replay is bit-identical to eager stepping; the pole stays up."""
    import torch
    import mujoco_template as mt
    from mujoco_template.batched_controllers import BatchedLQRController

    model = load_model("cartpole")
    n = 512
    qpos, qvel, _ = random_states(model, "cartpole", n, seed=12)
    outs = []
    for graph in (False, True):
        ctrl = BatchedLQRController(Q=np.diag([10.0, 100.0, 1.0, 1.0]), R=np.array([[0.01]]))
        env = mt.BatchedEnv(model, n, controller=ctrl)
        env.reset()
        env.data.qpos.copy_(torch.as_tensor(qpos.T.copy(), device=env.data.qpos.device))
        env.data.qvel.copy_(torch.as_tensor(qvel.T.copy(), device=env.data.qpos.device))
        if graph:
            env.enable_cuda_graph(True)
        last = None
        for _ in range(300):
            last = env.step(return_obs=False)
        torch.cuda.synchronize()
        assert last.info["A"].shape == (n, 4, 4) and last.info["B"].shape == (n, 4, 1)
        outs.append((env.data.qpos.cpu().numpy(), env.data.qvel.cpu().numpy(), last.info["A"].cpu().numpy(), env.data.time))
        assert int(env.data.flags.max()) == 0
        assert float(env.data.qpos[1].abs().max()) < 0.05      # every pole is upright after 3 s
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1])
    assert np.array_equal(outs[0][2], outs[1][2]) and outs[0][3] == outs[1][3]
    # (A, B) of env 0 at the final state agree with the oracle's mjd_transitionFD
    om, od = oracle_for(model)
    env2 = mt.BatchedEnv(model, n)
    A, B = env.linearize()
    od.qpos[:] = env.data.qpos[:, 0].cpu().numpy(); od.qvel[:] = env.data.qvel[:, 0].cpu().numpy()
    od.ctrl[:] = env.data.ctrl[:, 0].cpu().numpy(); od.qacc_warmstart[:] = env.data.qacc_warmstart[:, 0].cpu().numpy()
    Ao, Bo = od.transition_fd(1e-6, True)
    assert _rel(A[0].cpu().numpy(), Ao) <= AB_RTOL and _rel(B[0].cpu().numpy(), Bo) <= AB_RTOL
    assert env.data.backend.batch.kernel_variant == "cartpole" and env2.data.backend.batch.kernel_variant == "cartpole"


def test_batched_observations_and_jacobians():
    import torch
    import mujoco_template as mt

    model = load_model("drone")
    n = 16

    class Hold:
        capabilities = mt.ControllerCapabilities(needs_jacobians=("site:imu", "subtreecom:x2"))
        def prepare(self, m, d): pass
        def __call__(self, m, d, t): d.ctrl[:] = 3.2495625

    env = mt.BatchedEnv(model, n, controller=Hold(), obs_spec=mt.ObservationSpec(include_time=True, sites_pos=("imu",), as_dict=False))
    obs0 = env.reset("hover")
    assert obs0.shape == (7 + 6 + 3 + 1, n)
    res = env.step(2)
    assert isinstance(res.info["jacobians"], list) and res.info["jacobians"][0]["site:imu"]["jacp"].shape == (n, 3, 6)
    assert "jacr" not in res.info["jacobians"][0]["subtreecom:x2"]
    assert torch.allclose(env.data.qpos[2], torch.full((n,), 0.3, dtype=torch.float64, device=env.data.qpos.device), atol=1e-9)
    assert env.data.time == 0.01 + 0.01


# FP32 mode: stated divergence bounds |qpos_fp32 - qpos_fp64| (max over coordinates; median / max over 128 envs) at 100, 300
# and 1000 steps.  Measured on B200 with tools/fp32_divergence.py (256 envs; profiles/fp32_divergence_r02.jsonl, table in
# BASELINE.md); the bounds below leave a factor 5-10 over the measurement.  The error starts at the FP32 rounding level of the
# state (6e-8 relative) and grows like exp(rate * t); "rate" is the measured exponent between 100 and 1000 steps.
#   regime                                           median 100 / 300 / 1000        max 100 / 300 / 1000      rate [1/s]
#   pendulum, passive swing |theta0| <= 2 rad        1.0e-7  2.3e-7  6.3e-7         6.6e-7  2.4e-6  4.2e-5     0.41
#   pendulum, released within 0.05 rad of upright    1.3e-6  3.8e-6  2.5e-3         5.8e-6  6.9e-4  (wraps)    1.68
#   cartpole, passive damped                         1.6e-7  2.0e-7  2.1e-7         1.2e-6  5.9e-6  6.8e-6     0.03
#   drone, hover thrust held (open loop, unstable)   4.6e-7  1.4e-5  5.2e-2         2.0e-6  2.6e-3  (metres)   1.29
#   humanoid, falling from stand_on_left_leg         1.8e-6  1.0e-4  1.4e-4         1.3e-2  5.7e-1  2.6e-1     0.96
#   humanoid, at rest on the floor                   1.4e-6  2.9e-6  7.7e-6         9.3e-5  8.0e-5  7.4e-5     0.38
# Regular regimes carry a 1000-step bound; the unstable ones (inverted pendulum, open-loop drone, a falling humanoid whose
# contact times shift) are bounded over the horizon in which exp(rate * t) * 6e-8 is still small, and by their medians.
FP32_BOUNDS = {
    # regime: {steps: (median bound, max bound or None)}
    ("pendulum", "swing"): {100: (1e-6, 5e-6), 300: (2e-6, 2e-5), 1000: (5e-6, 5e-4)},
    ("pendulum", "upright"): {100: (1e-5, 5e-5), 300: (5e-5, 5e-3)},
    ("cartpole", "passive"): {100: (2e-6, 1e-5), 300: (2e-6, 5e-5), 1000: (2e-6, 1e-4)},
    ("drone", "hover"): {100: (5e-6, 2e-5), 300: (2e-4, 3e-2)},
    ("humanoid", "falling"): {100: (2e-5, 1e-1), 300: (1e-3, None), 1000: (2e-3, None)},
    ("humanoid", "rest"): {100: (2e-5, 1e-3), 300: (3e-5, 1e-3), 1000: (1e-4, 1e-3)},
}


def test_fp32_mode_divergence_bound_1000_steps():
    """Optional FP32 mode (B2_F32): the stated trajectory-divergence bounds against the FP64 path (table above)."""
    import torch
    from mujoco_template import _mj as mj

    n = 128
    for (name, regime), bounds in FP32_BOUNDS.items():
        model = load_model(name)
        qpos, qvel, ctrl = random_states(model, name, n, seed=21)
        ctrl[:] = 0
        pre = 0
        if regime == "swing":
            qpos[:, 0] = np.linspace(-2.0, 2.0, n); qvel[:] = 0
        elif regime == "upright":
            qpos[:, 0] = np.pi + np.linspace(-0.05, 0.05, n); qvel[:] = 0
        elif regime == "hover":
            ctrl[:] = 3.2495625
        elif regime == "rest":
            pre = 1500
        if pre:
            d = mj.BatchData(model, n)
            d.qpos.copy_(torch.as_tensor(qpos.T.copy(), device="cuda")); d.qvel.copy_(torch.as_tensor(qvel.T.copy(), device="cuda"))
            mj.mj_step(model, d, pre)
            qpos, qvel = d.qpos.cpu().numpy().T.copy(), d.qvel.cpu().numpy().T.copy()
        traj = {}
        for prec in (64, 32):
            d = mj.BatchData(model, n, precision=prec)
            dt = d.qpos.dtype
            d.qpos.copy_(torch.as_tensor(qpos.T.copy(), device="cuda").to(dt))
            d.qvel.copy_(torch.as_tensor(qvel.T.copy(), device="cuda").to(dt))
            d.ctrl.copy_(torch.as_tensor(ctrl.T.copy(), device="cuda").to(dt))
            done, out = 0, {}
            for k in sorted(bounds):
                mj.mj_step(model, d, k - done); done = k
                out[k] = d.qpos.double().cpu().numpy()
            traj[prec] = out
            assert int(d.flags.max()) == 0 and np.all(np.isfinite(out[max(bounds)]))
        for k, (med_bound, max_bound) in bounds.items():
            err = np.abs(traj[64][k] - traj[32][k]).max(axis=0)
            print(f"fp32 divergence, {name} / {regime}, {k} steps: median {np.median(err):.2e} max {err.max():.2e}")
            assert np.median(err) <= med_bound, (name, regime, k, float(np.median(err)))
            if max_bound is not None:
                assert err.max() <= max_bound, (name, regime, k, float(err.max()))


@pytest.mark.parametrize("name,n", [("cartpole", 8192), ("drone", 4100), ("humanoid", 64)])
def test_step_host_pipeline_matches_device_path(name, n):
    """b2_step_host (host buffers, chunked copy/compute pipeline replayed as a CUDA graph) == device path."""
    import torch
    from mujoco_template import _capi, _mj as mj

    model = load_model(name)
    qpos, qvel, ctrl = random_states(model, name, n, seed=31)
    if name == "drone":
        ctrl[:] = 3.3
    data = _batch(model, n)
    _upload(data, qpos, qvel, ctrl)
    nv, nu = model.nv, model.nu
    hq = torch.as_tensor(qpos.T.copy()).pin_memory(); hv = torch.as_tensor(qvel.T.copy()).pin_memory()
    hu = torch.as_tensor(ctrl.T.copy()).pin_memory(); hw = torch.zeros((nv, n), dtype=torch.float64).pin_memory()
    hA = torch.zeros((2 * nv, 2 * nv, n), dtype=torch.float64).pin_memory(); hB = torch.zeros((2 * nv, nu, n), dtype=torch.float64).pin_memory()
    st = _capi.State(hq.data_ptr(), hv.data_ptr(), hu.data_ptr(), hw.data_ptr(), None)
    lin = name != "humanoid"
    for rep in range(3):  # first call captures the graph, later calls replay it
        if lin:
            A, B = data.backend.linearize(1e-6, True)
        mj.mj_step(model, data, 2)
        data.backend.batch.step_host(st, 2, lin, 1e-6, hA.data_ptr() if lin else None, hB.data_ptr() if lin else None, 0)
        assert np.array_equal(hq.numpy(), data.qpos.cpu().numpy()), rep
        assert np.array_equal(hv.numpy(), data.qvel.cpu().numpy()), rep
        assert np.array_equal(hw.numpy(), data.qacc_warmstart.cpu().numpy()), rep
        if lin:
            assert np.array_equal(hA.numpy(), A.cpu().numpy()) and np.array_equal(hB.numpy(), B.cpu().numpy()), rep


def test_step_host_async_half_batches_equal_the_synchronous_call():
    """B2_HOST_ASYNC + b2_step_host_wait: two half-batches, each a closed loop through its own pinned buffers and driven
    alternately (wait, submit), land bit for bit where one synchronous b2_step_host over the whole batch does."""
    import torch
    from mujoco_template import _capi, _mj as mj

    model = load_model("cartpole")
    n, half = 512, 256
    qpos, qvel, ctrl = random_states(model, "cartpole", n, seed=33)
    nv, nu = model.nv, model.nu

    def buffers(sl):
        hq = torch.as_tensor(qpos[sl].T.copy()).pin_memory(); hv = torch.as_tensor(qvel[sl].T.copy()).pin_memory()
        hu = torch.as_tensor(ctrl[sl].T.copy()).pin_memory(); m = hq.shape[1]
        hw = torch.zeros((nv, m), dtype=torch.float64).pin_memory()
        hA = torch.zeros((2 * nv, 2 * nv, m), dtype=torch.float64).pin_memory(); hB = torch.zeros((2 * nv, nu, m), dtype=torch.float64).pin_memory()
        return hq, hv, hu, hw, hA, hB

    whole = buffers(slice(0, n))
    data = _batch(model, n)
    st = _capi.State(*(t.data_ptr() for t in whole[:4]), None)
    parts = []
    for sl in (slice(0, half), slice(half, n)):
        bufs = buffers(sl)
        parts.append((_capi.NativeBatch(data.backend.batch.model, half, 0), _capi.State(*(t.data_ptr() for t in bufs[:4]), None), bufs))
    nsteps = 6
    for _ in range(nsteps):
        data.backend.batch.step_host(st, 1, True, 1e-6, whole[4].data_ptr(), whole[5].data_ptr(), 0)
    for b, s, bufs in parts:
        b.step_host(s, 1, True, 1e-6, bufs[4].data_ptr(), bufs[5].data_ptr(), 0, wait=False)
    for _ in range(nsteps - 1):
        for b, s, bufs in parts:
            b.step_host_wait()
            b.step_host(s, 1, True, 1e-6, bufs[4].data_ptr(), bufs[5].data_ptr(), 0, wait=False)
    for b, s, bufs in parts:
        b.step_host_wait()
        b.step_host_wait()  # idempotent
    for k in range(6):
        got = torch.cat([parts[0][2][k], parts[1][2][k]], dim=-1).numpy()
        assert np.array_equal(got, whole[k].numpy()), k
    assert np.abs(whole[4].numpy()).max() > 0


@pytest.mark.parametrize("name,graph", [("drone", False), ("drone", True), ("cartpole", False), ("humanoid", False)])
def test_lazy_derived_outputs_equal_eager_ones(name, graph):
    """step(return_obs=False) runs without derived outputs (b2_step_lazy: the pre-step state is parked); reading
    data.xpos / sensordata / qacc afterwards materialises exactly what the eager step writes."""
    import torch
    import mujoco_template as mt

    class Hold:  # a controller, so that the CUDA-graph path is exercised too
        capabilities = mt.ControllerCapabilities()
        def prepare(self, m, d): pass
        def __call__(self, m, d, t): d.ctrl.mul_(1.0)

    model = load_model(name)
    n = 96
    qpos, qvel, ctrl = random_states(model, name, n, seed=31)
    out = {}
    for lazy in (True, False):
        env = mt.BatchedEnv(model, n, controller=Hold())
        env.reset(1 if name == "humanoid" else None)
        dev = env.data.qpos.device
        env.data.qpos.copy_(torch.as_tensor(qpos.T.copy(), device=dev)); env.data.qvel.copy_(torch.as_tensor(qvel.T.copy(), device=dev))
        env.data.ctrl.copy_(torch.as_tensor(ctrl.T.copy(), device=dev))
        env.forward()
        if graph:
            env.enable_cuda_graph(True)
        for _ in range(5):
            env.step(return_obs=not lazy)
            if lazy:
                assert env.data.backend.derived_stale
        names = ["qpos", "qvel", "xpos", "xquat", "geom_xpos", "subtree_com", "qacc", "qfrc_bias", "ncon", "nefc"]
        if model.nsensordata:
            names.append("sensordata")
        if model.nsite:
            names.append("site_xpos")
        out[lazy] = {k: getattr(env.data, k).clone() for k in names}
        assert not env.data.backend.derived_stale
    for k in out[True]:
        assert torch.equal(out[True][k], out[False][k]), k


def test_control_tick_on_the_warp_engine():
    """humanoid: b2_control_tick = control-law launch + warp-engine FD + warp-engine step; the derived arrays of the
    tick are produced lazily from the parked pre-step state, as on the small models."""
    from mujoco_template import _mj as mj

    model = load_model("humanoid")
    n = 6
    qpos, qvel, _ = random_states(model, "humanoid", n, seed=17)
    rng = np.random.default_rng(0)
    K = rng.normal(0, 0.02, (model.nu, 2 * model.nv))
    qref, uref = np.array(model.key_qpos[1]), np.zeros(model.nu)
    out = {}
    for fused in (True, False):
        data = _batch(model, n)
        _upload(data, qpos, qvel, np.zeros((n, model.nu)))
        data.backend.batch.lqr_set_gain(K, qref, uref)
        for _ in range(3):
            if fused:
                A, B = data.backend.control_tick(1e-6, True, True, derived=False)
                assert data.backend.derived_stale
            else:
                data.backend.batch.lqr_control(data.backend.state_struct())
                A, B = data.backend.linearize(1e-6, True)
                data.backend.step(1)
        out[fused] = [x.clone() for x in (data.qpos, data.qvel, data.ctrl, A, B, data.xpos, data.qacc)]
        assert not data.backend.derived_stale
    for k, (a, b) in enumerate(zip(out[True], out[False])):
        assert a.shape == b.shape and bool((a == b).all()), k   # the same kernels on the same inputs: bit-identical
    assert float(out[True][2].abs().max()) > 1e-3               # the law did produce controls


@pytest.mark.parametrize("name", ["cartpole", "drone"])
def test_fused_lqr_control_kernel_matches_torch_reference(name):
    """b2_lqr_control (one launch) == the same tick written with torch ops, incl. quaternion error and ctrl clamp."""
    import torch
    import mujoco_template as mt
    from mujoco_template.batched_controllers import BatchedLQRController

    model = load_model(name)
    n = 200
    qpos, qvel, _ = random_states(model, name, n, seed=51)
    kw = dict(Q=np.diag([10.0, 100.0, 1.0, 1.0]), R=np.array([[0.01]])) if name == "cartpole" else \
        dict(qpos_ref=model.key_qpos[0], ctrl_ref=model.key_ctrl[0], R=np.eye(4) * 0.1)
    out = []
    for fused in (True, False):
        ctrl = BatchedLQRController(needs_linearization=False, fused=fused, **kw)
        env = mt.BatchedEnv(model, n, controller=ctrl)
        env.data.qpos.copy_(torch.as_tensor(qpos.T.copy(), device=env.data.qpos.device))
        env.data.qvel.copy_(torch.as_tensor(qvel.T.copy(), device=env.data.qpos.device))
        if name == "cartpole":
            env.data.qpos[0, :4] = 50.0    # far away: the +-200 ctrlrange clamp is hit
        ctrl(model, env.data, 0.0)
        torch.cuda.synchronize()
        out.append(env.data.ctrl.cpu().numpy().copy())
    assert np.allclose(out[0], out[1], rtol=1e-12, atol=1e-12)
    if name == "cartpole":
        assert np.all(np.abs(out[0][0, :4]) == 200.0)


def test_batched_recorder_matches_single_env_csv(tmp_path):
    """BatchedStateControlRecorder rows of env k == StateControlRecorder rows of a single Env started from the same state."""
    import csv
    import torch
    import mujoco_template as mt

    model = load_model("cartpole")
    n, T = 8, 13
    qpos, qvel, _ = random_states(model, "cartpole", n, seed=61)

    class Push:
        capabilities = mt.ControllerCapabilities()
        def prepare(self, m, d): pass
        def __call__(self, m, d, t): d.ctrl[:] = 0.5

    benv = mt.BatchedEnv(model, n, controller=Push())
    benv.data.qpos.copy_(torch.as_tensor(qpos.T.copy(), device=benv.data.qpos.device))
    benv.data.qvel.copy_(torch.as_tensor(qvel.T.copy(), device=benv.data.qpos.device))
    path = tmp_path / "batched.csv"
    with mt.BatchedStateControlRecorder(benv, log_path=path, env_indices=[1, 5], chunk_steps=4, store_rows=True) as rec:
        steps = mt.run_passive_headless(benv, max_steps=T, hooks=rec, return_obs=False)
    assert steps == T and rec.steps == T and len(rec.rows) == 2 * T
    rows = list(csv.reader(open(path)))
    assert rows[0] == ["env", "time_s", "qpos[slider]", "qvel[slider]", "qpos[hinge]", "qvel[hinge]", "ctrl[cart_force]"]
    assert len(rows) == 1 + 2 * T
    for k in (1, 5):
        env = mt.Env(mt.ModelHandle(model), controller=Push())
        env.reset()
        env.data.qpos[:] = qpos[k]; env.data.qvel[:] = qvel[k]
        single = mt.StateControlRecorder(env)
        mt.run_passive_headless(env, max_steps=T, hooks=single, return_obs=False)
        mine = [r[1:] for r in rec.rows if r[0] == k]
        assert len(mine) == T
        for a, b in zip(mine, single.rows):
            assert np.allclose(np.array(a, dtype=float), np.array(b, dtype=float), rtol=0, atol=1e-13)


def test_batched_recorder_probe_columns_against_the_oracle(tmp_path):
    """Probe columns of the batched recorder (reference logging.py:175-176,241-242; the drone example's imu_x/y/z_m and
    goal_distance_m, examples/drone/drone_common.py:47-75): ArrayProbe columns ride in the recorder's gather launch,
    a callable probe is evaluated on tensors; with lazily stepped envs (return_obs=False) the derived arrays a probe
    reads are those of the step just taken.  Values against the oracle's site_xpos."""
    import torch
    import mujoco_template as mt
    from mujoco_template import _mj as mj

    model = load_model("drone")
    n, T = 6, 9
    qpos, qvel, _ = random_states(model, "drone", n, seed=62)
    imu = mj.mj_name2id(model, mj.mjtObj.mjOBJ_SITE, "imu")
    goal = np.array([5.0, -4.0, 2.3])

    class Hover:
        capabilities = mt.ControllerCapabilities()
        def prepare(self, m, d): pass
        def __call__(self, m, d, t): d.ctrl[:] = 3.4

    benv = mt.BatchedEnv(model, n, controller=Hover())
    dev = benv.data.qpos.device
    benv.data.qpos.copy_(torch.as_tensor(qpos.T.copy(), device=dev)); benv.data.qvel.copy_(torch.as_tensor(qvel.T.copy(), device=dev))
    benv.forward()
    sel = [0, 3, 4]
    goal_t = torch.as_tensor(goal, device=dev)

    def goal_distance(e, _result):
        p = e.data.site_xpos[3 * imu: 3 * imu + 3][:, sel]
        return (p - goal_t[:, None]).norm(dim=0)

    probes = [mt.ArrayProbe("imu_x_m", "site_xpos", 3 * imu), mt.ArrayProbe("imu_y_m", "site_xpos", 3 * imu + 1),
              mt.ArrayProbe("imu_z_m", "site_xpos", 3 * imu + 2), mt.DataProbe("goal_distance_m", goal_distance),
              mt.ArrayProbe("qacc_z", "qacc", 2)]
    with mt.BatchedStateControlRecorder(benv, log_path=tmp_path / "d.csv", env_indices=sel, chunk_steps=4, store_rows=True,
                                        probes=probes) as rec:
        mt.run_passive_headless(benv, max_steps=T, hooks=rec, return_obs=False)
    assert rec.columns[-5:] == ("imu_x_m", "imu_y_m", "imu_z_m", "goal_distance_m", "qacc_z")
    assert len(rec.rows) == len(sel) * T
    om, od = oracle_for(model)
    for k in sel:
        od.reset(); od.qpos[:] = qpos[k]; od.qvel[:] = qvel[k]; od.ctrl[:] = 3.4
        mine = [r for r in rec.rows if r[0] == k]
        for t in range(T):
            od.step()  # derived arrays of mj_step are those of the pre-integration forward pass (reference Appendix C.4)
            row = np.array(mine[t][1:], dtype=float)
            assert np.allclose(row[-5:-2], od.site_xpos[imu], rtol=0, atol=1e-11)
            assert abs(row[-2] - np.linalg.norm(od.site_xpos[imu] - goal)) < 1e-11
            assert abs(row[-1] - od.qacc[2]) < 1e-9 * max(1.0, abs(od.qacc[2]))
    with pytest.raises(mt.ConfigError):
        mt.BatchedStateControlRecorder(benv, probes=[mt.ArrayProbe("bad", "site_xpos", 999)])


@pytest.mark.parametrize("name,n", [("cartpole", 1000), ("pendulum", 33), ("drone", 70), ("cartpole-generic", 257)])
@pytest.mark.parametrize("precision", [64, 32])
def test_fused_control_tick_equals_three_launch_sequence(monkeypatch, name, n, precision):
    """b2_control_tick (control law evaluated inside the kernels; for Euler models the step rides in the FD launch and
    the derived arrays are produced lazily by b2_refresh_derived) == b2_lqr_control, b2_linearize, b2_step in sequence,
    and the FP64 result matches the oracle driven by the same control law."""
    import torch
    import mujoco_template as mt

    if name.endswith("-generic"):
        monkeypatch.setenv("B2_DISABLE_SPEC", "1")
        name = name.split("-")[0]
    model = load_model(name)
    euler = int(model.opt.integrator) == 0
    qpos, qvel, _ = random_states(model, name, n, seed=21)
    qref = np.array(model.key_qpos[0]) if name == "drone" else np.array(model.qpos0)
    uref = np.array(model.key_ctrl[0]) if name == "drone" else np.zeros(model.nu)
    if name == "cartpole":
        qpos[0] = [1.9995, 0.1]; qvel[0] = [3.0, 0.0]       # env 0 runs into the slider limit: constraint rows in the FD
    out = {}
    for fused in (True, False):
        ctl = mt.batched_controllers.BatchedLQRController(qpos_ref=qref, ctrl_ref=uref, Q=np.eye(2 * model.nv), R=np.eye(model.nu))
        benv = mt.BatchedEnv(model, n, controller=ctl, precision=precision)
        benv.fuse_control_tick = fused
        dev, dt = benv.data.qpos.device, benv.data.qpos.dtype
        benv.data.qpos.copy_(torch.as_tensor(qpos.T.copy(), device=dev, dtype=dt))
        benv.data.qvel.copy_(torch.as_tensor(qvel.T.copy(), device=dev, dtype=dt))
        c0 = mt._capi.launch_count()
        hist = []
        for s_ in range(5):
            res = benv.step(return_obs=False)
            if fused and euler:
                assert benv.data.backend.derived_stale      # nothing has read a derived array yet
            launches = mt._capi.launch_count()
            derived = (benv.data.qacc.clone(), benv.data.xpos.clone())   # first read materialises them (one forward launch)
            if fused and euler:
                assert mt._capi.launch_count() == launches + 1 and not benv.data.backend.derived_stale
            hist.append((res.info["A"].clone(), res.info["B"].clone(), benv.data.qpos.clone(), benv.data.qvel.clone(),
                         benv.data.ctrl.clone()) + derived)
        # FD(+step) + commit + lazy forward | FD + step | law + FD + step (+ the lazy forward: step(return_obs=False) on an
        # Euler model leaves the derived arrays to b2_refresh_derived as well -- BatchedEnv(derived="lazy"), the default)
        expect = 5 * (3 if euler else 2) if fused else (5 * 4 if euler else 5 * 3)
        assert mt._capi.launch_count() - c0 == expect
        out[fused] = hist
    tol = 1e-12 if precision == 64 else 2e-4
    for a, b in zip(out[True], out[False]):
        for k, (x, y) in enumerate(zip(a, b)):
            assert x.shape == y.shape
            if precision == 32 and k < 2:
                continue  # FP32 differences at eps = 1e-6 are rounding noise in either path
            # (A, B): rounding differences between the two kernels are amplified by 1/eps in the difference quotient
            bound = (1e-7 if k < 2 else tol) * max(1.0, float(y.abs().max()))
            assert float((x - y).abs().max()) <= bound, (k, float((x - y).abs().max()))
    if precision == 64:
        om, od = oracle_for(model)
        K = ctl.K
        for e in (0, 1, n - 1):
            od.reset(); od.qpos[:] = qpos[e]; od.qvel[:] = qvel[e]
            for s in range(5):
                x = np.concatenate([od.differentiate_pos(1.0, qref, np.array(od.qpos)), od.qvel])
                u = uref - K @ x
                lim = np.asarray(model.actuator_ctrllimited, bool)
                od.ctrl[:] = np.where(lim, np.clip(u, model.actuator_ctrlrange[:, 0], model.actuator_ctrlrange[:, 1]), u)
                Ao, Bo = od.transition_fd(1e-6, True)
                A, B, q, v, uu, _, _ = out[True][s]
                assert np.max(np.abs(A[e].cpu().numpy() - Ao)) <= 1e-6 * max(1.0, np.max(np.abs(Ao)))
                assert np.max(np.abs(B[e].cpu().numpy() - Bo)) <= 1e-6 * max(1.0, np.max(np.abs(Bo)))
                od.step()
                assert np.max(np.abs(q[:, e].cpu().numpy() - od.qpos)) <= 1e-9 * max(1.0, np.max(np.abs(od.qpos)))
                assert np.max(np.abs(v[:, e].cpu().numpy() - od.qvel)) <= 1e-9 * max(1.0, np.max(np.abs(od.qvel)))


SCENARIO_FIXTURES = ("pendulum_pd", "pendulum_passive", "cartpole_pid", "drone_lqr", "humanoid_lqr")


def _scenario(name):
    z = np.load(os.path.join(GOLDEN, f"scenario_{name}.npz"))
    return {k: z[k] for k in z.files}


@pytest.mark.parametrize("name", SCENARIO_FIXTURES)
def test_reference_scenario_every_step_in_one_launch(name):
    """The reference's example scenarios (its own PD / PID / LQR controllers run on the oracle-backed Env and recorded by
    tests/golden/make_scenario_golden.py: 400 .. 2000 steps each) through the CUDA path: env t of one batch starts from the
    recorded state before step t -- state, applied control and qacc_warmstart -- and a single b2_step launch must land every
    env on the recorded state after step t.  Covers the drone's whole point-to-point flight and the humanoid's balance, loss
    of balance and fall with its changing contacts."""
    import torch
    from mujoco_template import _mj as mj

    f = _scenario(name)
    model = load_model(str(f["model"]))
    n = int(f["steps"])
    q_before = np.vstack([f["qpos0"][None], f["qpos"][:-1]]); v_before = np.vstack([f["qvel0"][None], f["qvel"][:-1]])
    w_before = np.vstack([f["warm0"][None], f["warm"][:-1]])
    data = mj.BatchData(model, n)
    dev = data.qpos.device
    data.qpos.copy_(torch.as_tensor(q_before.T.copy(), device=dev)); data.qvel.copy_(torch.as_tensor(v_before.T.copy(), device=dev))
    data.qacc_warmstart.copy_(torch.as_tensor(w_before.T.copy(), device=dev))
    if model.nu:
        data.ctrl.copy_(torch.as_tensor(f["ctrl"].T.copy(), device=dev))
    mj.mj_step(model, data)
    torch.cuda.synchronize()
    assert int((data.flags != 0).sum()) == 0
    eq = np.abs(data.qpos.cpu().numpy().T - f["qpos"]) / np.maximum(1.0, np.abs(f["qpos"]))
    ev = np.abs(data.qvel.cpu().numpy().T - f["qvel"]) / np.maximum(1.0, np.abs(f["qvel"]))
    assert eq.max() <= 1e-9 and ev.max() <= 1e-9, (name, float(eq.max()), float(ev.max()), int(ev.max(axis=1).argmax()))


@pytest.mark.parametrize("name", SCENARIO_FIXTURES)
def test_reference_scenario_through_env_and_recorder(name, tmp_path):
    """The same scenarios driven the way the reference's harness drives them (runtime.py:303-410): `Env` on the CUDA path,
    `StateControlRecorder` CSV, `run_passive_headless(duration, max_steps)` -- with the recorded controls replayed by a
    controller.  Step counts follow the reference's loop-exit rule (801 for the drone's 8 s, 1201 for the humanoid's 6 s);
    the CSV header is the reference schema; rows match the recording while rounding differences stay small (the controls are
    replayed open loop and every controlled scenario sits at an unstable equilibrium: first 100 steps; the passive pendulum:
    the whole run).  test_reference_scenario_every_step_in_one_launch checks every step of every scenario to 1e-9."""
    import csv

    import mujoco_template as mt

    f = _scenario(name)
    model = load_model(str(f["model"]))
    ctrl = f["ctrl"]

    class Replay:
        capabilities = mt.ControllerCapabilities()
        k = 0
        def prepare(self, m, d): pass
        def __call__(self, m, d, t):
            if m.nu:
                d.ctrl[:] = ctrl[min(self.k, len(ctrl) - 1)]
            self.k += 1

    env = mt.Env(mt.ModelHandle(model), controller=Replay() if model.nu else None)
    env.reset()
    env.data.qpos[:] = f["qpos0"]; env.data.qvel[:] = f["qvel0"]
    if model.nu:
        env.data.ctrl[:] = f["ctrl0"]
    env.handle.forward()
    header = [str(h) for h in f["header"]]
    nprobe = len(header) - (1 + model.nq + model.nv + max(model.nu, 1))
    log = tmp_path / "log.csv"
    rec = mt.StateControlRecorder(env, log_path=log, store_rows=True)
    duration = None if np.isnan(f["duration"]) else float(f["duration"])
    max_steps = None if int(f["max_steps"]) < 0 else int(f["max_steps"])
    with rec:
        steps = mt.run_passive_headless(env, duration=duration, max_steps=max_steps, hooks=[rec])
    assert steps == int(f["steps"])
    with open(log) as fh:
        rows = list(csv.reader(fh))
    assert rows[0] == header[:len(header) - nprobe]
    got = np.array(rows[1:], dtype=float)
    ref = f["rows"][:, :got.shape[1]]
    n = steps if name == "pendulum_passive" else 100  # replayed controls are open loop: upright equilibria are unstable
    err = np.abs(got[:n] - ref[:n]) / np.maximum(1.0, np.abs(ref[:n]))
    assert err.max() <= 1e-7, (name, float(err.max()))


def test_dlqr_kernel_matches_scipy_dare():
    """b2_dlqr (doubling-iteration DARE + gain, one warp per env) == scipy.linalg.solve_discrete_are per system:
    cartpole and drone (A, B) from the oracle's FD at perturbed setpoints, and random stabilisable systems."""
    import torch
    from scipy.linalg import solve_discrete_are

    from conftest import load_model, oracle_for, random_states
    from mujoco_template.batched_controllers import batched_dlqr_gain

    for name, nsys in (("cartpole", 6), ("drone", 3)):
        model = load_model(name)
        om, od = oracle_for(model)
        qpos, qvel, ctrl = random_states(model, name, nsys, seed=4)
        As, Bs = [], []
        for e in range(nsys):
            od.reset()
            od.qpos[:] = qpos[e]; od.qvel[:] = 0.1 * qvel[e]; od.ctrl[:] = ctrl[e] if name == "drone" else 0.0
            A, B = od.transition_fd(1e-6, True)
            As.append(A); Bs.append(B)
        A, B = np.stack(As), np.stack(Bs)
        nx, nu = A.shape[1], B.shape[2]
        Q, R = np.diag(np.linspace(1.0, 3.0, nx)), 0.1 * np.eye(nu)
        K, P, status = batched_dlqr_gain(torch.as_tensor(A, device="cuda"), torch.as_tensor(B, device="cuda"), Q, R, return_status=True)
        assert int(status.min()) > 0 and int(status.max()) <= 40
        K, P = K.cpu(), P.cpu()
        for e in range(nsys):
            Pe = solve_discrete_are(A[e], B[e], Q, R)
            Ke = np.linalg.solve(R + B[e].T @ Pe @ B[e], B[e].T @ Pe @ A[e])
            assert np.max(np.abs(P[e].numpy() - Pe)) <= 1e-8 * np.max(np.abs(Pe)), (name, e)
            assert np.max(np.abs(K[e].numpy() - Ke)) <= 1e-8 * max(1.0, np.max(np.abs(Ke))), (name, e)
            assert np.max(np.abs(np.linalg.eigvals(A[e] - B[e] @ K[e].numpy()))) < 1.0
    rng = np.random.default_rng(0)
    A = rng.normal(0, 0.6, (32, 5, 5)); B = rng.normal(0, 1.0, (32, 5, 2))
    K, P = batched_dlqr_gain(torch.as_tensor(A, device="cuda"), torch.as_tensor(B, device="cuda"), np.eye(5), np.eye(2))
    K, P = K.cpu(), P.cpu()
    for e in range(32):
        Pe = solve_discrete_are(A[e], B[e], np.eye(5), np.eye(2))
        assert np.max(np.abs(P[e].numpy() - Pe)) <= 1e-8 * np.max(np.abs(Pe))

    # the humanoid's 54 x 54 system (one warp, 205 KB of shared memory): the reference's balance controller set-up
    model = load_model("humanoid")
    om, od = oracle_for(model)
    od.reset(1)
    od.forward()
    A, B = od.transition_fd(1e-6, True)
    Q = np.zeros((54, 54)); Q[:27, :27] = np.eye(27); Q[:6, :6] *= 10.0
    R = np.eye(21)
    K, P, status = batched_dlqr_gain(torch.as_tensor(A, device="cuda")[None], torch.as_tensor(B, device="cuda")[None], Q, R, return_status=True)
    Pe = solve_discrete_are(A, B, Q, R)
    Ke = np.linalg.solve(R + B.T @ Pe @ B, B.T @ Pe @ A)
    assert int(status[0]) > 0
    assert np.max(np.abs(P[0].cpu().numpy() - Pe)) <= 1e-6 * np.max(np.abs(Pe))
    assert np.max(np.abs(K[0].cpu().numpy() - Ke)) <= 1e-6 * np.max(np.abs(Ke))
    # and straight from a BatchedEnv's linearisation: info['A'] / info['B'] are views of the kernel's input layout
    import mujoco_template as mt
    from mujoco_template.batched_controllers import BatchedLQRController

    cart = load_model("cartpole")
    ctl = BatchedLQRController(Q=np.diag([10.0, 100.0, 1.0, 1.0]), R=np.array([[0.01]]))
    env = mt.BatchedEnv(cart, 64, controller=ctl)
    env.reset()
    res = env.step()
    Kb, Pb = batched_dlqr_gain(res.info["A"], res.info["B"], np.diag([10.0, 100.0, 1.0, 1.0]), np.array([[0.01]]))
    assert tuple(Kb.shape) == (64, 1, 4)
    assert np.allclose(Kb[0].cpu().numpy(), ctl.K, rtol=1e-6, atol=1e-8)  # env 0 sits at the controller's setpoint
    # a large batch right behind the FD kernel (whatever that left in shared memory must not matter: the first version of
    # the kernel multiplied its uninitialised product buffers by zero, which failed 0.1 % of the envs of a 65,536 batch)
    from mujoco_template import _mj as mj

    drone = load_model("drone")
    n = 32768
    qpos, qvel, _ = random_states(drone, "drone", 4096, seed=8)
    d = mj.BatchData(drone, n)
    d.qpos.copy_(torch.as_tensor(np.tile(qpos, (8, 1)).T.copy(), device="cuda")); d.qvel.copy_(torch.as_tensor(np.tile(qvel, (8, 1)).T.copy(), device="cuda"))
    d.ctrl.fill_(3.2495625)
    for _ in range(3):
        A, B = d.backend.linearize(1e-6, True)
        Kd, Pd, st = batched_dlqr_gain(A.permute(2, 0, 1), B.permute(2, 0, 1), np.eye(12), np.eye(4), return_status=True)
        assert int((st <= 0).sum()) == 0 and bool(torch.isfinite(Kd).all()) and bool(torch.isfinite(Pd).all())
    assert torch.equal(Kd[:4096], Kd[4096:8192])  # tiled states: identical gains, whichever warp / block computed them


def test_time_varying_lqr_resynthesises_every_tick_and_stabilises():
    """BatchedTVLQRController: every tick, every env's gain from its own latest (A, B) (b2_dlqr, the thread-per-env kernel for
    the 4 x 1 cartpole) applied by b2_lqr_control_env.  Checked against scipy's DARE on the same (A, B), against the oracle
    for the applied control, and by its effect: 4,096 cartpoles from the config's initial states end upright."""
    import torch
    from scipy.linalg import solve_discrete_are

    import mujoco_template as mt
    from mujoco_template.batched_controllers import BatchedTVLQRController

    model = load_model("cartpole")
    n = 4096
    Q, R = np.diag([10.0, 100.0, 1.0, 1.0]), np.array([[0.01]])
    ctl = BatchedTVLQRController(Q=Q, R=R)
    env = mt.BatchedEnv(model, n, controller=ctl)
    env.reset()
    qpos, qvel, _ = random_states(model, "cartpole", n, seed=3)
    dev = env.data.qpos.device
    env.data.qpos.copy_(torch.as_tensor(qpos.T.copy(), device=dev)); env.data.qvel.copy_(torch.as_tensor(qvel.T.copy(), device=dev))
    env.forward()
    res = env.step()                                   # tick 0: setpoint gain, produces (A0, B0)
    A0, B0 = res.info["A"].clone(), res.info["B"].clone()
    q1, v1 = env.data.qpos.clone(), env.data.qvel.clone()
    env.step()                                         # tick 1: gains from (A0, B0), applied to the state after tick 0
    K, P, status = ctl.gains
    assert int(status.min()) > 0
    u1 = env.data.ctrl.clone()
    for e in (0, 17, n - 1):
        Ae, Be = A0[e].cpu().numpy(), B0[e].cpu().numpy()
        Pe = solve_discrete_are(Ae, Be, Q, R)
        Ke = np.linalg.solve(R + Be.T @ Pe @ Be, Be.T @ Pe @ Ae)
        assert np.max(np.abs(K[e].cpu().numpy() - Ke)) <= 1e-8 * np.max(np.abs(Ke))
        x = np.concatenate([q1[:, e].cpu().numpy() - model.qpos0, v1[:, e].cpu().numpy()])
        u = float(np.clip(-(Ke @ x)[0], model.actuator_ctrlrange[0, 0], model.actuator_ctrlrange[0, 1]))
        assert abs(float(u1[0, e]) - u) <= 1e-7 * max(1.0, abs(u))
    assert float((K - torch.as_tensor(ctl.K, device=dev)).abs().max()) > 1e-3     # the gains do differ from the setpoint gain
    env.enable_cuda_graph(True)                          # the whole tick (DARE, law, FD, step) replays as one graph
    for _ in range(600):
        env.step(return_obs=False)
    torch.cuda.synchronize()
    assert int((env.data.flags != 0).sum()) == 0
    assert float(env.data.qpos[1].abs().max()) < 1e-3 and float(env.data.qvel.abs().max()) < 1e-2
