"""Sensor Jacobians of mjd_transitionFD (C = d sensordata / dx, D = d sensordata / du) on the CPU oracle, checked against
identities that do not come from the finite differences: state readings, point Jacobians, the site frame, the cutoff
clip and the ctrlrange rules.  The GPU tests hold b2_linearize_sensors to this reference."""
import os
import warnings

import numpy as np
import pytest

from conftest import load_model, oracle_for, random_states
from sensor_fd_reference import transition_fd_sensors
from test_oracle_analytic import SENSOR_XML

EPS = 1e-6
JAC_ATOL = 1e-7  # centred differences of smooth functions at eps = 1e-6: truncation and rounding well below this


def sensor_rig(integrator: str = "Euler"):
    from mujoco_template import _mj as mj

    xml = SENSOR_XML.format(dt=0.002)
    if integrator == "RK4":
        xml = xml.replace("<option ", '<option integrator="RK4" ')
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return mj.MjModel.from_xml_string(xml)


def rows(model, name):
    i = model.names["sensor"].index(name)
    return slice(int(model.sensor_adr[i]), int(model.sensor_adr[i] + model.sensor_dim[i]))


def rig_state(od, seed=5):
    rng = np.random.default_rng(seed)
    od.qpos[:3] = rng.uniform(-0.5, 0.5, 3)
    q = rng.normal(size=4)
    od.qpos[6:10] = q / np.linalg.norm(q)
    od.qvel[:] = rng.normal(size=od.qvel.size)
    od.ctrl[:] = [0.3, -0.2]


@pytest.mark.parametrize("integrator", ["Euler", "RK4"])
def test_rig_sensor_jacobians_against_identities(integrator):
    model = sensor_rig(integrator)
    assert model.opt.integrator == (1 if integrator == "RK4" else 0)
    nv = model.nv
    om, od = oracle_for(model)
    rig_state(od)
    q0, v0, w0 = od.qpos.copy(), od.qvel.copy(), od.qacc_warmstart.copy()
    C, D = transition_fd_sensors(model, od, EPS, True)
    assert C.shape == (model.nsensordata, 2 * nv) and D.shape == (model.nsensordata, model.nu)
    # the state is restored
    assert np.array_equal(od.qpos, q0) and np.array_equal(od.qvel, v0) and np.array_equal(od.qacc_warmstart, w0)
    od.forward()  # nominal kinematics for the Jacobians below
    # jointpos / jointvel: unit rows of the position / velocity block
    unit = np.zeros(2 * nv)
    unit[model.jnt_dofadr[model.names["joint"].index("slide")]] = 1
    assert np.allclose(C[rows(model, "s_pos")][0], unit, atol=JAC_ATOL)
    unit = np.zeros(2 * nv)
    unit[nv + model.jnt_dofadr[model.names["joint"].index("twist")]] = 1
    assert np.allclose(C[rows(model, "s_vel")][0], unit, atol=JAC_ATOL)
    # framepos: the point Jacobian at the nominal state; no dependence on the velocity
    probe = model.names["body"].index("probe")
    for name, (kind, obj) in {"p_site": ("site", 0), "p_xbody": ("body", probe), "p_body": ("bodycom", probe)}.items():
        jacp, _ = od.jac(kind, obj)
        assert np.allclose(C[rows(model, name), :nv], jacp, atol=JAC_ATOL), name
        assert np.all(C[rows(model, name), nv:] == 0), name
    # gyro / velocimeter: the site-frame angular / linear velocity is R_site' jac qvel, linear in qvel
    for site, (gyro, velo) in enumerate((("gyro", "velo"), ("gyro2", "velo2"))):
        jacp, jacr = od.jac("site", site)
        R = od.site_xmat[site].reshape(3, 3)
        assert np.allclose(C[rows(model, gyro), nv:], R.T @ jacr, atol=JAC_ATOL), gyro
        assert np.allclose(C[rows(model, velo), nv:], R.T @ jacp, atol=JAC_ATOL), velo
    # only the accelerometers see the controls (the other readings precede the step's integration)
    acc = np.zeros(model.nsensordata, bool)
    acc[rows(model, "acc")] = acc[rows(model, "acc2")] = True
    assert np.all(D[~acc] == 0)
    assert np.max(np.abs(D[rows(model, "acc")])) > 1e-3


def test_cutoff_clips_the_accelerometer_rows():
    """acc2 (cutoff 5): a component held at the clip does not move under any perturbation -- its rows are zero -- while the
    unclipped components keep their derivatives."""
    model = sensor_rig()
    om, od = oracle_for(model)
    rig_state(od)
    od.qvel[6:9] = [0.0, 0.0, 12.0]   # fast spin of the floater: centripetal acceleration at imu2 well above 5
    od.qvel[3:6] = [2.0, -1.0, 0.5]
    od.forward()
    a = od.sensordata[rows(model, "acc2")].copy()
    clipped = np.abs(a) == 5.0
    assert clipped.any() and not clipped.all(), a
    C, D = transition_fd_sensors(model, od, EPS, True)
    r = np.arange(model.nsensordata)[rows(model, "acc2")]
    assert np.all(C[r[clipped]] == 0) and np.all(D[r[clipped]] == 0)
    assert np.all(np.max(np.abs(C[r[~clipped]]), axis=1) > 1e-3)


def test_drone_sensor_jacobians_and_ctrlrange_columns():
    """Drone IMU (gyro, accelerometer, framequat): gyro = R_site' jacr qvel; only the accelerometer sees the controls; the
    thrust map is affine, so a one-sided column at a ctrlrange bound equals the centred column inside the range, and a
    control outside the range has a zero column, as in B."""
    model = load_model("drone")
    nv = model.nv
    om, od = oracle_for(model)
    qpos, qvel, ctrl = random_states(model, "drone", 1, seed=11)
    od.qpos[:] = qpos[0]; od.qvel[:] = qvel[0]; od.ctrl[:] = [6.0, 6.5, 7.0, 7.5]
    C_in, D_in = transition_fd_sensors(model, od, EPS, True)
    od.forward()
    jacp, jacr = od.jac("site", 0)
    R = od.site_xmat[0].reshape(3, 3)
    assert np.allclose(C_in[rows(model, "body_gyro"), nv:], R.T @ jacr, atol=JAC_ATOL)
    assert np.all(D_in[rows(model, "body_gyro")] == 0) and np.all(D_in[rows(model, "body_quat")] == 0)
    assert np.max(np.abs(D_in[rows(model, "body_linacc")])) > 1e-2
    od.ctrl[:] = [0.0, 13.0, 14.0, 7.5]  # lower bound: forward, upper bound: backward, outside: no column
    C_b, D_b = transition_fd_sensors(model, od, EPS, True)
    assert np.allclose(D_b[:, :2], D_in[:, :2], rtol=1e-6, atol=1e-8)
    assert np.all(D_b[:, 2] == 0)
    assert np.allclose(D_b[:, 3], D_in[:, 3], rtol=1e-6, atol=1e-8)
    # one-sided everywhere (centered = False): the same columns to first order
    C_f, D_f = transition_fd_sensors(model, od, EPS, False)
    assert np.allclose(D_f, D_b, rtol=1e-5, atol=1e-6)


REF = os.environ.get("B2_REFERENCE", "")
DRONE_XML = os.path.join(REF, "examples/drone/scene.xml")


@pytest.mark.parametrize("case", ["rig_euler", "rig_rk4", "drone"])
def test_sensor_jacobians_match_upstream(case):
    """C / D against upstream mjd_transitionFD wherever the mujoco package is installed (the drone also needs
    B2_REFERENCE, a checkout of the original mujoco-template project)."""
    mujoco = pytest.importorskip("mujoco")
    from mujoco_template import _mj as mj

    if case == "drone":
        if not os.path.exists(DRONE_XML):
            pytest.skip("reference tree not present")
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ours = mj.MjModel.from_xml_path(DRONE_XML)
        theirs = mujoco.MjModel.from_xml_path(DRONE_XML)
    else:
        ours = sensor_rig("RK4" if case == "rig_rk4" else "Euler")
        xml = SENSOR_XML.format(dt=0.002)
        theirs = mujoco.MjModel.from_xml_string(xml.replace("<option ", '<option integrator="RK4" ') if case == "rig_rk4" else xml)
    om, od = oracle_for(ours)
    md = mujoco.MjData(theirs)
    if theirs.nkey:
        mujoco.mj_resetDataKeyframe(theirs, md, 0)
        od.reset(0)
    rng = np.random.default_rng(1)
    dv = 0.05 * rng.normal(size=theirs.nv)
    md.qvel[:] += dv; od.qvel[:] += dv
    if theirs.nu:
        u = rng.uniform(0, 1, theirs.nu) if case != "drone" else np.array([0.0, 13.0, 6.0, 7.0])
        md.ctrl[:] = u; od.ctrl[:] = u
    nx, ns, nu = 2 * theirs.nv, theirs.nsensordata, theirs.nu
    A, B, C, D = np.zeros((nx, nx)), np.zeros((nx, nu)), np.zeros((ns, nx)), np.zeros((ns, nu))
    mujoco.mjd_transitionFD(theirs, md, EPS, True, A, B, C, D)
    Co, Do = transition_fd_sensors(ours, od, EPS, True)
    scale = max(1.0, float(np.max(np.abs(C))), float(np.max(np.abs(D))) if D.size else 0.0)
    assert np.max(np.abs(Co - C)) <= 1e-6 * scale and (not D.size or np.max(np.abs(Do - D)) <= 1e-6 * scale)
