"""Live parity against a real MuJoCo, wherever one is installed (SURVEY.md 8c pin 4).

Without the ``mujoco`` package this module is skipped and the oracle stays "parity unpinned".  On any machine with
``pip install mujoco`` (>= 3.1) it pins the oracle -- and therefore the CUDA path, which the GPU tests hold to the
oracle -- to upstream: model constants from our MJCF compiler, per-step trajectories, mjd_transitionFD, Jacobians,
sensors and inverse dynamics, on inline models and (when ``B2_REFERENCE`` names a checkout of the original
mujoco-template project) on the four example models.
"""
import os
import warnings

import numpy as np
import pytest

mujoco = pytest.importorskip("mujoco")

from conftest import oracle_for  # noqa: E402
from test_host_logic import BASE_XML  # noqa: E402
from test_mjcf_compiler import ARM_XML  # noqa: E402
from test_oracle_analytic import SENSOR_XML  # noqa: E402

REF = os.environ.get("B2_REFERENCE", "")
EXAMPLES = {
    "pendulum": "examples/pendulum/pendulum.xml", "cartpole": "examples/cartpole/cartpole.xml",
    "drone": "examples/drone/scene.xml", "humanoid": "examples/humanoid/humanoid.xml",
}
INLINE = {"fixture": BASE_XML, "arm": ARM_XML, "sensor_rig": SENSOR_XML.format(dt=0.002)}


def _ours_from(kind, key):
    from mujoco_template import _mj as mj

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return mj.MjModel.from_xml_string(INLINE[key]) if kind == "inline" else mj.MjModel.from_xml_path(os.path.join(REF, EXAMPLES[key]))


def _theirs_from(kind, key):
    return mujoco.MjModel.from_xml_string(INLINE[key]) if kind == "inline" else mujoco.MjModel.from_xml_path(os.path.join(REF, EXAMPLES[key]))


CASES = [("inline", k) for k in INLINE] + [("example", k) for k in EXAMPLES]


def _skip_missing(kind, key):
    if kind == "example" and not os.path.exists(os.path.join(REF, EXAMPLES[key])):
        pytest.skip("reference tree not present")


def _rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b))))) if a.size else 0.0


@pytest.mark.parametrize("kind,key", CASES)
def test_compiled_constants_match_upstream(kind, key):
    _skip_missing(kind, key)
    ours, theirs = _ours_from(kind, key), _theirs_from(kind, key)
    for dim in ("nq", "nv", "nu", "nbody", "njnt", "ngeom", "nsite", "nsensordata"):
        assert getattr(ours, dim) == getattr(theirs, dim), dim
    for field in ("body_mass", "body_inertia", "body_pos", "body_quat", "body_ipos", "body_iquat", "body_subtreemass",
                  "body_invweight0", "dof_invweight0", "dof_damping", "dof_armature", "jnt_range", "jnt_stiffness",
                  "qpos0", "qpos_spring", "geom_size", "geom_pos", "geom_quat", "site_pos", "site_quat",
                  "actuator_ctrlrange", "actuator_forcerange"):
        assert _rel(getattr(ours, field), getattr(theirs, field)) <= 1e-12, field
    assert abs(ours.stat.meaninertia - theirs.stat.meaninertia) <= 1e-12 * max(1.0, theirs.stat.meaninertia)


@pytest.mark.parametrize("kind,key", CASES)
def test_trajectory_linearisation_sensors_match_upstream(kind, key):
    _skip_missing(kind, key)
    ours, theirs = _ours_from(kind, key), _theirs_from(kind, key)
    om, od = oracle_for(ours)
    md = mujoco.MjData(theirs)
    rng = np.random.default_rng(0)
    if theirs.nkey:
        mujoco.mj_resetDataKeyframe(theirs, md, 0)
        od.reset(0)
    nv, nu = theirs.nv, theirs.nu
    dv = 0.05 * rng.normal(size=nv)
    md.qvel[:] += dv; od.qvel[:] += dv
    lo = np.where(theirs.actuator_ctrllimited, theirs.actuator_ctrlrange[:, 0], -1.0) if nu else np.zeros(0)
    hi = np.where(theirs.actuator_ctrllimited, theirs.actuator_ctrlrange[:, 1], 1.0) if nu else np.zeros(0)
    for step in range(200):
        if nu:
            u = md.ctrl + 0.1 * (hi - lo) * rng.uniform(-1, 1, nu) if step else 0.5 * (lo + hi) + 0.0 * lo
            u = np.clip(u, lo, hi)
            md.ctrl[:] = u; od.ctrl[:] = u
        if step % 50 == 0:
            A = np.zeros((2 * nv, 2 * nv)); B = np.zeros((2 * nv, nu))
            mujoco.mjd_transitionFD(theirs, md, 1e-6, True, A, B, None, None)
            Ao, Bo = od.transition_fd(1e-6, True)
            assert _rel(Ao, A) <= 1e-6 and _rel(Bo, B) <= 1e-6, step
        mujoco.mj_step(theirs, md)
        od.step()
        assert _rel(od.qpos, md.qpos) <= 1e-9 and _rel(od.qvel, md.qvel) <= 1e-9, step
        assert od.ncon == md.ncon, step
        if theirs.nsensordata:
            assert _rel(od.sensordata, md.sensordata) <= 1e-9, step
    mujoco.mj_forward(theirs, md); od.forward()
    assert _rel(od.xpos, md.xpos) <= 1e-10 and _rel(od.subtree_com, md.subtree_com) <= 1e-10
    assert _rel(od.qfrc_bias, md.qfrc_bias) <= 1e-9 and _rel(od.qacc, md.qacc) <= 1e-8
    for b in range(1, theirs.nbody):
        jp, jr = np.zeros((3, nv)), np.zeros((3, nv))
        mujoco.mj_jacBody(theirs, md, jp, jr, b)
        jpo, jro = od.jac("body", b)
        assert _rel(jpo, jp) <= 1e-10 and _rel(jro, jr) <= 1e-10
        mujoco.mj_jacSubtreeCom(theirs, md, jp, b)
        assert _rel(od.jac("subtreecom", b)[0], jp) <= 1e-10
    md.qacc[:] = 0.1 * rng.normal(size=nv)
    mujoco.mj_inverse(theirs, md)
    assert _rel(od.inverse(np.array(md.qacc)), md.qfrc_inverse) <= 1e-8
