"""Host model compiler: MJCF subset -> compiled model (CPU only)."""
import os
import warnings

import numpy as np
import pytest

from conftest import GOLDEN, MODEL_NAMES, load_model

REF = os.environ.get("B2_REFERENCE", "")  # checkout of the original mujoco-template project
REF_XML = {"pendulum": "examples/pendulum/pendulum.xml", "cartpole": "examples/cartpole/cartpole.xml",
           "drone": "examples/drone/scene.xml", "humanoid": "examples/humanoid/humanoid.xml"}

ARM_XML = """
<mujoco model="two-link">
  <compiler angle="degree"/>
  <option timestep="0.004" integrator="RK4"/>
  <default>
    <joint damping="0.3"/>
    <default class="thin"><geom size="0.02"/></default>
  </default>
  <worldbody>
    <geom name="ground" type="plane" size="2 2 .1"/>
    <body name="upper" pos="0 0 1" childclass="thin">
      <joint name="shoulder" type="hinge" axis="0 1 0" range="-90 90"/>
      <geom name="upper_g" type="capsule" fromto="0 0 0 0 0 -0.4"/>
      <body name="lower" pos="0 0 -0.4">
        <joint name="elbow" type="hinge" axis="0 1 0" limited="false" range="-10 10" stiffness="2" springref="15"/>
        <geom name="lower_g" type="capsule" fromto="0 0 0 0 0 -0.3" size="0.03" density="500"/>
        <site name="hand" pos="0 0 -0.3"/>
      </body>
    </body>
  </worldbody>
  <actuator>
    <motor name="m0" joint="shoulder" gear="5" ctrlrange="-1 1"/>
    <position name="p1" joint="elbow" kp="20"/>
  </actuator>
  <keyframe><key name="bent" qpos="0.3 -0.5" ctrl="0.1 0.2"/></keyframe>
</mujoco>
"""


def test_two_link_arm_compiles_with_expected_structure():
    from mujoco_template import _mj as mj

    m = mj.MjModel.from_xml_string(ARM_XML)
    assert (m.nq, m.nv, m.nu, m.nbody, m.njnt, m.ngeom, m.nsite, m.nkey) == (2, 2, 2, 3, 2, 3, 1, 1)
    assert m.opt.timestep == 0.004 and m.opt.integrator == 1
    assert list(m.body_parentid) == [0, 0, 1] and list(m.dof_parentid) == [-1, 0]
    assert list(m.jnt_limited) == [1, 0]                      # autolimits: range => limited; explicit false wins
    assert np.allclose(m.jnt_range[0], np.deg2rad([-90, 90]))  # degrees -> radians for hinges
    assert np.isclose(m.qpos_spring[1], np.deg2rad(15)) and m.jnt_stiffness[1] == 2
    assert np.allclose(m.dof_damping, 0.3)
    # capsule from 'fromto': half-length, centre, and mass = density * (cylinder + sphere)
    r, half = 0.02, 0.2
    assert np.allclose(m.geom_size[1][:2], [r, half]) and np.allclose(m.geom_pos[1], [0, 0, -0.2])
    vol = np.pi * r * r * 2 * half + 4 / 3 * np.pi * r ** 3
    assert np.isclose(m.body_mass[1], 1000 * vol)
    assert np.allclose(m.body_ipos[1], [0, 0, -0.2])
    # actuators: motor gear/ctrlrange (autolimits), position servo -> affine bias
    assert np.allclose(m.actuator_gear[0][0], 5) and list(m.actuator_ctrllimited) == [1, 0]
    assert np.allclose(m.actuator_gainprm, [1, 20]) and np.allclose(m.actuator_biasprm[1], [0, -20, 0])
    assert np.allclose(m.key_qpos[0], [0.3, -0.5]) and np.allclose(m.key_ctrl[0], [0.1, 0.2])
    # collision candidates: plane vs both capsules; parent-child capsule pair filtered
    pairs = sorted(zip(m._c["pair_geom1"].tolist(), m._c["pair_geom2"].tolist()))
    assert pairs == [(0, 1), (0, 2)]
    assert mj.mj_name2id(m, mj.mjtObj.mjOBJ_SITE, "hand") == 0 and mj.mj_name2id(m, mj.mjtObj.mjOBJ_BODY, "nope") == -1
    assert m.body("lower").id == 2 and m.joint(1).name == "elbow"


def test_example_model_dimensions():
    dims = {"pendulum": (1, 1, 1, 2), "cartpole": (2, 2, 1, 3), "drone": (7, 6, 4, 2), "humanoid": (28, 27, 21, 17)}
    for name in MODEL_NAMES:
        m = load_model(name)
        assert (m.nq, m.nv, m.nu, m.nbody) == dims[name]
    h = load_model("humanoid")
    assert h.ntendon == 2 and h.nkey == 4 and h.njnt == 22 and h.ngeom == 20
    assert abs(h.body_mass.sum() - 40.844) < 1e-2       # the standard DeepMind humanoid
    assert h.names["key"] == ["squat", "stand_on_left_leg", "prone", "supine"]
    # free joint takes no class defaults (armature/damping stay 0), hinges do
    assert np.all(h.dof_armature[:6] == 0) and np.all(h.dof_armature[6:] == 0.01)
    d = load_model("drone")
    assert np.allclose(d.actuator_gear[:, 2], 1) and np.allclose(np.abs(d.actuator_gear[:, 5]), 0.11)
    assert d.opt.density == 1.225 and d._c["has_fluid"] == 1 and d.ngeom == 11 and d.nsite == 5


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "examples")),
                    reason="needs a checkout of the original mujoco-template project (B2_REFERENCE)")
@pytest.mark.parametrize("name", MODEL_NAMES)
def test_committed_model_files_match_a_fresh_compile(name):
    from mujoco_template import _mj as mj

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        fresh = mj.MjModel.from_xml_path(os.path.join(REF, REF_XML[name]))
    assert fresh.blob == load_model(name).blob


def test_unsupported_features_fail_loudly():
    from mujoco_template import ConfigError
    from mujoco_template import _mj as mj

    bad = [
        '<mujoco><option integrator="implicit"/><worldbody/></mujoco>',
        '<mujoco><option cone="elliptic"/><worldbody/></mujoco>',
        '<mujoco><worldbody><body><joint type="ball"/><geom size=".1"/></body></worldbody></mujoco>',
        '<mujoco><worldbody><body><joint/><geom type="box" size=".1 .1 .1"/></body><body pos="1 0 0"><joint/>'
        '<geom type="box" size=".1 .1 .1"/></body></worldbody></mujoco>',   # box-box needs a convex collider
        '<mujoco><worldbody><body><joint/></body></worldbody></mujoco>',      # moving body without mass
        '<mujoco><worldbody><body><joint/><geom size=".1"/></body></worldbody><equality><weld body1="world"/></equality></mujoco>',
    ]
    for xml in bad:
        with pytest.raises(ConfigError):
            mj.MjModel.from_xml_string(xml)
    with pytest.raises(ConfigError):
        mj.MjModel.from_xml_path("/nonexistent/model.xml")


def test_compiled_model_roundtrip(tmp_path):
    from mujoco_template import _mj as mj

    m = mj.MjModel.from_xml_string(ARM_XML)
    path = tmp_path / "arm.b2m"
    m.save_compiled(str(path))
    m2 = mj.MjModel.from_compiled(str(path))
    assert m2.blob == m.blob and m2.names == m.names


def test_sensor_compilation_and_unsupported_kinds():
    from mujoco_template import ConfigError
    from mujoco_template import _mj as mj
    from test_oracle_analytic import SENSOR_XML

    m = mj.MjModel.from_xml_string(SENSOR_XML.format(dt=0.002))
    assert m.nsensor == 15 and list(m.sensor_adr[:4]) == [0, 1, 2, 5] and m.sensor_cutoff[-1] == 5.0
    assert mj.mj_name2id(m, mj.mjtObj.mjOBJ_SENSOR, "gyro") == 9 and mj.mj_id2name(m, mj.mjtObj.mjOBJ_SENSOR, 0) == "s_pos"
    drone = load_model("drone")
    assert drone.nsensordata == 10 and drone.names["sensor"] == ["body_gyro", "body_linacc", "body_quat"]
    base = '<mujoco><worldbody><body name="b"><joint name="j"/><geom size=".1"/><site name="s"/></body></worldbody><sensor>{}</sensor></mujoco>'
    for bad in ('<touch site="s"/>', '<framepos objtype="site" objname="s" reftype="body" refname="b"/>',
                '<jointpos joint="nope"/>', '<framequat objtype="camera" objname="s"/>'):
        with pytest.raises(ConfigError):
            mj.MjModel.from_xml_string(base.format(bad))
