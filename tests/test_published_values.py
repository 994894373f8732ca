"""Known answers published with the real engine's output.

The reference ships DeepMind's LQR tutorial as source text only (``LQR.txt`` of the original mujoco-template project; ``LQR.txt:158-163``
``mujoco.mj_inverse(model, data); print(data.qfrc_inverse)``, ``:165-205`` the height sweep and ``print('desired forces:',
qfrc0)``).  The tutorial notebook as published upstream (mujoco/python/LQR.ipynb) carries the output cells of exactly
these statements, produced by MuJoCo itself on the humanoid model the reference uses (``examples/humanoid/humanoid.xml``,
keyframe 1 ``stand_on_left_leg``).  The vectors below are quoted from that published output (``np.set_printoptions(precision=3)``:
three decimals).  They were written down BEFORE the oracle was run on the case -- every printed digit matched -- and they
are the only numbers in this repo that come from a run of the real engine:

* ``qfrc_inverse`` for ``qacc = 0`` at the keyframe: the humanoid's weight (400.68 N) minus what its four penetrating foot
  contacts push back at that penetration, and the joint torques that hold the pose.  The entry pins the MJCF compile
  (masses and inertias from the geoms, keyframe), kinematics, the bias forces of a 27-dof tree, contact detection and
  the whole row construction of the constraint stage (impedance, ``aref``, pyramidal ``R`` from ``solref`` / ``solimp`` /
  ``invweight0``), through ``mj_inverse``'s per-row force law.
* the height offset at which the vertical force vanishes (the title of the tutorial's plot) and the leading entries of
  ``desired forces`` at that offset.

What they do not pin: the Newton solver's iterates (``mj_inverse`` needs no solve) and the integrators.
"""
import numpy as np
import pytest

from conftest import load_model, oracle_for

QFRC_INVERSE_AT_KEYFRAME = np.array([
    0.0, 0.0, 275.879, -33.186, 4.995, -6.688, -4.305, 3.693, -15.451, -10.906, 0.412, -1.613, -9.793, -2.312,
    -0.366, -5.913, -0.417, -1.914, 5.759, 2.665, -0.202, -5.755, 0.994, 1.141, -1.987, 3.821, 1.151])
BEST_OFFSET_MM = -0.5070
DESIRED_FORCES_HEAD = np.array([0.0, 0.0, -0.191, -3.447, 0.222, -0.817, 2.586, 14.637, -18.64])
PRINTED = 5.1e-4  # half a unit of the third printed decimal


def test_oracle_humanoid_inverse_dynamics_equals_the_published_tutorial_output():
    model = load_model("humanoid")
    om, od = oracle_for(model)
    od.reset(1)
    od.forward()
    qfrc = od.inverse(np.zeros(model.nv))
    assert od.ncon == 4
    assert np.max(np.abs(qfrc - QFRC_INVERSE_AT_KEYFRAME)) < PRINTED, qfrc
    offsets = np.linspace(-0.001, 0.001, 2001)
    force = []
    for off in offsets:
        od.reset(1); od.forward(); od.qpos[2] += off
        force.append(od.inverse(np.zeros(model.nv))[2])
    best = offsets[int(np.argmin(np.abs(force)))]
    assert abs(best * 1000 - BEST_OFFSET_MM) < 1e-9
    od.reset(1); od.forward(); od.qpos[2] += best
    desired = od.inverse(np.zeros(model.nv))
    assert np.max(np.abs(desired[:9] - DESIRED_FORCES_HEAD)) < PRINTED, desired[:9]
    assert np.max(np.abs(desired[9:15] - QFRC_INVERSE_AT_KEYFRAME[9:15])) < PRINTED   # right leg and arms: untouched by the offset
    assert np.max(np.abs(desired[21:] - QFRC_INVERSE_AT_KEYFRAME[21:])) < PRINTED


@pytest.mark.gpu
def test_cuda_humanoid_inverse_dynamics_equals_the_published_tutorial_output():
    """The same statements through the drop-in's mujoco-shaped API on the CUDA path (b2_forward / b2_inverse)."""
    from mujoco_template import _mj as mj

    model = load_model("humanoid")
    data = mj.MjData(model)
    mj.mj_resetDataKeyframe(model, data, 1)
    mj.mj_forward(model, data)
    data.qacc[:] = 0.0
    mj.mj_inverse(model, data)
    assert np.max(np.abs(np.array(data.qfrc_inverse) - QFRC_INVERSE_AT_KEYFRAME)) < PRINTED
    mj.mj_resetDataKeyframe(model, data, 1)
    mj.mj_forward(model, data)
    data.qacc[:] = 0.0
    data.qpos[2] += BEST_OFFSET_MM * 1e-3
    mj.mj_inverse(model, data)
    assert np.max(np.abs(np.array(data.qfrc_inverse)[:9] - DESIRED_FORCES_HEAD)) < PRINTED
