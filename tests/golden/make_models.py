"""Generate tests/golden/models/*.b2m from the reference's example MJCF files.

Needs a checkout of the original mujoco-template project:
    B2_REFERENCE=<checkout> python tests/golden/make_models.py
Tests, smoke() and bench.py load these compiled-model files instead of the XML, so they run
without that checkout.  They are derived artefacts of OUR compiler.
"""
import os
import sys
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "mujoco-template_b200"))
from mujoco_template import _mj as mj  # noqa: E402

REF = os.environ.get("B2_REFERENCE", "")
MODELS = {
    "pendulum": "examples/pendulum/pendulum.xml",
    "cartpole": "examples/cartpole/cartpole.xml",
    "drone": "examples/drone/scene.xml",
    "humanoid": "examples/humanoid/humanoid.xml",
}

if __name__ == "__main__":
    out = os.path.join(ROOT, "tests", "golden", "models")
    os.makedirs(out, exist_ok=True)
    warnings.simplefilter("ignore")
    for name, rel in MODELS.items():
        m = mj.MjModel.from_xml_path(os.path.join(REF, rel))
        m.save_compiled(os.path.join(out, f"{name}.b2m"))
        print(name, "nq", m.nq, "nv", m.nv, "nu", m.nu, "npair", m._c["npair"])
