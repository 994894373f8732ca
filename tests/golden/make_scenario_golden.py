"""Generates tests/golden/scenario_*.npz: the reference's example scenarios (its own controllers, imported unmodified from
the original mujoco-template checkout's examples/) run on the oracle-backed Env, recorded step by step.  The fixtures
let the test suite replay the same trajectories without that checkout: on the oracle (tests/test_reference_scenarios.py)
and through the CUDA path (tests/test_gpu_parity.py::test_reference_scenario_*).

    B2_REFERENCE=<checkout> python tests/golden/make_scenario_golden.py          # writes next to this file

Each file holds: qpos0 / qvel0 / ctrl0 / warm0 (state before the first step), ctrl[t] (what the controller wrote before step
t), qpos[t] / qvel[t] / warm[t] (state and qacc_warmstart after step t), time[t], header + rows of the StateControlRecorder
CSV (the humanoid's first ROWS_KEPT rows only: its CSV repeats qpos / qvel / ctrl and no test reads further), duration /
max_steps.
"""
import importlib
import os
import sys
import tempfile
from types import SimpleNamespace

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.join(ROOT, "mujoco-template_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import warnings  # noqa: E402

warnings.simplefilter("ignore")
import mujoco_template as mt  # noqa: E402
from mujoco_template import _mj as mj  # noqa: E402
from oracle_backend import OracleBackend  # noqa: E402
import test_reference_scenarios as T  # noqa: E402

MODEL_OF = {"pendulum_pd": "pendulum", "pendulum_passive": "pendulum", "cartpole_pid": "cartpole", "drone_lqr": "drone",
            "humanoid_lqr": "humanoid"}
ROWS_KEPT = {"humanoid_lqr": 100}  # keeps the file under 1 MB


def main():
    mt.PassiveRunSettings, mt.PassiveRunHarness = T._Settings, T._Harness
    mt.AdaptiveCameraSettings = lambda **kw: SimpleNamespace(**kw)
    mj.NativeBackend = lambda model, nenv=1, **kw: OracleBackend(model)
    sys.path.append(T.REF)
    for name, (module_name, expected_steps, _) in T.SCENARIOS.items():
        mod = importlib.import_module(module_name)
        harness, cfg = mod.HARNESS, mod.CONFIG
        env = harness.env_factory()
        if harness.seed_fn is not None:
            harness.seed_fn(env)
        probes = harness.probes(env) if callable(harness.probes) else harness.probes
        start = dict(qpos0=np.array(env.data.qpos), qvel0=np.array(env.data.qvel), ctrl0=np.array(env.data.ctrl),
                     warm0=np.array(env.data.qacc_warmstart))
        ctrl, qpos, qvel, time, warm = [], [], [], [], []

        def tap(_result):
            ctrl.append(np.array(env.data.ctrl)); qpos.append(np.array(env.data.qpos)); qvel.append(np.array(env.data.qvel))
            time.append(float(env.data.time)); warm.append(np.array(env.data.qacc_warmstart))

        with tempfile.TemporaryDirectory() as tmp:
            rec = mt.StateControlRecorder(env, log_path=os.path.join(tmp, "log.csv"), store_rows=True, probes=tuple(probes or ()))
            with rec:
                steps = mt.run_passive_headless(env, duration=cfg.run.simulation.duration_seconds,
                                                max_steps=cfg.run.simulation.max_steps, hooks=[tap, rec])
            header = open(os.path.join(tmp, "log.csv")).readline().strip().split(",")
            rows = np.loadtxt(os.path.join(tmp, "log.csv"), delimiter=",", skiprows=1)
        assert steps == expected_steps, (name, steps)
        out = os.path.join(HERE, f"scenario_{name}.npz")
        np.savez_compressed(out, model=MODEL_OF[name], steps=steps, header=np.array(header), rows=rows[:ROWS_KEPT.get(name)],
                            ctrl=np.array(ctrl).reshape(steps, -1), qpos=np.array(qpos), qvel=np.array(qvel), time=np.array(time),
                            warm=np.array(warm),
                            duration=np.array(np.nan if cfg.run.simulation.duration_seconds is None else cfg.run.simulation.duration_seconds),
                            max_steps=np.array(-1 if cfg.run.simulation.max_steps is None else cfg.run.simulation.max_steps), **start)
        print(name, steps, "steps ->", os.path.relpath(out, ROOT), f"{os.path.getsize(out) / 1024:.0f} KB")


if __name__ == "__main__":
    main()
