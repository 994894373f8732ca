"""Device time per launch of b2_linearize against b2_linearize_sensors, and against what C / D cost without the sensor
variant: 1 + 2 (2nv + nu) b2_forward launches over perturbed copies of the batch (sensordata read back from each).

    python tools/sensor_fd_bench.py --tag r01 [--sizes 14,16,18] [--reps 10]

Workloads: the drone on its specialised kernels and on the generic ones (B2_DISABLE_SPEC=1 at model creation), and the
sensor rig of tests/test_oracle_analytic.py (nv = 9, 44 readings, generic), at N = 2^14 / 2^16 / 2^18 in FP64 and FP32.
Each timed launch is bracketed by CUDA events after a warm-up; L2 is overwritten (192 MB memset, outside the events)
between timed launches.  Writes profiles/sensor_fd_<tag>.json with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "mujoco-template_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

EPS = 1e-6


def load(name: str, generic: bool):
    from mujoco_template import _mj as mj
    from test_oracle_analytic import SENSOR_XML

    old = os.environ.get("B2_DISABLE_SPEC")
    os.environ["B2_DISABLE_SPEC"] = "1" if generic else "0"
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            if name == "rig":
                model = mj.MjModel.from_xml_string(SENSOR_XML.format(dt=0.002))
            else:
                model = mj.MjModel.from_compiled(os.path.join(ROOT, "tests", "golden", "models", f"{name}.b2m"))
            model.native  # the kernel set is chosen here
    finally:
        if old is None:
            os.environ.pop("B2_DISABLE_SPEC")
        else:
            os.environ["B2_DISABLE_SPEC"] = old
    return model


def seed_state(data, model, name, n):
    from conftest import random_states

    if name == "drone":
        qpos, qvel, ctrl = random_states(model, "drone", n, seed=0)
    else:
        rng = np.random.default_rng(0)
        qpos = np.tile(model.qpos0, (n, 1))
        qpos[:, :3] = rng.uniform(-0.5, 0.5, (n, 3))
        q = rng.normal(size=(n, 4))
        qpos[:, 6:10] = q / np.linalg.norm(q, axis=1, keepdims=True)
        qvel = rng.normal(size=(n, model.nv))
        ctrl = rng.uniform(-1, 1, (n, model.nu))
    for dst, src in ((data.qpos, qpos), (data.qvel, qvel), (data.ctrl, ctrl)):
        dst.copy_(torch.as_tensor(src.T.copy(), dtype=dst.dtype))
    data.qacc_warmstart.zero_()


def timed(fn, flush, reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms)), float(np.min(ms)), float(np.max(ms))


def composed(model, data, scratch, out_C, out_D):
    """C / D from b2_forward alone: nominal + a plus and a minus forward pass per column, on a scratch batch."""
    sb = scratch.backend
    nv, nu = model.nv, model.nu
    dq = sb._tmp("dq", nv)

    def forward_at(kind, i, sign):
        scratch.qpos.copy_(data.qpos); scratch.qvel.copy_(data.qvel); scratch.ctrl.copy_(data.ctrl)
        scratch.qacc_warmstart.copy_(data.qacc_warmstart)
        if kind == 0:
            dq.zero_(); dq[i] = 1.0
            sb._pre(); sb.batch.integrate_pos(scratch.qpos.data_ptr(), dq.data_ptr(), sign * EPS, sb.stream)
        elif kind == 1:
            scratch.qvel[i] += sign * EPS
        elif kind == 2:
            scratch.ctrl[i] += sign * EPS
        sb.forward()
        return scratch.sensordata.clone()

    forward_at(-1, 0, 0)  # the nominal reading (a user needs it for one-sided columns)
    for kind, count, out, off in ((0, nv, out_C, 0), (1, nv, out_C, nv), (2, nu, out_D, 0)):
        for i in range(count):
            out[:, off + i] = (forward_at(kind, i, 1) - forward_at(kind, i, -1)) * (0.5 / EPS)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", required=True)
    ap.add_argument("--sizes", default="14,16,18")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None, help="output path (default profiles/sensor_fd_<tag>.json)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("sensor_fd_bench: needs a CUDA device")
    from mujoco_template import _mj as mj

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    card = {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}
    flush = torch.empty(192 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda:0")
    results = []
    for name, generic in (("drone", False), ("drone", True), ("rig", True)):
        model = load(name, generic)
        nx, ns = 2 * model.nv, model.nsensordata
        for prec in (64, 32):
            for lg in (int(s) for s in args.sizes.split(",")):
                n = 1 << lg
                data = mj.BatchData(model, n, precision=prec)
                seed_state(data, model, name, n)
                be = data.backend
                dt = be.dtype
                bufs = [torch.empty(s, device="cuda:0", dtype=dt) for s in ((nx, nx, n), (nx, model.nu, n), (ns, nx, n), (ns, model.nu, n))]
                st = be.state_struct()
                lin = timed(lambda: be.batch.linearize(st, EPS, True, bufs[0].data_ptr(), bufs[1].data_ptr()), flush, args.reps)
                sens = timed(lambda: be.batch.linearize_sensors(st, EPS, True, *[b.data_ptr() for b in bufs]), flush, args.reps)
                row = {"workload": name, "kernels": be.batch.kernel_variant, "precision": prec, "N": n,
                       "linearize_ms": lin, "linearize_sensors_ms": sens, "ratio_sensors_over_linearize": sens[0] / lin[0]}
                if lg <= 16:  # the composed path keeps 1 + 2 (2nv + nu) readings of the batch; one size per workload is enough
                    scratch = mj.BatchData(model, n, precision=prec)
                    C = torch.empty((ns, nx, n), device="cuda:0", dtype=dt)
                    D = torch.empty((ns, model.nu, n), device="cuda:0", dtype=dt)
                    comp = timed(lambda: composed(model, data, scratch, C, D), flush, max(3, args.reps // 3))
                    row["composed_forward_ms"] = comp
                    row["forward_launches"] = 1 + 2 * (nx + model.nu)
                    row["speedup_sensors_over_composed"] = comp[0] / sens[0]
                    err = float((C - bufs[2]).abs().max()) / max(1.0, float(bufs[2].abs().max()))
                    row["composed_vs_sensors_rel_diff_C"] = err
                    del scratch, C, D
                results.append(row)
                print(json.dumps(row), flush=True)
                del data, bufs
                torch.cuda.empty_cache()
    out = {"card": card, "eps": EPS, "timing": "median / min / max of device-event times per launch (ms); L2 flushed between launches",
           "results": results}
    path = args.out or os.path.join(ROOT, "profiles", f"sensor_fd_{args.tag}.json")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
