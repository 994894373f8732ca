"""Device time of an open-loop rollout with per-step controls: b2_rollout against the loop a user writes without it.

    python tools/rollout_bench.py --tag r01 [--reps 5]

Variants, per workload (FP64):
  (a) b2_rollout recording qpos / qvel (+ sensordata on the drone)
  (b) b2_rollout with the control sequence only (nothing recorded)
  (c) the loop  ctrl <- U[t]; b2_step(1); traj_q[t] <- qpos; traj_v[t] <- qvel  (+ sensordata on the drone), captured in
      one CUDA graph so that Python is not in the timing
  (d) b2_step(T) with the controls held: the ceiling
Workloads: cartpole N = 65,536, T = 100 and 1,000; drone N = 262,144, T = 100, random in-range thrust from a free-flight
start; humanoid N = 16,384, T = 200 from stand_on_left_leg (warp engine).  Every timed call starts from the same state and
is bracketed by CUDA events after a warm-up; L2 is overwritten (192 MB memset, outside the events) between timed calls.
Reports env-steps/s and, for (a), the recording's algorithmic bytes/s: 8 (nu + nq + nv [+ nsensordata]) per env-step
(control row read, state rows written).  Writes profiles/rollout_<tag>.json with the card's name and power limit read
in the same run.
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

WORKLOADS = (("cartpole", 65536, 100), ("cartpole", 65536, 1000), ("drone", 262144, 100), ("humanoid", 16384, 200))


def load(name):
    from mujoco_template import _mj as mj

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return mj.MjModel.from_compiled(os.path.join(ROOT, "tests", "golden", "models", f"{name}.b2m"))


def controls(model, name, n, T):
    g = torch.Generator(device="cuda:0").manual_seed(1)
    U = torch.rand((T, model.nu, n), device="cuda:0", dtype=torch.float64, generator=g)
    if name == "humanoid":
        return (U * 2 - 1) * 0.2
    lo = torch.as_tensor(model.actuator_ctrlrange[:, 0], device="cuda:0")[None, :, None]
    hi = torch.as_tensor(model.actuator_ctrlrange[:, 1], device="cuda:0")[None, :, None]
    return lo + (hi - lo) * U  # in range


def timed(fn, reset, flush, reps):
    for _ in range(2):
        reset(); fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        reset()
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms)), float(np.min(ms)), float(np.max(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="output path (default profiles/rollout_<tag>.json)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("rollout_bench: needs a CUDA device")
    from conftest import random_states
    from mujoco_template import _mj as mj

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    card = {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}
    flush = torch.empty(192 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda:0")
    results = []
    for name, n, T in WORKLOADS:
        model = load(name)
        data = mj.BatchData(model, n)
        be = data.backend
        qpos, qvel, ctrl = random_states(model, name, n, seed=0)
        start = [torch.as_tensor(a.T.copy(), device="cuda:0") for a in (qpos, qvel, ctrl)]

        def reset():
            for dst, src in zip((data.qpos, data.qvel, data.ctrl), start):
                dst.copy_(src)
            data.qacc_warmstart.zero_(); data.flags.zero_()

        U = controls(model, name, n, T)
        sens = model.nsensordata > 0
        traj = [torch.empty((T, d, n), device="cuda:0", dtype=torch.float64) for d in (model.nq, model.nv, model.nsensordata)]
        out_a = (traj[0], traj[1], traj[2] if sens else None)
        t_a = timed(lambda: be.rollout(U, T, True, out=out_a), reset, flush, args.reps)
        reset(); be.rollout(U, T, True, out=out_a); torch.cuda.synchronize()
        final_a = data.qpos.clone()
        t_b = timed(lambda: be.rollout(U, T, False), reset, flush, args.reps)

        def loop():
            for t in range(T):
                data.ctrl.copy_(U[t])
                be.step(1)
                traj[0][t].copy_(data.qpos); traj[1][t].copy_(data.qvel)
                if sens:
                    traj[2][t].copy_(data.sensordata)

        reset(); loop()  # warm-up outside capture
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            loop()
        t_c = timed(graph.replay, reset, flush, args.reps)
        reset(); graph.replay(); torch.cuda.synchronize()
        diff = float((data.qpos - final_a).abs().max()) / max(1.0, float(final_a.abs().max()))
        t_d = timed(lambda: be.step(T), reset, flush, args.reps)
        del graph
        steps = n * T
        rec_bytes = 8 * (model.nu + model.nq + model.nv + model.nsensordata) * steps
        row = {"workload": name, "N": n, "T": T, "kernels": be.batch.kernel_variant, "records_sensordata": sens,
               "a_rollout_record_ms": t_a, "b_rollout_ms": t_b, "c_graph_loop_ms": t_c, "d_step_held_ms": t_d,
               "env_steps_per_s": {k: steps / (v[0] * 1e-3) for k, v in (("a", t_a), ("b", t_b), ("c", t_c), ("d", t_d))},
               "a_recording_bytes": rec_bytes, "a_recording_bytes_per_s": rec_bytes / (t_a[0] * 1e-3),
               "speedup_a_over_c": t_c[0] / t_a[0], "a_over_d": t_a[0] / t_d[0],
               "final_qpos_rel_diff_a_vs_c": diff}
        results.append(row)
        print(json.dumps(row), flush=True)
        del data, be, traj, U, out_a
        torch.cuda.empty_cache()
    out = {"card": card, "precision": "FP64",
           "timing": "median / min / max of device-event times per call (ms); L2 overwritten between calls; state reset outside the events",
           "results": results}
    path = args.out or os.path.join(ROOT, "profiles", f"rollout_{args.tag}.json")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
