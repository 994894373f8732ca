"""Device time of the transition Jacobians along a control sequence: b2_linearize_rollout against the loops a user writes
without it.

    python tools/linearize_rollout_bench.py --tag r01 [--reps 3]

Variants, per workload (FP64, centred differences, eps = 1e-6; every variant produces A_t, B_t for t < T and the nominal
states x_0 .. x_T):
  (1) new    b2_linearize_rollout: on the lane engine the nominal rollout plus one FD launch over every (step, env)
  (2) eager  the Python loop  x <- x0;  for t: ctrl <- U[t]; b2_linearize -> A[t], B[t]; b2_step(1); X[t+1] <- x
  (3) graph  the same loop captured in one CUDA graph and replayed
The loops start with the copy of x0 into the state (so that every call starts from the same state, as (1) does without a
copy), and record the state after every step, which (1) records too.
Workloads: cartpole, drone and pendulum (model-specialised kernels) at N = 1, 16, 256, 4,096 and 65,536 with T = 32 and
128; the humanoid (warp engine, where (1) is the same loop run inside the library) at N = 1, 16, 256 and 4,096 with T = 32.
Timing: device events around a window of k back-to-back calls, k chosen so that the window lasts at least 50 ms (k <= 2000);
per-call time = window / k; median / min / max over --reps windows after two warm-up calls.  L2 is overwritten (192 MB
memset) before every window, not between the calls inside it: at small N the working set of every variant stays
L2-resident across the window alike.  The outputs of the three variants are compared at every timed size (largest
relative difference of A, B and the state rows, relative to max(1, max |x|)).  Writes
profiles/linearize_rollout_<tag>.json with the card's name, power limit and max SM clock read in the same run.
"""
import argparse
import json
import math
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

SIZES = (1, 16, 256, 4096, 65536)
WORKLOADS = ([(name, n, T) for name in ("cartpole", "drone", "pendulum") for T in (32, 128) for n in SIZES]
             + [("humanoid", n, 32) for n in (1, 16, 256, 4096)])
EPS = 1e-6
WINDOW_MS = 50.0


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


def timed(fn, flush, reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); e1.synchronize()
    k = max(1, min(2000, math.ceil(WINDOW_MS / max(e0.elapsed_time(e1), 1e-3))))
    ms = []
    for _ in range(reps):
        flush.zero_()
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1) / k)
    return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms)), "calls_per_window": k}


def rel(a, b):
    return float((a - b).abs().max()) / max(1.0, float(b.abs().max()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="output path (default profiles/linearize_rollout_<tag>.json)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("linearize_rollout_bench: needs a CUDA device")
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
        start = [torch.as_tensor(a.T.copy(), device="cuda:0") for a in (qpos, qvel, ctrl)] + [torch.zeros_like(data.qacc_warmstart)]
        for dst, src in zip((data.qpos, data.qvel, data.ctrl, data.qacc_warmstart), start):
            dst.copy_(src)
        U = controls(model, name, n, T)
        nx, f64 = 2 * model.nv, dict(device="cuda:0", dtype=torch.float64)
        new = be.linearize_rollout(U, T, EPS, True, False)  # fresh outputs, then reused: fixed addresses
        t_new = timed(lambda: be.linearize_rollout(U, T, EPS, True, False, out=new), flush, args.reps)
        A = torch.empty((T, nx, nx, n), **f64)
        B = torch.empty((T, nx, model.nu, n), **f64)
        X = [torch.empty((T + 1, d, n), **f64) for d in (model.nq, model.nv)]

        def loop():
            for dst, src in zip((data.qpos, data.qvel, data.ctrl, data.qacc_warmstart), start):
                dst.copy_(src)
            X[0][0].copy_(data.qpos); X[1][0].copy_(data.qvel)
            for t in range(T):
                data.ctrl.copy_(U[t])
                be.linearize(EPS, True, out=(A[t], B[t]))
                be.step(1, derived=False)
                X[0][t + 1].copy_(data.qpos); X[1][t + 1].copy_(data.qvel)

        t_eager = timed(loop, flush, args.reps)
        loop(); torch.cuda.synchronize()
        out_eager = [x.clone() for x in (A, B, X[0], X[1])]
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            loop()
        t_graph = timed(graph.replay, flush, args.reps)
        A.fill_(7.0); X[0].fill_(7.0)
        graph.replay(); torch.cuda.synchronize()
        out_graph = (A, B, X[0], X[1])
        out_new = (new[0], new[1], new[4], new[5])
        diff = {"new_vs_eager": max(rel(a, b) for a, b in zip(out_new, out_eager)),
                "graph_vs_eager": max(rel(a, b) for a, b in zip(out_graph, out_eager))}
        del graph
        row = {"workload": name, "N": n, "T": T, "kernels": be.batch.kernel_variant, "new": t_new, "eager_loop": t_eager,
               "graph_loop": t_graph, "eager_over_new": t_eager["median_ms"] / t_new["median_ms"],
               "graph_over_new": t_graph["median_ms"] / t_new["median_ms"], "max_rel_diff": diff}
        results.append(row)
        print(json.dumps(row), flush=True)
        del data, be, new, A, B, X, U, out_eager, out_graph, out_new
        torch.cuda.empty_cache()
    out = {"card": card, "precision": "FP64", "eps": EPS, "centered": True,
           "timing": (f"per-call device-event time (ms): median / min / max over {args.reps} windows of k back-to-back calls "
                      f"(window >= {WINDOW_MS:.0f} ms, k <= 2000), after two warm-up calls; L2 overwritten before every window, "
                      "not between the calls inside it"),
           "results": results}
    path = args.out or os.path.join(ROOT, "profiles", f"linearize_rollout_{args.tag}.json")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
