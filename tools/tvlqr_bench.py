"""Device time of the time-varying LQR backward pass (b2_tvlqr) and of the closed-loop rollout (b2_rollout_feedback)
against what a user writes without them.

    python tools/tvlqr_bench.py --tag r01 [--reps 3]

b2_tvlqr, per workload (FP64; A_t, B_t from b2_linearize_rollout about per-env random states under in-range controls;
Q = I, R = 0.1 I, Qf = 10 Q, linear terms q, r, reg = 1e-6):
  (1) new    b2_tvlqr: one launch (a thread per env for the cartpole, a warp per env for the drone and humanoid)
  (2) torch  the same recursion as one batched torch.linalg call sequence per step (cholesky, cholesky_solve, matmul)
             on (T, N, nx, nx) copies of A and B made outside the timed window
  plus the bytes of A and B the kernel reads over its time, against the HBM bandwidth of the data sheet (7.7 TB/s).
b2_rollout_feedback, per workload (nominal: the linearised rollout; start 0.01 off it; gains and feedforward from (1)):
  (3) law    b2_rollout_feedback, recording the controls and states
  (4) open   b2_rollout of the same length under the nominal controls, recording the states: the cost of the law is
             (3) - (4)
  (5) graph  the loop  law; b2_step(1)  (the law in torch, with b2_differentiate_pos) captured in one CUDA graph
Every rollout variant starts with the copy of the start state into the batch.
Workloads: cartpole N = 65,536, T = 100; drone N = 16,384, T = 100; humanoid N = 1,024, T = 32 (warp engine: the library
runs the law launch, one warp step and the row copies per step).
Timing: device events around a window of k back-to-back calls, k chosen so that the window lasts at least 50 ms
(k <= 2000); per-call time = window / k; median / min / max over --reps windows after two warm-up calls.  L2 is
overwritten (192 MB memset) before every window.  The outputs of compared variants are checked at every timed size
(largest relative difference, relative to max(1, max |x|)).  Writes profiles/tvlqr_<tag>.json with the card's name,
power limit and max SM clock read in the same run.
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

WORKLOADS = (("cartpole", 65536, 100), ("drone", 16384, 100), ("humanoid", 1024, 32))
WINDOW_MS = 50.0
HBM_TBS = 7.7  # data sheet, HGX B200, one GPU


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
    return lo + (hi - lo) * (0.25 + 0.5 * U)


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


def torch_tvlqr(A, B, Q, R, Qf, q, r, reg, K, k):
    """The recursion of include/b2mj.h with batched torch calls: A (T, N, nx, nx), B (T, N, nx, nu), q (T+1, N, nx),
    r (T, N, nu); writes K (T, N, nu, nx), k (T, N, nu)."""
    T, n, nx, nu = A.shape[0], A.shape[1], A.shape[2], B.shape[3]
    P = Qf.expand(n, nx, nx).clone()
    s = q[T].clone()
    I = reg * torch.eye(nu, dtype=A.dtype, device=A.device)
    for t in range(T - 1, -1, -1):
        At, Bt = A[t], B[t]
        PA, PB = P @ At, P @ Bt
        Atr, Btr = At.transpose(1, 2), Bt.transpose(1, 2)
        Qx = q[t] + (Atr @ s[..., None])[..., 0]
        Qu = r[t] + (Btr @ s[..., None])[..., 0]
        Quu, Qux = R + Btr @ PB, Btr @ PA
        L = torch.linalg.cholesky(Quu + I)
        K[t] = torch.cholesky_solve(Qux, L)
        k[t] = -torch.cholesky_solve(Qu[..., None], L)[..., 0]
        Kt, kt = K[t], k[t]
        Ktr = Kt.transpose(1, 2)
        P = Q + Atr @ PA + Ktr @ (Quu @ Kt - Qux) - Qux.transpose(1, 2) @ Kt
        P = 0.5 * (P + P.transpose(1, 2))
        s = Qx + (Qux.transpose(1, 2) @ kt[..., None])[..., 0] - (Ktr @ (Qu + (Quu @ kt[..., None])[..., 0])[..., None])[..., 0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="output path (default profiles/tvlqr_<tag>.json)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tvlqr_bench: needs a CUDA device")
    import mujoco_template as mt
    from conftest import random_states
    from mujoco_template import _capi

    q_smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True)
    card = {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q_smi.stdout.strip()}
    flush = torch.empty(192 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda:0")
    f64 = dict(device="cuda:0", dtype=torch.float64)
    results = []
    for name, n, T in WORKLOADS:
        model = load(name)
        env = mt.BatchedEnv(model, n)
        data, be = env.data, env.data.backend
        qpos, qvel, ctrl = random_states(model, name, n, seed=0)
        start = [torch.as_tensor(a.T.copy(), device="cuda:0") for a in (qpos, qvel, ctrl)] + [torch.zeros_like(data.qacc_warmstart)]

        def reset(off=0.0):
            for dst, src in zip((data.qpos, data.qvel, data.ctrl, data.qacc_warmstart), start):
                dst.copy_(src)
            if off:
                data.qvel.add_(off)

        reset()
        U = controls(model, name, n, T)
        A, B, _, _, Xq, Xv, _, _ = be.linearize_rollout(U, T, 1e-6, True, False)
        nx, nu = 2 * model.nv, model.nu
        g = torch.Generator(device="cuda:0").manual_seed(2)
        qlin = torch.randn((T + 1, nx, n), generator=g, **f64)
        rlin = torch.randn((T, nu, n), generator=g, **f64)
        Q, R = np.eye(nx), 0.1 * np.eye(nu)
        Qf, reg = 10 * Q, 1e-6
        K, k = torch.empty((T, nu, nx, n), **f64), torch.empty((T, nu, n), **f64)
        P0, dV, status = torch.empty((nx, nx, n), **f64), torch.empty((2, n), **f64), torch.zeros(n, dtype=torch.int32, device="cuda:0")
        stream = torch.cuda.current_stream().cuda_stream

        def new():
            _capi.tvlqr(0, 64, T, nx, nu, n, A.data_ptr(), B.data_ptr(), Q.reshape(-1), R.reshape(-1), Qf.reshape(-1), qlin.data_ptr(),
                        rlin.data_ptr(), reg, K.data_ptr(), k.data_ptr(), P0.data_ptr(), dV.data_ptr(), status.data_ptr(), stream)

        t_new = timed(new, flush, args.reps)
        new(); torch.cuda.synchronize()
        assert int(status.abs().max()) == 0
        Ab, Bb = A.permute(0, 3, 1, 2).contiguous(), B.permute(0, 3, 1, 2).contiguous()
        qb, rb = qlin.permute(0, 2, 1).contiguous(), rlin.permute(0, 2, 1).contiguous()
        Qt, Rt, Qft = (torch.as_tensor(M, **f64) for M in (Q, R, Qf))
        Kb, kb = torch.empty((T, n, nu, nx), **f64), torch.empty((T, n, nu), **f64)
        t_torch = timed(lambda: torch_tvlqr(Ab, Bb, Qt, Rt, Qft, qb, rb, reg, Kb, kb), flush, args.reps)
        torch_tvlqr(Ab, Bb, Qt, Rt, Qft, qb, rb, reg, Kb, kb)
        diff_tvlqr = max(rel(K.permute(0, 3, 1, 2), Kb), rel(k.permute(0, 2, 1), kb))
        ab_bytes = T * n * (nx * nx + nx * nu) * 8
        gbs = ab_bytes / (t_new["median_ms"] * 1e-3) / 1e9
        del Ab, Bb, Kb, kb, qb, rb
        # closed-loop rollout about the nominal, 0.01 off it
        Kv, kv = K, k
        ctrl_traj, q_traj, v_traj = (torch.empty((T, d, n), **f64) for d in (nu, model.nq, model.nv))
        q2, v2 = torch.empty((T, model.nq, n), **f64), torch.empty((T, model.nv, n), **f64)
        alpha = torch.full((n,), 0.5, **f64)

        def law():
            reset(0.01)
            be.rollout_feedback(U, Xq, Xv, Kv, kv, alpha, T, False, out=(ctrl_traj, q_traj, v_traj, None), derived=False)

        def open_loop():
            reset(0.01)
            be.rollout(U, T, False, out=(q2, v2, None), derived=False)

        t_law = timed(law, flush, args.reps)
        t_open = timed(open_loop, flush, args.reps)
        law(); torch.cuda.synchronize()
        fb = [x.clone() for x in (ctrl_traj, q_traj, v_traj)]
        # the loop law; b2_step(1), captured in one CUDA graph
        dq = torch.empty_like(data.qvel)
        lo = torch.as_tensor(model.actuator_ctrlrange[:, 0], **f64)[:, None]
        hi = torch.as_tensor(model.actuator_ctrlrange[:, 1], **f64)[:, None]
        lim = torch.as_tensor(np.asarray(model.actuator_ctrllimited, dtype=bool), device="cuda:0")[:, None]
        lq, lv, lu = torch.empty_like(q_traj), torch.empty_like(v_traj), torch.empty_like(ctrl_traj)

        def loop():
            reset(0.01)
            for t in range(T):
                be._pre()
                be.batch.differentiate_pos(dq.data_ptr(), 1.0, Xq[t].data_ptr(), data.qpos.data_ptr(), be.stream)
                x = torch.cat([dq, data.qvel - Xv[t]], 0)
                u = U[t] + alpha[None] * kv[t] - torch.einsum("ajn,jn->an", Kv[t], x)
                data.ctrl.copy_(torch.where(lim, torch.minimum(torch.maximum(u, lo), hi), u))
                be.step(1, derived=False)
                lu[t].copy_(data.ctrl); lq[t].copy_(data.qpos); lv[t].copy_(data.qvel)

        loop(); torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            loop()
        t_graph = timed(graph.replay, flush, args.reps)
        lq.fill_(7.0)
        graph.replay(); torch.cuda.synchronize()
        diff_fb = max(rel(a, b) for a, b in zip(fb, (lu, lq, lv)))
        del graph
        row = {"workload": name, "N": n, "T": T, "nx": nx, "nu": nu, "kernels": be.batch.kernel_variant,
               "tvlqr": {"new": t_new, "torch_linalg": t_torch, "torch_over_new": t_torch["median_ms"] / t_new["median_ms"],
                         "A_B_bytes": ab_bytes, "A_B_read_GBps": gbs, "share_of_hbm_datasheet": gbs / (HBM_TBS * 1e3),
                         "max_rel_diff_K_k": diff_tvlqr},
               "rollout": {"feedback": t_law, "open_loop": t_open, "graph_law_step_loop": t_graph,
                           "law_cost_ms": t_law["median_ms"] - t_open["median_ms"],
                           "graph_loop_over_feedback": t_graph["median_ms"] / t_law["median_ms"],
                           "max_rel_diff_feedback_vs_loop": diff_fb}}
        results.append(row)
        print(json.dumps(row), flush=True)
        del env, data, be, A, B, K, k, Xq, Xv
        torch.cuda.empty_cache()
    out = {"card": card, "precision": "FP64",
           "timing": (f"per-call device-event time (ms): median / min / max over {args.reps} windows of k back-to-back calls "
                      f"(window >= {WINDOW_MS:.0f} ms, k <= 2000), after two warm-up calls; L2 overwritten before every window, "
                      "not between the calls inside it"),
           "results": results}
    path = args.out or os.path.join(ROOT, "profiles", f"tvlqr_{args.tag}.json")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
