"""Device time of the trajectory cost and its gradients (b2_traj_cost) against what a user writes without it, against the
other calls of an iLQR iteration of the same size, and the parts of one batched_ilqr iteration.

    python tools/traj_cost_bench.py --tag r01 [--reps 3] [--out PATH]

Per workload (FP64; the trajectory is b2_linearize_rollout's nominal under in-range controls from per-env random states;
qpos_ref a goal pose broadcast to every env and step, qvel_ref and ctrl_ref per-env random, all materialised; Q, Qf
non-diagonal SPD, R = 0.1 I):
  (1) new     b2_traj_cost with J, q and r: one launch
  (2) torch   the same cost and gradients composed by a user: T+1 b2_differentiate_pos launches into a (T+1, nv, N)
              buffer, then einsums for M e, J and R w.  It omits the Jr^-1 of free joints (so it is exact for the cartpole
              only, and a lower bound on the work for the drone and humanoid).
  plus the algorithmic bytes of (1) -- reads (T+1)(2nq + 2nv) + 2T nu, writes (T+1) 2nv + T nu + 1 reals per env --
  over its time, against the HBM bandwidth of the data sheet (7.7 TB/s).
  (3) b2_tvlqr on (1)'s q / r, (4) b2_rollout_feedback recording controls and states: the other calls of an iteration.
  (5) one batched_ilqr iteration (iters = 1: linearize_rollout, traj_cost, tvlqr, the line search, the state restores),
      end to end with device events, and its parts: linearize_rollout, traj_cost(grad), tvlqr and one line-search trial
      (rollout_feedback + traj_cost), each timed on its own.
Workloads: cartpole N = 65,536, T = 100 (about 0.8 GB per call, above L2); drone N = 16,384, T = 100; humanoid
N = 1,024, T = 32 (warp engine).
Timing: device events around a window of k back-to-back calls, k chosen so that the window lasts at least 50 ms
(k <= 2000); per-call time = window / k; median / min / max over --reps windows after two warm-up calls.  L2 is
overwritten (192 MB memset) before every window.  Writes profiles/traj_cost_<tag>.json (or --out) with the card's name,
power limit and max SM clock read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "mujoco-template_b200"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

from tvlqr_bench import HBM_TBS, controls, load, rel, timed  # noqa: E402

WORKLOADS = (("cartpole", 65536, 100), ("drone", 16384, 100), ("humanoid", 1024, 32))


def spd(rng, n):
    U, _ = np.linalg.qr(rng.normal(size=(n, n)))
    M = U @ np.diag(np.geomspace(1.0, 10.0, n)) @ U.T
    return 0.5 * (M + M.T)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="output path (default profiles/traj_cost_<tag>.json)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("traj_cost_bench: needs a CUDA device")
    import mujoco_template as mt
    from conftest import random_states
    from mujoco_template import _capi
    from mujoco_template.batched_controllers import batched_ilqr

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
        nq, nv, nu, nx = model.nq, model.nv, model.nu, 2 * model.nv
        qpos, qvel, ctrl = random_states(model, name, n, seed=0)
        for dst, src in zip((data.qpos, data.qvel, data.ctrl), (qpos, qvel, ctrl)):
            dst.copy_(torch.as_tensor(src.T.copy(), **f64))
        data.qacc_warmstart.zero_()
        U = controls(model, name, n, T)
        A, B, _, _, Xq, Xv, _, _ = be.linearize_rollout(U, T, 1e-6, True, False)
        rng = np.random.default_rng(3)
        Q, R, Qf = spd(rng, nx), 0.1 * np.eye(nu), 10 * spd(rng, nx)
        Qh, Rh, Qfh = Q.reshape(-1), R.reshape(-1), Qf.reshape(-1)
        goal = torch.as_tensor(model.key_qpos[0] if len(model.key_qpos) else model.qpos0, **f64)
        qref = goal[None, :, None].expand(T + 1, nq, n).contiguous()
        g = torch.Generator(device="cuda:0").manual_seed(4)
        vref = 0.1 * torch.randn((T + 1, nv, n), generator=g, **f64)
        uref = torch.randn((T, nu, n), generator=g, **f64)
        J, q, r = torch.empty(n, **f64), torch.empty((T + 1, nx, n), **f64), torch.empty((T, nu, n), **f64)

        def new():
            be.traj_cost(Xq, Xv, U, qref, vref, uref, Qh, Rh, Qfh, T, True, out=(J, q, r))

        t_new = timed(new, flush, args.reps)
        new(); torch.cuda.synchronize()
        reals = (T + 1) * (2 * nq + 2 * nv) + 2 * T * nu + (T + 1) * nx + T * nu + 1
        gbs = reals * 8 * n / (t_new["median_ms"] * 1e-3) / 1e9
        # the torch composition: T+1 differentiate_pos launches, then einsums
        dq = torch.empty((T + 1, nv, n), **f64)
        Qt, Rt, Qft = (torch.as_tensor(M, **f64) for M in (Q, R, Qf))

        def composed():
            be._pre()
            for t in range(T + 1):
                be.batch.differentiate_pos(dq[t].data_ptr(), 1.0, qref[t].data_ptr(), Xq[t].data_ptr(), be.stream)
            e = torch.cat([dq, Xv - vref], 1)
            y = torch.einsum("ij,tjn->tin", Qt, e[:T])
            yT = Qft @ e[T]
            w = U - uref
            rr = torch.einsum("ij,tjn->tin", Rt, w)
            Jt = 0.5 * ((e[:T] * y).sum((0, 1)) + (e[T] * yT).sum(0) + (w * rr).sum((0, 1)))
            return Jt, torch.cat([y, yT[None]], 0), rr

        t_torch = timed(composed, flush, args.reps)
        Jt, qt, rt = composed()
        diff = {"J": rel(J, Jt), "r": rel(r, rt), "q_without_Jr_inv": rel(q, qt)}
        # the other calls of an iteration
        K, k = torch.empty((T, nu, nx, n), **f64), torch.empty((T, nu, n), **f64)
        P0, dV, status = torch.empty((nx, nx, n), **f64), torch.empty((2, n), **f64), torch.zeros(n, dtype=torch.int32, device="cuda:0")
        stream = torch.cuda.current_stream().cuda_stream

        def tvlqr():
            _capi.tvlqr(0, 64, T, nx, nu, n, A.data_ptr(), B.data_ptr(), Qh, Rh, Qfh, q.data_ptr(), r.data_ptr(), 1e-6, K.data_ptr(),
                        k.data_ptr(), P0.data_ptr(), dV.data_ptr(), status.data_ptr(), stream)

        t_tvlqr = timed(tvlqr, flush, args.reps)
        tvlqr()
        x0 = [t.clone() for t in (data.qpos, data.qvel, data.qacc_warmstart)]
        tq, tv, tu = torch.empty((T + 1, nq, n), **f64), torch.empty((T + 1, nv, n), **f64), torch.empty((T, nu, n), **f64)
        tq[0], tv[0] = x0[0], x0[1]
        alpha = torch.full((n,), 0.5, **f64)

        def restore():
            for dst, src in zip((data.qpos, data.qvel, data.qacc_warmstart), x0):
                dst.copy_(src)

        def feedback():
            restore()
            be.rollout_feedback(U, Xq, Xv, K, k, alpha, T, False, out=(tu, tq[1:], tv[1:], None), derived=False)

        def trial():
            feedback()
            be.traj_cost(tq, tv, tu, qref, vref, uref, Qh, Rh, Qfh, T, False, out=(J, None, None))

        t_fb = timed(feedback, flush, args.reps)
        t_trial = timed(trial, flush, args.reps)
        Wt = torch.empty((T + 1, nv, n), **f64)
        t_lin = timed(lambda: be.linearize_rollout(U, T, 1e-6, True, False, out=(A, B, None, None, Xq, Xv, Wt, None)), flush, args.reps)
        # one batched_ilqr iteration, end to end (its host-side decisions synchronise once per trial)
        Uv = U.permute(2, 0, 1)
        refs = dict(qpos_ref=goal, qvel_ref=vref.permute(2, 0, 1), ctrl_ref=uref.permute(2, 0, 1))
        info = {}

        def ilqr():
            info["out"] = batched_ilqr(env, Uv, Q, R, Qf, iters=1, **refs)

        t_ilqr = timed(ilqr, flush, args.reps)
        row = {"workload": name, "N": n, "T": T, "nx": nx, "nu": nu, "kernels": be.batch.kernel_variant,
               "traj_cost": {"new": t_new, "torch_composed": t_torch, "torch_over_new": t_torch["median_ms"] / t_new["median_ms"],
                             "algorithmic_bytes": reals * 8 * n, "GBps": gbs, "share_of_hbm_datasheet": gbs / (HBM_TBS * 1e3),
                             "max_rel_diff_vs_torch": diff},
               "same_size": {"tvlqr": t_tvlqr, "rollout_feedback": t_fb,
                             "traj_cost_over_tvlqr": t_new["median_ms"] / t_tvlqr["median_ms"],
                             "traj_cost_over_rollout_feedback": t_new["median_ms"] / t_fb["median_ms"]},
               "ilqr_iteration": {"batched_ilqr_iters_1": t_ilqr, "linearize_rollout": t_lin, "traj_cost_grad": t_new, "tvlqr": t_tvlqr,
                                  "line_search_trial": t_trial,
                                  "worst_J_over_envs_history": [float(x) for x in info["out"]["J_history"].max(1).values.cpu()]}}
        results.append(row)
        print(json.dumps(row), flush=True)
        del env, data, be, A, B, K, k, Xq, Xv, q, r, qref, vref, uref, dq, info
        torch.cuda.empty_cache()
    out = {"card": card, "precision": "FP64",
           "timing": (f"per-call device-event time (ms): median / min / max over {args.reps} windows of k back-to-back calls "
                      "(window >= 50 ms, k <= 2000), after two warm-up calls; L2 overwritten before every window, "
                      "not between the calls inside it"),
           "results": results}
    path = args.out or os.path.join(ROOT, "profiles", f"traj_cost_{args.tag}.json")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
