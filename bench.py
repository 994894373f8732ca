#!/usr/bin/env python
"""Headline benchmark of the batched physics path (contract: see the task brief / DESIGN.md).

A "step" = one pass of the hot path over one batch of synthetic input.  The N=1 workload is
BASELINE.json configs[1]: cartpole, 65,536 envs per GPU, FP64, every step = batched LQR control
tick + FD (A, B) linearisation of every env (10 perturbed rollouts per env in one launch) +
one physics step.  Metric: env-steps/s, whole job (all GPUs).

    python bench.py --gpus 1 --steps 200 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29500 bench.py --gpus 8 --steps 200 --warmup 5
    python bench.py --impl reference --steps 5 --warmup 1     # CPU arm: oracle on host cores
    python bench.py --dump-outputs out/   # also write the last timed step's outputs (seeded inputs: comparable across builds)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import warnings

# NCCL_DEBUG=VERSION makes NCCL print its version banner to stdout (WARN does too), ahead of the one JSON line rank 0 owes
# the driver: drop the request (an explicit INFO / TRACE setting is left alone)
if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
    del os.environ["NCCL_DEBUG"]

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "mujoco-template_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
MODEL_FILE = {m: os.path.join(ROOT, "tests", "golden", "models", f"{m}.b2m") for m in ("pendulum", "cartpole", "drone", "humanoid")}
# algorithmic bytes per env-step / per linearisation (FP64), SURVEY.md section 8(d) / BASELINE.md section 4
STEP_BYTES = {"pendulum": 40, "cartpole": 72, "drone": 240, "humanoid": 1480}
LIN_BYTES = {"pendulum": 72, "cartpole": 200, "drone": 1672, "humanoid": 33224}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="cartpole", choices=list(MODEL_FILE))
    ap.add_argument("--nenv", type=int, default=None, help="envs per GPU (default: BASELINE config for the model)")
    ap.add_argument("--no-linearize", action="store_true", help="step only (no per-step FD linearisation)")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="headline workload only (no drone / humanoid lines in `secondary`)")
    ap.add_argument("--e2e-host-controller", action="store_true", help="e2e leg: evaluate the LQR law in NumPy on the host instead of on the device")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU-baseline sample duration")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of each workload returned (state, controls, (A, B); rank 0's envs) "
                         "to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    return args


# --dump-outputs writes at most this much per workload (a run times at most four workloads: 64 MiB in all); a workload
# whose outputs are larger is written for a fixed, seeded sample of its envs
DUMP_BYTES_PER_WORKLOAD = 16 << 20


def dump_outputs(directory: str, prefix: str, env, result) -> None:
    """What a caller of env.step() receives from one step -- the state and controls in env.data, (A, B) in result.info --
    as float64 arrays with the env axis first, one DIR/<prefix><name>.npy each."""
    import torch

    arrays = {k: getattr(env.data, k).T for k in ("qpos", "qvel", "ctrl")}
    arrays.update({k: result.info[k] for k in ("A", "B") if k in result.info})
    nenv = arrays["qpos"].shape[0]
    keep = min(nenv, DUMP_BYTES_PER_WORKLOAD // sum(8 * (t.numel() // nenv) for t in arrays.values()))
    envs = np.sort(np.random.default_rng(0).choice(nenv, keep, replace=False)) if keep < nenv else slice(None)
    os.makedirs(directory, exist_ok=True)
    for k, t in arrays.items():
        np.save(os.path.join(directory, prefix + k + ".npy"), np.ascontiguousarray(t.to("cpu", dtype=torch.float64).numpy()[envs]))


DEFAULT_NENV = {"pendulum": 65536, "cartpole": 65536, "drone": 262144, "humanoid": 16384}


def load_model(name: str):
    from mujoco_template import _mj as mj

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return mj.MjModel.from_compiled(MODEL_FILE[name])


def synth_states(model, name: str, n: int, seed: int):
    """Synthetic randomized initial states (SURVEY.md section 8d). AoS (n, dim)."""
    rng = np.random.default_rng(seed)
    qpos = np.tile(model.qpos0, (n, 1))
    qvel = np.zeros((n, model.nv))
    if name == "pendulum":
        qpos[:, 0] = rng.uniform(-np.pi, np.pi, n)
    elif name == "cartpole":
        qpos[:, 0] = rng.uniform(-1, 1, n)
        qpos[:, 1] = rng.uniform(-0.2, 0.2, n)
        qvel[:] = rng.uniform(-0.5, 0.5, (n, 2))
    elif name == "drone":
        qpos[:] = model.key_qpos[0]
        qpos[:, 2] = rng.uniform(1, 3, n)
        rv = rng.normal(0, 0.1, (n, 3))
        ang = np.linalg.norm(rv, axis=1, keepdims=True)
        qpos[:, 3] = np.cos(ang[:, 0] / 2)
        qpos[:, 4:7] = rv / np.maximum(ang, 1e-12) * np.sin(ang / 2)
        qvel[:] = rng.normal(0, 0.1, (n, model.nv))
    elif name == "humanoid":
        qpos[:] = model.key_qpos[1]
        qpos[:, 7:] += rng.normal(0, 0.02, (n, model.nq - 7))
        qvel[:] = rng.normal(0, 0.01, (n, model.nv))
    return qpos, qvel


def bind_to_gpu_numa_node(local: int) -> dict:
    """One process per GPU: run this rank's host threads (and therefore first-touch its pinned buffers) on the NUMA node
    the GPU hangs off.  The e2e leg moves ~17 MB per step and rank across PCIe; with eight ranks on a two-socket host,
    buffers on the far socket put that traffic on the socket interconnect.  Best effort: no sysfs entry, no binding."""
    info = {"bound": False}
    try:
        import torch

        import pynvml as nv

        nv.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(local).uuid)
        h = nv.nvmlDeviceGetHandleByUUID(uuid if uuid.startswith("GPU-") else "GPU-" + uuid)
        bus_id = nv.nvmlDeviceGetPciInfo(h).busId
        bus_id = (bus_id.decode() if isinstance(bus_id, bytes) else bus_id).lower()
        node = -1
        for cand in (bus_id, bus_id[-12:]):  # NVML prints an 8-digit PCI domain, sysfs a 4-digit one
            path = f"/sys/bus/pci/devices/{cand}/numa_node"
            if os.path.exists(path):
                node = int(open(path).read().strip())
                break
        if node < 0:
            return info
        cpus: set[int] = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            info = {"bound": True, "numa_node": node, "cpus": len(cpus)}
    except Exception as exc:  # pragma: no cover - depends on the host
        info["error"] = str(exc)[:80]
    return info


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons during the timed region (B200_PROFILING.md recipe).  Polled through NVML every
    10 ms (nvidia-smi -lms cannot sample that fast; a faster poll from eight ranks perturbs the host side of the
    measurement), plus one explicit sample while the queued timed steps are executing (`sample_now`);
    `nvidia-smi --query-gpu` once is the fallback when NVML is not importable."""

    PERIOD_S = 0.010

    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, gpu_index: int, uuid: str | None = None):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.uuid = uuid
        self.sm: list[float] = []
        self.reasons: set[str] = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self.first = threading.Event()
        self.in_region = False
        self.region_samples = 0
        self._lock = threading.Lock()

    def run(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = None
            if self.uuid:
                try:
                    h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + self.uuid) if not self.uuid.startswith("GPU-") else self.uuid)
                except Exception:
                    h = None
            if h is None:
                h = nv.nvmlDeviceGetHandleByIndex(self.gpu)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self._nv, self._h = nv, h
            while not self._stop_evt.is_set():
                self.sample_now()
                self.first.set()
                time.sleep(self.PERIOD_S)
        except Exception:
            try:  # one-shot fallback
                q = "clocks.sm,clocks.max.sm"
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                     capture_output=True, text=True, timeout=20).stdout.strip().split(",")
                self.sm.append(float(out[0])); self.max_mhz = float(out[1])
            except Exception:
                pass
            self.first.set()

    def sample_now(self):
        nv, h = getattr(self, "_nv", None), getattr(self, "_h", None)
        if nv is None:
            return
        with self._lock:
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
            try:
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
            except Exception:
                mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
            for name, bit in self.BAD.items():
                if mask & bit:
                    self.reasons.add(name)
            if self.in_region:
                self.region_samples += 1

    def stop(self) -> dict:
        self._stop_evt.set()
        self.join(timeout=5)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.sm), "samples_in_timed_region": self.region_samples, "source": "NVML polled every 10 ms + one sample while the queued timed steps execute"}


CPU_KIND_NOTE = ("oracle = C restatement of mj_step / mjd_transitionFD, built -O3 -march=native with FP contraction for this arm "
                 "(compiled on this host into a temporary directory); mujoco itself is not installable offline")


def _cpu_model(model):
    """The CPU arm's oracle: the optimised build (never the parity build)."""
    from oracle.oracle import OracleModel

    return OracleModel(model.blob, dict(nq=model.nq, nv=model.nv, nu=model.nu, nbody=model.nbody, njnt=model.njnt,
                                        ngeom=model.ngeom, nsite=model.nsite, ntendon=model.ntendon), variant="fast")


def _cpu_probe_rate(om, model, name: str, linearize: bool, cores: int, seed: int) -> float:
    """env-steps/s of a short all-core run: the sample grows until it takes >= 0.1 s, so that thread start-up and page
    faults do not dominate the estimate."""
    n_probe = max(cores * 4, 64)
    rate = 1.0
    for _ in range(8):
        qpos, qvel = synth_states(model, name, n_probe, seed)
        ctrl = np.zeros((n_probe, model.nu))
        t0 = time.perf_counter()
        om.batch_rollout(qpos, qvel, ctrl, nsteps=2, lin=linearize, nthreads=cores)
        dt = max(time.perf_counter() - t0, 1e-6)
        rate = n_probe * 2 / dt
        if dt >= 0.1:
            break
        n_probe = int(min(n_probe * 8, 1 << 20))
    return rate


def cpu_oracle_rate(model, name: str, linearize: bool, target_seconds: float, seed: int = 123):
    """Oracle (CPU restatement of mj_step / mjd_transitionFD) on all host cores over a bounded sample."""
    om = _cpu_model(model)
    cores = os.cpu_count() or 1
    probe_rate = _cpu_probe_rate(om, model, name, linearize, cores, seed)
    nsteps = 10
    n = int(min(max(probe_rate * target_seconds / nsteps, cores), 1 << 20))
    for _ in range(3):  # the short probe under-estimates the rate (thread start-up): grow the sample if needed
        qpos, qvel = synth_states(model, name, n, seed + 1)
        ctrl = np.zeros((n, model.nu))
        t0 = time.perf_counter()
        om.batch_rollout(qpos, qvel, ctrl, nsteps=nsteps, lin=linearize, nthreads=cores)
        dt = time.perf_counter() - t0
        if dt >= 0.5 * target_seconds or n >= (1 << 20):
            break
        n = int(min(n * target_seconds / max(dt, 1e-3), 1 << 20))
    return dict(value=n * nsteps / dt, unit=UNIT, cores=cores, kind="port",
                sample=f"{n} envs x {nsteps} steps of the same workload ({'FD linearisation + ' if linearize else ''}step), "
                       f"{dt:.1f} s wall, pthread shards over {cores} threads; " + CPU_KIND_NOTE)


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the path.  The reference delegates to the
    `mujoco` wheel, which is not installable offline, so this times the oracle port on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.model
    model = load_model(name)
    lin = not args.no_linearize
    om = _cpu_model(model)
    cores = os.cpu_count() or 1
    # bounded sample: about 1.5 s of all-core work per step (about 20 s for the whole run), sized from a measured probe
    rate = _cpu_probe_rate(om, model, name, lin, cores, 5)
    n = int(max(cores, min(1 << 18, 1.5 * rate, 20.0 * rate / max(args.steps + args.warmup, 1))))
    qpos, qvel = synth_states(model, name, n, 7)
    ctrl = np.zeros((n, model.nu))
    warm = np.zeros((n, model.nv))
    # every step is one pass of the hot path (FD linearisation + mj_step of every env of the sample) from the configured
    # initial-state distribution -- the GPU arm's envs are held there by their controller, an uncontrolled CPU rollout
    # would drift into the floor and time the contact solver instead.  The median step counts (the host is a shared VM).
    q0, v0 = qpos.copy(), qvel.copy()
    times = []
    for i in range(args.warmup + args.steps):
        np.copyto(qpos, q0); np.copyto(qvel, v0); warm[:] = 0
        t0 = time.perf_counter()
        om.batch_rollout(qpos, qvel, ctrl, warm, nsteps=1, lin=lin, nthreads=cores)
        if i >= args.warmup:
            times.append(time.perf_counter() - t0)
    dt = float(np.median(times)) * args.steps
    value = n * args.steps / dt
    sample = (f"{n} envs per timed step, drawn from the state distribution of the {DEFAULT_NENV[name]}-env workload and sized for ~20 s "
              f"of CPU work over the run, all {cores} host threads; " + CPU_KIND_NOTE)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(name, DEFAULT_NENV[name], lin), "sample_envs_per_step": n},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# BASELINE.json configs[2] / configs[3]: i.i.d. random controls per step and actuator, generated on the device
RANDOM_CTRL = {"drone": (0.0, 13.0), "humanoid": (-0.2, 0.2)}


def workload_name(name: str, nenv: int, lin: bool) -> str:
    if lin:
        tail = "batched LQR + per-step FD (A,B) linearisation + 1 step"
    elif name in RANDOM_CTRL:
        tail = "1 step per launch, random controls U(%g, %g) drawn on the device every step (Philox, b2_random_controls)" % RANDOM_CTRL[name]
        if name == "drone":
            tail += ", episode reset to the initial state below z = 0.5 m"
    else:
        tail = "1 step per launch, zero control"
    return f"{name} batched rollout, N={nenv} envs/GPU, FP64, " + tail


def make_controller(name: str, lin: bool, seed: int = 0, tv_lqr: bool = False):
    """The controller of a workload (counted as the controller, not as the path: SURVEY.md section 8d)."""
    import torch

    from mujoco_template import ControllerCapabilities
    from mujoco_template.batched_controllers import BatchedLQRController

    if lin:
        if name == "cartpole":
            if tv_lqr:  # gains of every env re-synthesised every tick from the env's own (A, B): b2_dlqr + b2_lqr_control_env
                from mujoco_template.batched_controllers import BatchedTVLQRController

                return BatchedTVLQRController(Q=np.diag([10.0, 100.0, 1.0, 1.0]), R=np.array([[0.01]]))
            return BatchedLQRController(Q=np.diag([10.0, 100.0, 1.0, 1.0]), R=np.array([[0.01]]))

        class HoldLin:
            capabilities = ControllerCapabilities(needs_linearization=True)
            def prepare(self, m, d): pass
            def __call__(self, m, d, t): pass
        return HoldLin()
    if name in RANDOM_CTRL:
        from mujoco_template.batched_controllers import BatchedRandomController

        # one library launch per tick (b2_random_controls): Philox controls + for the drone the episode reset of a batched
        # rollout driver -- a drone that comes within 0.5 m of the floor starts again from its initial state (config #3 is
        # free flight: "expect no ground contact")
        lo, hi = RANDOM_CTRL[name]
        return BatchedRandomController(lo, hi, seed=seed, reset_below=(2, 0.5) if name == "drone" else None)
    return None


def run_workload(ctx, name: str, lin: bool, nenv: int, steps: int, warmup: int, *, use_graph: bool, want_e2e: bool,
                 e2e_host_controller: bool, cpu_seconds: float, tv_lqr: bool = False, dump: tuple | None = None) -> dict:
    """Times one workload on this rank's GPU and returns the fields of its JSON line (rank 0's copy is printed)."""
    import torch
    import torch.distributed as dist

    from mujoco_template import BatchedEnv, _capi

    world, rank, local, dev, flush = ctx["world"], ctx["rank"], ctx["local"], ctx["dev"], ctx["flush"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    model = load_model(name)
    controller = make_controller(name, lin, seed=rank, tv_lqr=tv_lqr)
    env = BatchedEnv(model, nenv, controller=controller, device=local)
    env.reset(0 if name == "drone" else (1 if name == "humanoid" else None))
    qpos, qvel = synth_states(model, name, nenv, seed=rank)  # each rank owns its own shard of envs
    env.data.qpos.copy_(torch.as_tensor(qpos.T.copy(), device=dev))
    env.data.qvel.copy_(torch.as_tensor(qvel.T.copy(), device=dev))
    env.forward()
    if name == "drone" and not lin and controller is not None:
        controller.set_reset_state(env.data.qpos, env.data.qvel)

    # per-kernel device times for the roofline: short eager passes with CUDA events around each library launch --
    # first the launches one by one (controller / FD / step), then the fused control tick the timed loop runs
    fuse_default = getattr(env, "fuse_control_tick", False)
    kernel_ms = {}
    for fused in ((False, True) if (lin and fuse_default) else (False,)):
        env.data.backend.profile = {}
        env.fuse_control_tick = fused
        for _ in range(max(warmup, 3)):
            env.step(return_obs=False)
        env.data.backend.profile = {}
        for _ in range(10):
            flush.zero_()
            env.step(return_obs=False)
        torch.cuda.synchronize()
        for k in ("random_controls", "lqr_control", "lqr_control_env", "linearize", "step", "control_tick"):
            v = env.data.backend.kernel_ms(k)[-10:]
            if v:
                kernel_ms[k] = v
    env.data.backend.profile = None
    env.fuse_control_tick = fuse_default
    c0 = _capi.launch_count()
    env.step(return_obs=False)
    per_step_launches = _capi.launch_count() - c0  # library kernels per step (controller tick, FD, step)
    use_graph = use_graph and controller is not None
    if use_graph:
        env.enable_cuda_graph(True)
        for _ in range(3):  # eager call, capture + replay, replay
            env.step(return_obs=False)
    # the timed rollout starts from the configured initial-state distribution (the warm-up / profiling steps above have
    # moved the envs: drones under random thrust eventually reach the floor, the humanoid falls)
    env.data.qpos.copy_(torch.as_tensor(qpos.T.copy(), device=dev))
    env.data.qvel.copy_(torch.as_tensor(qvel.T.copy(), device=dev))
    env.data.qacc_warmstart.zero_()
    env.forward()
    barrier()
    launches0 = _capi.launch_count()
    sampler = ClockSampler(local, ctx["gpu_uuid"])
    sampler.start()
    sampler.first.wait(timeout=10)
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    barrier()
    sampler.in_region = True
    wall0 = time.perf_counter()
    # The host must never be the thing that is timed: the steps are queued behind a spin kernel (torch.cuda._sleep, outside
    # every event pair), 64 at a time, so that each event pair brackets device work that was already waiting in the stream
    # when the device got to it -- no Python, launch latency or rank-to-rank host contention inside the pairs.
    spin_cycles = int(ctx["sm_hz"] * 0.004)
    for i in range(steps):
        if i % 64 == 0:
            torch.cuda._sleep(spin_cycles)
        flush.zero_()  # evict state / outputs from L2 between timed iterations (outside the event pair)
        starts[i].record()
        result = env.step(return_obs=False)
        stops[i].record()
    sampler.sample_now()  # the queued steps are executing now
    barrier()
    wall = time.perf_counter() - wall0
    sampler.in_region = False
    clocks = sampler.stop()
    if dump is not None and rank == 0:  # (directory, file-name prefix); before anything else touches the batch
        dump_outputs(*dump, env, result)
    step_ms = [a.elapsed_time(b) for a, b in zip(starts, stops)]
    total_ms = float(sum(step_ms))
    # graph replays re-launch the captured kernels without passing through the C-ABI counter
    launches = (_capi.launch_count() - launches0) if not use_graph else per_step_launches * steps
    rank_ms = [total_ms / steps]
    if world > 1:
        gathered = [torch.zeros(1, device=dev, dtype=torch.float64) for _ in range(world)]
        dist.all_gather(gathered, torch.tensor([total_ms / steps], device=dev, dtype=torch.float64))
        rank_ms = [float(g.item()) for g in gathered]
    total_ms = max(rank_ms) * steps
    value = nenv * world * steps / (total_ms * 1e-3)

    # untimed: the path's only collective -- gather per-env returns (here: final |x|) across ranks
    ret = env.data.qpos[0].abs().contiguous()
    allret = env.gather(ret)
    flags_bad = int((env.data.flags != 0).sum().item())
    env.forward()  # refresh derived outputs (contact / solver statistics are reported beside the throughput)
    contact_stats = {"mean_ncon": float(env.data.ncon.float().mean().item()), "mean_nefc": float(env.data.nefc.float().mean().item()),
                     "mean_newton_iter": float(env.data.solver_iter.float().mean().item())}

    # ---- roofline of the dominant kernel
    dom = "linearize" if lin else "step"
    if lin and not kernel_ms.get("linearize"):
        dom = "control_tick"  # fused LQR + FD + step launch
    dom_ms = float(np.mean(kernel_ms[dom])) if kernel_ms.get(dom) else float("nan")
    alg_bytes = (LIN_BYTES[name] if lin else STEP_BYTES[name]) * nenv
    traffic = None
    for tname in ("ncu_traffic_r02.json", "ncu_traffic_r01.json"):
        tfile = os.path.join(ROOT, "profiles", tname)
        if traffic is None and os.path.exists(tfile):
            traffic = json.load(open(tfile)).get(f"{name}:{dom}:{nenv}")
    variant = env.data.backend.batch.kernel_variant
    if "warp" in variant:  # large models: warp engine
        kernel_label = "k_warp_linearize" if lin else "k_warp_step_ls"
    else:
        kernel_label = f"k_{dom}<{variant}>"
    achieved = alg_bytes / (dom_ms * 1e-3) / 1e9
    ms_step = total_ms / steps
    mean_of = lambda k: float(np.mean(kernel_ms[k])) if kernel_ms.get(k) else None
    # what the timed step consists of: the fused control tick (FD launch with the env advance riding in it + the state
    # commit) when it is used, else the kernels launched one by one
    in_step = ("control_tick",) if (lin and fuse_default and kernel_ms.get("control_tick")) else tuple(k for k in ("random_controls", "lqr_control", "linearize", "step") if kernel_ms.get(k))
    share = {k: mean_of(k) / ms_step for k in in_step}
    roofline = {"bound": "hbm", "achieved": achieved, "peak": ctx["peak_gbs"], "unit": "GB/s", "frac": achieved / ctx["peak_gbs"],
                "traffic": traffic, "kernel": kernel_label,
                "kernel_ms": dom_ms, "algorithmic_bytes_per_launch": alg_bytes, "peak_source": ctx["peak_src"],
                "kernel_share_of_step": share,
                "kernel_ms_launched_separately": {k: mean_of(k) for k in ("random_controls", "lqr_control", "linearize", "step") if kernel_ms.get(k)},
                "kernel_share_note": "share = device time of the launches the timed step consists of / ms_per_step; with a "
                                     "linearising controller that is b2_control_tick (control law + FD + the env advance in one "
                                     "launch, then the state commit); kernel_ms_launched_separately lists the same work as "
                                     "individual launches (the roofline kernel is timed there)",
                "note": "not HBM bound: a CUDA-core kernel bound by FP64 issue and dependency latency, see roofline_fp64 (SURVEY.md section 8d)"}
    # executed FP64 work: rollouts per launch x flops per step-evaluation
    evals = nenv * ((2 * (2 * model.nv + model.nu)) if lin else 1)
    flops_per_eval, flops_src = flops_per_step_eval(name, lin)
    tf = evals * flops_per_eval / (dom_ms * 1e-3) / 1e12
    roofline_fp64 = {"bound": "fp64_fma", "achieved": tf, "peak": ctx["fp64_peak"], "unit": "TFLOP/s", "frac": tf / ctx["fp64_peak"],
                     "step_evals_per_launch": evals, "flops_per_step_eval": flops_per_eval,
                     "flops_source": flops_src, "peak_source": "b2_fp_peak DFMA microbenchmark, this run"}
    # the ALGORITHMIC count of the same work: the oracle's op counter (tools/op_count.py -> profiles/op_count_r02.json)
    oc_file = os.path.join(ROOT, "profiles", "op_count_r02.json")
    if os.path.exists(oc_file):
        oc = json.load(open(oc_file))["models"][name]
        alg = (oc["linearize_plus_step"]["flops"] - oc["step"]["flops"]) if lin else oc["step"]["flops"]
        roofline_fp64["algorithmic_flops_per_launch_unit"] = alg
        roofline_fp64["algorithmic_unit"] = "one mjd_transitionFD (1 + 2(2nv+nu) serial mj_steps upstream)" if lin else "one mj_step"
        roofline_fp64["algorithmic_tflops"] = alg * nenv / (dom_ms * 1e-3) / 1e12
        roofline_fp64["algorithmic_frac"] = roofline_fp64["algorithmic_tflops"] / ctx["fp64_peak"]
        roofline_fp64["algorithmic_note"] = ("oracle op count (add/mul/div/sqrt = 1, transcendental call = 20) of the scalar algorithm on this "
                                             "workload's states; the kernels execute fewer flops than that where they reuse stages across "
                                             "rollouts or fold the model into the instruction stream")

    # ---- e2e: host buffers through the C-ABI (b2_step_host): H2D state+ctrl, linearise+step, D2H state+(A,B)
    e2e = None
    if want_e2e:
        nq, nv, nu = model.nq, model.nv, model.nu
        hq = torch.as_tensor(qpos.T.copy()).pin_memory(); hv = torch.as_tensor(qvel.T.copy()).pin_memory()
        hu = torch.zeros((nu, nenv), dtype=torch.float64).pin_memory(); hw = torch.zeros((nv, nenv), dtype=torch.float64).pin_memory()
        hA = torch.empty((2 * nv, 2 * nv, nenv), dtype=torch.float64).pin_memory() if lin else None
        hB = torch.empty((2 * nv, nu, nenv), dtype=torch.float64).pin_memory() if lin else None
        st = _capi.State(hq.data_ptr(), hv.data_ptr(), hu.data_ptr(), hw.data_ptr(), None)
        K = getattr(controller, "K", None)
        batch = env.data.backend.batch
        e2e_steps = max(3, min(steps, 50))

        qn, vn, un = hq.numpy(), hv.numpy(), hu.numpy()
        tmp = np.empty(nenv)
        lo = float(model.actuator_ctrlrange[0, 0]) if model.nu else 0.0
        hi = float(model.actuator_ctrlrange[0, 1]) if model.nu else 0.0

        device_lqr = K is not None and not e2e_host_controller
        if device_lqr:
            batch.lqr_set_gain(K, np.asarray(controller._qref_np, dtype=float), np.asarray(controller._uref_np, dtype=float))
        rctrl = RANDOM_CTRL.get(name) if not lin else None
        if rctrl is not None:
            # the host-side controller of configs #3 / #4: random controls per env and actuator, drawn once and held over the
            # e2e steps (drawing 1e6 doubles per step on the host would time NumPy's generator, not the path)
            un[:] = np.random.default_rng(1234 + rank).uniform(rctrl[0], rctrl[1], un.shape)

        def host_step():
            if device_lqr:  # control law on the device: H2D state, [LQR, FD, step] per chunk, D2H state + ctrl + (A, B)
                batch.step_host(st, 1, lin, 1e-6, hA.data_ptr() if lin else None, hB.data_ptr() if lin else None, 0, device_lqr=True)
                return
            if K is not None:  # host-side LQR tick on the host copy of the state: u = clip(-K [q; v]), no temporaries
                rows = (qn[0], qn[1], vn[0], vn[1])
                np.multiply(rows[0], -K[0, 0], out=un[0])
                for k in range(1, 4):
                    np.multiply(rows[k], -K[0, k], out=tmp)
                    np.add(un[0], tmp, out=un[0])
                np.clip(un[0], lo, hi, out=un[0])
            batch.step_host(st, 1, lin, 1e-6, hA.data_ptr() if lin else None, hB.data_ptr() if lin else None, 0)

        for _ in range(3):
            host_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            host_step()
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        h2d = (nq + nv + (0 if device_lqr else nu) + nv) * nenv * 8
        d2h = (nq + nv + nv + (nu if device_lqr else 0) + (2 * nv * (2 * nv + nu) if lin else 0)) * nenv * 8
        e2e_s = float(tt.item()) / e2e_steps
        e2e = {"value": nenv * world / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "steps": e2e_steps, "ms_per_step": e2e_s * 1e3,
               "pcie_gbs_per_gpu": {"h2d": h2d / e2e_s / 1e9, "d2h": d2h / e2e_s / 1e9},
               "pcie_note": "PCIe Gen5 x16 moves ~55 GB/s per direction in practice; d2h / 55 is the fraction of the link the "
                            "(A, B) + state read-back uses",
               "pcie_d2h_frac_of_55gbs": d2h / e2e_s / 1e9 / 55.0,
               "api": "b2_step_host (C-ABI, pinned host buffers, " + ("device LQR law, ctrl returned" if device_lqr else ("host LQR tick" if K is not None else "controls held in the host buffer")) +
                      (", (A, B) written by the FD kernel straight into the mapped host buffers" if lin and os.environ.get("B2_HOST_STAGED") != "1" else "") + ")"}
        # ---- the same exchange with the env batch as `parts` sub-batches, each a closed loop through host buffers of its
        # own (state in, state + ctrl + (A, B) out), submitted without waiting (B2_HOST_ASYNC) and completed one step
        # later: one part's (A, B) cross PCIe while the next part computes.  Every env still does one H2D of its inputs
        # and one D2H of its results per step inside the timed region; only the idle time of the link goes away.
        parts = int(os.environ.get("B2_E2E_PARTS", "2"))
        if parts > 1 and nenv % parts == 0 and (device_lqr or K is None):
            npart = nenv // parts
            cap = batch.model
            subs = []
            for pidx in range(parts):
                sl = slice(pidx * npart, (pidx + 1) * npart)
                pq = hq[:, sl].contiguous().pin_memory(); pv = hv[:, sl].contiguous().pin_memory()
                pu = hu[:, sl].contiguous().pin_memory(); pw = hw[:, sl].contiguous().pin_memory()
                pA = torch.empty((2 * nv, 2 * nv, npart), dtype=torch.float64).pin_memory() if lin else None
                pB = torch.empty((2 * nv, nu, npart), dtype=torch.float64).pin_memory() if lin else None
                sb = _capi.NativeBatch(cap, npart, dev.index or 0, _capi.B2_F64)
                if device_lqr:
                    sb.lqr_set_gain(K, np.asarray(controller._qref_np, dtype=float), np.asarray(controller._uref_np, dtype=float))
                subs.append((sb, _capi.State(pq.data_ptr(), pv.data_ptr(), pu.data_ptr(), pw.data_ptr(), None), (pq, pv, pu, pw, pA, pB)))

            def submit(sub):
                sb, sst, bufs = sub
                sb.step_host(sst, 1, lin, 1e-6, bufs[4].data_ptr() if lin else None, bufs[5].data_ptr() if lin else None, 0,
                             device_lqr=device_lqr, wait=False)

            def run_pipelined(nsteps):
                for sub in subs:
                    submit(sub)
                for _ in range(nsteps - 1):
                    for sub in subs:
                        sub[0].step_host_wait()
                        submit(sub)
                for sub in subs:
                    sub[0].step_host_wait()

            run_pipelined(3)
            barrier()
            t0 = time.perf_counter()
            run_pipelined(e2e_steps)
            barrier()
            tt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            sp = float(tt.item()) / e2e_steps
            finite = all(bool(torch.isfinite(sub[2][0]).all()) for sub in subs)
            api_parts = ("; the batch as %d sub-batches of %d envs, each a closed loop through its own pinned host buffers, submitted "
                         "with B2_HOST_ASYNC and completed by b2_step_host_wait one step later" % (parts, npart))
            piped = {"value": nenv * world / sp, "ms_per_step": sp * 1e3,
                     "pcie_gbs_per_gpu": {"h2d": h2d / sp / 1e9, "d2h": d2h / sp / 1e9}, "parts": parts, "results_finite": finite}
            if piped["value"] > e2e["value"] and finite:  # the faster of the two ways to drive the same exchange is the headline
                e2e["synchronous"] = {"value": e2e["value"], "ms_per_step": e2e["ms_per_step"], "pcie_gbs_per_gpu": e2e["pcie_gbs_per_gpu"],
                                      "api": e2e["api"], "note": "one b2_step_host call per step over the whole batch, returning when the "
                                                                 "results are in the host buffers"}
                e2e.update(piped)
                e2e["pcie_d2h_frac_of_55gbs"] = d2h / sp / 1e9 / 55.0
                e2e["api"] += api_parts
            else:
                piped["api"] = e2e["api"] + api_parts
                e2e["async_parts"] = piped
            del subs
        if lin:
            # the same tick when the consumer of (A, B) lives on the device (a device-side gain synthesis such as b2_dlqr, or
            # the control law itself): (A, B) stay in HBM, the host exchanges state and controls only
            def host_step_ab_on_device():
                batch.step_host(st, 1, lin, 1e-6, None, None, 0, device_lqr=device_lqr)

            for _ in range(3):
                host_step_ab_on_device()
            barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                host_step_ab_on_device()
            barrier()
            tt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            s2 = float(tt.item()) / e2e_steps
            e2e["ab_kept_on_device"] = {"value": nenv * world / s2, "unit": UNIT, "ms_per_step": s2 * 1e3, "h2d_bytes_per_step": h2d,
                                        "d2h_bytes_per_step": d2h - 2 * nv * (2 * nv + nu) * nenv * 8,
                                        "note": "b2_step_host with host_A = host_B = NULL: (A, B) are computed every step and left in "
                                                "device memory for a device-side consumer; not the headline e2e"}
        del hq, hv, hu, hw, hA, hB

    cpu = None
    if rank == 0 and world == 1 and cpu_seconds > 0:
        os.sched_setaffinity(0, ctx["affinity0"])  # the CPU baseline uses every host core
        cpu = cpu_oracle_rate(model, name, lin, cpu_seconds)

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": max(warmup, 3),
        "ms_per_step": ms_step, "ms_per_step_per_rank": rank_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(name, nenv, lin) + (" -- time-varying LQR: every env's gain re-synthesised every tick from its own (A, B) (b2_dlqr)" if tv_lqr else ""), "model": name, "envs_per_gpu": nenv, "global_envs": nenv * world,
                   "l2": "flushed between timed iterations (192 MB memset outside the event pairs)",
                   "launch": "CUDA graph replay of one env.step()" if use_graph else "eager launches",
                   "timing": "CUDA event pair per step; steps queued 64 at a time behind a 4 ms spin kernel, so the pairs bracket "
                             "device work only (no host latency inside); sum over steps, max over ranks",
                   "rollout": f"timed steps are steps 0..{steps} of the rollout from the configured initial-state distribution",
                   "sharding": f"env batch split over {world} rank(s), no inter-step communication"},
        "linearizations_per_sec": (value if lin else 0.0),
        "step_evals_per_sec": value * ((2 * (2 * model.nv + model.nu) + 1) if lin else 1),
        "roofline": roofline, "roofline_fp64": roofline_fp64, "cpu_baseline": cpu, "e2e": e2e,
        "gpu_launches": int(launches), "clocks": clocks, "wall_s_timed_region": wall,
        "bad_env_flags": flags_bad, "gathered_returns": int(allret.numel()), "contact_stats": contact_stats,
        "kernel_variant": variant,
    }
    del env
    torch.cuda.empty_cache()
    return out


def flops_per_step_eval(name: str, lin: bool):
    """Executed FP64 flops per step-evaluation (2*dfma + dadd + dmul thread instructions), counted by ncu on the kernels
    themselves (profiles/ncu_*_r03q.txt, source-page sums): cartpole k_linearize 1.157e8 flops per 655,360 rollouts = 176.5
    -- one thread per env runs the shared position stage once for all velocity / control columns, control columns skip
    the velocity stage too, and the exact zeros / ones of the model are folded out of the instruction stream (ptx_fold.py;
    587 before that pass) -- and k_step 277 per step (962 before); drone k_step 5.25e8 / 262,144 = 2,002 (2,835 before);
    humanoid k_warp_step_ls 3.70e9 / 16,384 = 226,000 in the round-2 capture (profiles/ncu_hum_step_r02d.txt: 100 steps
    into the fall, ~5 contacts, 3.5 Newton iterations; 182,000 in round 1's lighter state).  The oracle's op counter
    (oracle.op_count, BASELINE.md section 4) gives the ALGORITHMIC count of one mj_step for the same states; the executed
    count is what the pipe-utilisation figure needs."""
    table = {"pendulum": 1000.0, "cartpole": 176.5 if lin else 277.0, "drone": 2002.0, "humanoid": 226000.0}
    src = "ncu-counted executed flops (profiles/)" if name != "pendulum" else "a-priori estimate (BASELINE.md section 4)"
    return table[name], src


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    import torch.distributed as dist

    from mujoco_template import _capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    affinity0 = os.sched_getaffinity(0)
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else {"bound": False, "note": "single rank: not bound"}
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    dev = torch.device(f"cuda:{local}")
    peaks_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_file):
        peak_gbs, peak_src = float(json.load(open(peaks_file))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak_gbs, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    try:
        gpu_uuid = str(torch.cuda.get_device_properties(local).uuid)
    except Exception:
        gpu_uuid = None
    ctx = {"world": world, "rank": rank, "local": local, "dev": dev, "affinity0": affinity0, "gpu_uuid": gpu_uuid,
           "flush": torch.empty(192 * 1024 * 1024 // 4, dtype=torch.float32, device=dev),  # > 126 MB L2
           "fp64_peak": _capi.fp_peak(64, local), "peak_gbs": peak_gbs, "peak_src": peak_src,
           "sm_hz": torch.cuda.get_device_properties(local).clock_rate * 1e3}
    name = args.model
    lin = not args.no_linearize
    common = dict(use_graph=not args.no_graph, want_e2e=not args.no_e2e, e2e_host_controller=args.e2e_host_controller)
    dump = lambda prefix: (args.dump_outputs, prefix) if args.dump_outputs else None  # noqa: E731
    out = run_workload(ctx, name, lin, args.nenv or DEFAULT_NENV[name], args.steps, args.warmup,
                       cpu_seconds=0.0 if args.no_cpu_baseline else args.cpu_seconds, dump=dump(""), **common)
    out["host_binding"] = numa
    # BASELINE.json configs[2] / configs[3] ride along with the headline workload (same run, same clocks, same rank
    # count): drone free flight under random thrust and the humanoid with contacts, step only
    if name == "cartpole" and lin and args.nenv is None and not args.no_secondary:
        out["secondary"] = {}
        for sname in ("drone", "humanoid"):
            sec = run_workload(ctx, sname, False, DEFAULT_NENV[sname], args.steps, args.warmup,
                               cpu_seconds=0.0 if args.no_cpu_baseline else min(args.cpu_seconds, 5.0), dump=dump(sname + "_"), **common)
            out["secondary"][sname] = {k: sec[k] for k in ("value", "unit", "ms_per_step", "ms_per_step_per_rank", "steps", "config", "roofline",
                                                           "roofline_fp64", "cpu_baseline", "e2e", "gpu_launches", "contact_stats",
                                                           "bad_env_flags", "kernel_variant", "clocks")}
        # config #2 read literally ("per-step FD (A, B) linearisation for LQR"): the same workload with every env's gain
        # re-synthesised every tick from its own latest (A, B) -- DARE + gain (b2_dlqr), per-env control law, FD, step
        tv = run_workload(ctx, "cartpole", True, DEFAULT_NENV["cartpole"], args.steps, args.warmup, use_graph=not args.no_graph,
                          want_e2e=False, e2e_host_controller=False, cpu_seconds=0.0, tv_lqr=True, dump=dump("cartpole_tv_lqr_"))
        out["secondary"]["cartpole_tv_lqr"] = {k: tv[k] for k in ("value", "unit", "ms_per_step", "ms_per_step_per_rank", "steps", "config",
                                                                  "gpu_launches", "bad_env_flags", "kernel_variant", "clocks")}
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
