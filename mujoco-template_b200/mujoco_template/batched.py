"""BatchedEnv: N independent copies of one model advanced by single kernel launches.

New relative to the reference (which has one env and no parallelism, SURVEY.md section 0); it
keeps ``Env``'s step semantics (reference ``mujoco_template/env.py:164-231``) -- control
decimation, controller -> (A, B) -> Jacobians -> step ordering, the one-or-list ``info`` rule
-- with every array carrying a trailing env axis:

* ``data.qpos`` ... are ``(dim, nenv)`` CUDA tensors (SoA, env index fastest) that the kernels
  update in place; a vectorised controller writes ``data.ctrl[:]`` without any host sync;
* ``info['A']`` is an ``(nenv, 2nv, 2nv)`` view and ``info['B']`` an ``(nenv, 2nv, nu)`` view of the
  SoA buffers the FD kernel wrote; Jacobians are ``(nenv, 3, nv)`` views.

Sharding across GPUs is by construction: one ``BatchedEnv`` per rank over its slice of envs
(``shard_range``); nothing is exchanged during stepping.
"""

from __future__ import annotations

import warnings

from collections.abc import Iterable, Iterator
from typing import Any

import numpy as np

from . import _capi
from . import _mj as mj
from ._typing import InfoDict
from .control import Controller
from .env import StepResult, _one_or_many
from .exceptions import ConfigError, NameLookupError, TemplateError
from .jacobians import resolve_jacobian_token
from .observations import ObservationSpec

_KIND_CODE = {"site": _capi.JAC_SITE, "body": _capi.JAC_BODY, "bodycom": _capi.JAC_BODYCOM, "subtreecom": _capi.JAC_SUBTREECOM}


def shard_range(total: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous block of env indices owned by ``rank`` (SURVEY.md section 8e)."""
    if world < 1 or not 0 <= rank < world:
        raise ConfigError("invalid rank/world for sharding")
    return (total * rank) // world, (total * (rank + 1)) // world


class BatchedObservationExtractor:
    """Tensor counterpart of ``ObservationExtractor``: same keys, trailing env axis."""

    def _warn_once(self, key: str, msg: str) -> None:
        if key not in self._warned:
            self._warned.add(key)
            warnings.warn(msg, RuntimeWarning, stacklevel=3)

    def __init__(self, model: mj.MjModel, spec: ObservationSpec):
        self._warned: set[str] = set()
        self.model, self.spec = model, spec
        O = mj.mjtObj

        def ids(objtype, names):
            out = []
            for n in names:
                i = mj.mj_name2id(model, objtype, n)
                if i < 0:
                    raise NameLookupError(f"Name not found in model: {n}")
                out.append(i)
            return out

        self.site_ids = ids(O.mjOBJ_SITE, spec.sites_pos)
        self.body_ids = ids(O.mjOBJ_BODY, spec.bodies_pos)
        self.geom_ids = ids(O.mjOBJ_GEOM, spec.geoms_pos)
        self.subtree_ids = ids(O.mjOBJ_BODY, spec.subtree_com)

    @staticmethod
    def _rows(src, ids):
        n = src.shape[1]
        return src.reshape(-1, 3, n)[ids]

    def __call__(self, data: mj.BatchData):
        import torch

        s = self.spec
        pick = (lambda t: t.clone()) if s.copy else (lambda t: t)
        out = {}
        if s.include_qpos:
            out["qpos"] = pick(data.qpos)
        if s.include_qvel:
            out["qvel"] = pick(data.qvel)
        if s.include_act:
            out["act"] = data.qpos.new_zeros((0, data.nenv))
        if s.include_ctrl:
            out["ctrl"] = pick(data.ctrl)
        if s.include_sensordata:
            if self.model.nsensordata == 0:
                self._warn_once("sensordata", "ObservationSpec requested sensordata but model has none; returning an empty array instead.")
                out["sensordata"] = data.qpos.new_zeros((0, data.nenv))
            else:
                out["sensordata"] = pick(data.sensordata)
        if s.include_time:
            out["time"] = data.qpos.new_full((1, data.nenv), float(data.time))
        if self.site_ids:
            out["sites_pos"] = self._rows(data.site_xpos, self.site_ids)
        if self.body_ids:
            out["bodies_pos"] = self._rows(data.xipos if s.bodies_inertial else data.xpos, self.body_ids)
        if self.geom_ids:
            out["geoms_pos"] = self._rows(data.geom_xpos, self.geom_ids)
        if self.subtree_ids:
            out["subtree_com"] = self._rows(data.subtree_com, self.subtree_ids)
        for name, producer in s.extras.items():
            if name in out:
                raise ValueError(f"extras[{name!r}] duplicates an existing observation key")
            fn = producer.fn if hasattr(producer, "fn") else producer
            out[name] = fn(self.model, data)
        if s.as_dict:
            return out
        parts = [out[k].reshape(-1, data.nenv) for k in sorted(out)]
        return torch.cat(parts, dim=0) if parts else data.qpos.new_zeros((0, data.nenv))


class BatchedEnv:
    def __init__(self, model: mj.MjModel, nenv: int, *, controller: Controller | None = None,
                 obs_spec: ObservationSpec | None = None, control_decimation: int = 1, device: int | None = None,
                 precision: int = 64, reward_fn=None, done_fn=None, info_fn=None, lin_eps: float = 1e-6,
                 data: mj.BatchData | None = None, derived: str = "lazy"):
        """``derived``: what ``step(return_obs=False)`` does about the derived arrays (``xpos``, ``site_xpos``,
        ``sensordata``, ...).  ``"lazy"`` (default): the step runs without them and parks its pre-step state; whoever reads
        ``data.xpos`` etc. afterwards gets the same values through one extra forward pass (``b2_refresh_derived``) -- right
        when nothing, or only an occasional hook, reads them.  ``"eager"``: every step exports them, as ``mj_step`` does --
        right when a hook, reward function or recorder reads them after every step.  The choice is the caller's and does
        not depend on call history."""
        if derived not in ("lazy", "eager"):
            raise ConfigError("derived must be 'lazy' or 'eager'")
        self.derived = derived
        if control_decimation < 1:
            raise ConfigError("control_decimation must be >= 1")
        if nenv < 1:
            raise ConfigError("nenv must be >= 1")
        self.model = model
        self.nenv = int(nenv)
        self.data = data if data is not None else mj.BatchData(model, nenv, device=device, precision=precision)
        self.controller = controller
        self.control_decimation = int(control_decimation)
        self.lin_eps = float(lin_eps)
        # a device-resident control law (BatchedLQRController) is evaluated inside the FD and step kernels
        # (b2_control_tick: two launches per tick instead of controller + FD + step)
        self.fuse_control_tick = True
        self.reward_fn, self.done_fn, self.info_fn = reward_fn, done_fn, info_fn
        self._obs_spec = obs_spec if obs_spec is not None else ObservationSpec(include_sensordata=False)
        self.extractor = BatchedObservationExtractor(model, self._obs_spec)
        self._substep = 0
        self._jac_ids: list[tuple[str, str, int]] = []
        if controller is not None:
            if model.nu == 0:
                raise TemplateError("Model has no actuators (nu=0).")
            self._jac_ids = [(tok,) + resolve_jacobian_token(model, tok) for tok in controller.capabilities.needs_jacobians]
            controller.prepare(self.model, self.data)

    @classmethod
    def from_xml_path(cls, xml_path: str, nenv: int, *, keyframe: int | str | None = None, auto_reset: bool = True,
                      **kwargs: Any) -> "BatchedEnv":
        env = cls(mj.MjModel.from_xml_path(xml_path), nenv, **kwargs)
        if keyframe is not None and not auto_reset:
            raise ConfigError("auto_reset=False is incompatible with specifying a keyframe")
        if auto_reset:
            env.reset(keyframe)
        return env

    # ---- lifecycle
    def _key_index(self, keyframe: int | str) -> int:
        if isinstance(keyframe, str):
            idx = mj.mj_name2id(self.model, mj.mjtObj.mjOBJ_KEY, keyframe)
            if idx < 0:
                raise NameLookupError(f"Keyframe name not found: {keyframe}")
            return idx
        idx = int(keyframe)
        if not 0 <= idx < self.model.nkey:
            raise ConfigError(f"Keyframe index out of range: {idx}")
        return idx

    def reset(self, keyframe: int | str | None = None):
        if keyframe is None:
            mj.mj_resetData(self.model, self.data)
        else:
            mj.mj_resetDataKeyframe(self.model, self.data, self._key_index(keyframe))
        mj.mj_forward(self.model, self.data)
        self._substep = 0
        if self.controller is not None:
            self.controller.prepare(self.model, self.data)
        return self.extractor(self.data)

    def forward(self) -> None:
        mj.mj_forward(self.model, self.data)

    # ---- hot path
    def linearize(self, eps: float | None = None, centered: bool = True, *, sensors: bool = False):
        """(A, B) of every env: ``(nenv, 2nv, 2nv)`` and ``(nenv, 2nv, nu)`` views of fresh SoA buffers -- or of the
        controller's own ``lin_out`` buffers when it provides them (a controller that consumes the linearisation on the
        device, e.g. ``BatchedTVLQRController``, needs them at a fixed address from tick to tick).

        ``sensors=True`` returns (A, B, C, D): also the sensor Jacobians C = d sensordata / dx ``(nenv, nsensordata, 2nv)``
        and D = d sensordata / du ``(nenv, nsensordata, nu)`` (fresh buffers), from the same FD launch."""
        out = getattr(self.controller, "lin_out", None)
        eps = self.lin_eps if eps is None else float(eps)
        if sensors:
            mats = self.data.backend.linearize_sensors(eps, centered, out=None if out is None else (*out, None, None))
            return tuple(t.permute(2, 0, 1) for t in mats)
        A, B = self.data.backend.linearize(eps, centered, out=out)
        return A.permute(2, 0, 1), B.permute(2, 0, 1)

    def jacobians(self, tokens: Iterable[str] | None = None):
        items = self._jac_ids if tokens is None else [(t,) + resolve_jacobian_token(self.model, t) for t in tokens]
        out = {}
        for token, kind, idx in items:
            want_rot = kind in ("site", "body")
            jp, jr = self.data.backend.jacobian(_KIND_CODE[kind], idx, want_rot)
            entry = {"jacp": jp.permute(2, 0, 1)}
            if want_rot:
                entry["jacr"] = jr.permute(2, 0, 1)
            out[token] = entry
        return out

    def _device_work(self, n: int, lazy: bool = False):
        """Controller ticks, (A, B), Jacobians and n physics steps: device work only (no host sync).

        ``lazy``: the caller does not read derived arrays now (``step(return_obs=False)``), so the last step runs without
        derived outputs and parks its pre-step state (``b2_step_lazy``); whoever reads ``data.xpos`` etc. later gets
        them from ``b2_refresh_derived`` -- same values, produced on demand."""
        lin_A, lin_B, jacs = [], [], []
        backend = self.data.backend
        pending = 0  # consecutive steps with no controller tick are fused into one launch
        fuse = (self.fuse_control_tick and self.controller is not None and not self._jac_ids
                and getattr(self.controller.capabilities, "needs_linearization", False)
                and hasattr(self.controller, "device_law_ready") and hasattr(backend, "control_tick"))
        for _ in range(n):
            if self.controller is not None and self._substep % self.control_decimation == 0:
                if pending:
                    backend.step(pending)
                    pending = 0
                if fuse and self.controller.device_law_ready(self.data):
                    # controller law + (A, B) + this step in one launch (b2_control_tick)
                    A, B = backend.control_tick(self.lin_eps, True, True, derived=False)
                    self._ticks_defer_derived = True
                    lin_A.append(A.permute(2, 0, 1))
                    lin_B.append(B.permute(2, 0, 1))
                    self._substep += 1
                    continue
                self.controller(self.model, self.data, float(self.data.time))
                caps = self.controller.capabilities
                if caps.needs_linearization:
                    A, B = self.linearize()
                    lin_A.append(A)
                    lin_B.append(B)
                if self._jac_ids:
                    jacs.append(self.jacobians())
            pending += 1
            self._substep += 1
        if pending:
            if lazy and hasattr(backend, "step_lazy") and int(self.model.opt.integrator) == 0:
                if pending > 1:
                    backend.step(pending - 1, derived=False)
                backend.step_lazy()
            else:
                backend.step(pending)
        return lin_A, lin_B, jacs

    def _advance_time(self, n: int) -> None:
        h = float(self.model.opt.timestep)
        for _ in range(n):
            self.data.time += h  # repeated addition, as upstream accumulates mjData.time

    def enable_cuda_graph(self, enabled: bool = True) -> None:
        """Replay ``step()`` (controller tick + (A, B) + Jacobians + physics step) as one CUDA graph.

        Valid when the controller is pure tensor code that does not depend on ``t`` and
        ``control_decimation == 1``.  The first graphed call runs eagerly, the second captures.
        ``info['A']`` / ``info['B']`` / Jacobians then alias graph-owned buffers that the next
        ``step()`` overwrites (clone them to keep a history)."""
        if enabled and self.control_decimation != 1:
            raise ConfigError("CUDA-graph stepping requires control_decimation == 1")
        self._graph_enabled = bool(enabled)
        self._graphs = {}  # one captured graph per flavour of step(): eager / lazy derived outputs

    def _graphed_work(self, lazy: bool = False):
        import torch

        g = self._graphs.setdefault(bool(lazy), {"warm": False, "graph": None, "out": None, "stale": False})
        backend = self.data.backend
        if not g["warm"]:  # eager first call: loads the kernels, makes the model image resident
            g["warm"] = True
            return self._device_work(1, lazy)
        if g["graph"] is None:
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                g["out"] = self._device_work(1, lazy)
            g["graph"] = graph
            g["stale"] = bool(backend.derived_stale)  # whether the captured work left the derived arrays for later
        else:
            self._substep += 1
        g["graph"].replay()
        backend.derived_stale = g["stale"]
        return g["out"]

    def step(self, n: int = 1, *, return_obs: bool = True) -> StepResult:
        if n < 1:
            raise ConfigError("BatchedEnv.step(n): n must be >= 1")
        info: InfoDict = {}
        # derived arrays are produced on demand when the caller takes no observation (see `derived` in __init__)
        lazy = not return_obs and self.derived == "lazy"
        if getattr(self, "_graph_enabled", False) and n == 1 and self.controller is not None:
            lin_A, lin_B, jacs = self._graphed_work(lazy)
        else:
            lin_A, lin_B, jacs = self._device_work(n, lazy)
        self._advance_time(n)
        if lin_A:
            info["A"], info["B"] = _one_or_many(lin_A), _one_or_many(lin_B)
        if jacs:
            info["jacobians"] = _one_or_many(jacs)
        obs = self.extractor(self.data) if return_obs else None
        reward = self.reward_fn(self.model, self.data, obs) if self.reward_fn else None
        done = self.done_fn(self.model, self.data, obs) if self.done_fn else False
        if self.info_fn:
            for key, value in self.info_fn(self.model, self.data, obs).items():
                if key in info:
                    raise TemplateError(f"info key collision: {key}")
                info[key] = value
        return StepResult(obs=obs, reward=reward, done=done, info=info)

    def rollout(self, nsteps: int) -> None:
        """``nsteps`` steps with the current controls held, fused in one kernel launch."""
        if nsteps < 1:
            raise ConfigError("nsteps must be >= 1")
        self.data.backend.step(int(nsteps))
        self._advance_time(int(nsteps))
        self._substep += int(nsteps)

    def passive(self, *, duration: float | None = None, max_steps: int | None = None, hooks=None,
                return_obs: bool = True) -> Iterator[StepResult]:
        from .runtime import iterate_passive

        yield from iterate_passive(self, duration=duration, max_steps=max_steps, hooks=hooks, return_obs=return_obs)

    # ---- end of run: the only collective of the path
    def gather(self, tensor, world_size: int | None = None):
        """All-gather a per-rank ``(..., nenv_local)`` tensor along the env axis (NCCL over NVLink)."""
        import torch
        import torch.distributed as dist

        if not dist.is_available() or not dist.is_initialized():
            return tensor
        world = dist.get_world_size() if world_size is None else world_size
        # shard_range hands out blocks that differ by one env when the total does not divide: exchange the block
        # lengths first and pad to the longest
        n_local = torch.tensor([tensor.shape[-1]], device=tensor.device, dtype=torch.int64)
        counts = [torch.zeros_like(n_local) for _ in range(world)]
        dist.all_gather(counts, n_local)
        counts = [int(c.item()) for c in counts]
        n_max = max(counts)
        send = tensor.contiguous()
        if send.shape[-1] < n_max:
            send = torch.nn.functional.pad(send, (0, n_max - send.shape[-1]))
        parts = [torch.empty_like(send) for _ in range(world)]
        dist.all_gather(parts, send)
        return torch.cat([p[..., :c] for p, c in zip(parts, counts)], dim=-1)


__all__ = ["BatchedEnv", "BatchedObservationExtractor", "shard_range"]
