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

    def rollout(self, nsteps: int | None = None, *, controls=None, record: bool = False):
        """``nsteps`` steps of every env in one kernel launch (the warp engine of large models: one launch per step).

        Open loop: the controller is not called.  Without ``controls`` the current controls are held.  ``controls`` is a
        ``(nenv, T, nu)`` tensor (any strides; on the batch's device, in its dtype): row t is applied at step t, and
        ``data.ctrl`` holds row T-1 afterwards.  ``nsteps`` may then be omitted; if given it must equal T.  It is handed to
        the kernel as a ``(T, nu, nenv)`` layout, which costs no copy when ``controls`` is already a permuted view of such a
        buffer.  Controls outside ``ctrlrange`` are clamped inside the physics, as in ``step``.

        ``record=True`` returns ``{"qpos": (nenv, T, nq), "qvel": (nenv, T, nv)}`` -- the state after every step -- plus
        ``"sensordata": (nenv, T, nsensordata)`` when the model has sensors (the reading each step leaves, as ``mj_step``
        leaves it), as permuted views of fresh ``(T, dim, nenv)`` buffers.  An env that diverges is flagged and frozen: its
        remaining rows repeat its frozen state, and its remaining sensor rows are NaN.  Otherwise returns None.
        ``data.time`` advances by T timesteps and the derived arrays are those of the last step."""
        backend = self.data.backend
        seq, nsteps = self._control_sequence("rollout", controls, nsteps)
        out = None
        if seq is None and not record:
            backend.step(nsteps)
        else:
            out = backend.rollout(seq, nsteps, record)
        self._advance_time(nsteps)
        self._substep += nsteps
        if not record:
            return None
        traj = {"qpos": out[0].permute(2, 0, 1), "qvel": out[1].permute(2, 0, 1)}
        if out[2] is not None:
            traj["sensordata"] = out[2].permute(2, 0, 1)
        return traj

    def rollout_feedback(self, controls, K, qpos, qvel, *, k=None, alpha=None, record: bool = False):
        """``T`` steps of every env under the time-varying LQR law about a nominal trajectory, in one kernel launch (the
        warp engine of large models: two per step).  At step t the control is

            u_t = clip(controls[:, t] + alpha k[:, t] - K[:, t] [q (-) qpos[:, t] ; v - qvel[:, t]], ctrlrange)

        where (-) is ``mj_differentiatePos`` (the tangent space of ``linearize_rollout``'s ``A``) and the clip applies to
        ctrl-limited actuators.  This is the forward pass of iLQR (``linearize_rollout`` -> ``batched_tvlqr`` ->
        ``rollout_feedback``) and time-varying LQR tracking of a nominal trajectory.  The controller is not called.

        ``controls`` ``(nenv, T, nu)`` is the nominal control sequence (validated as in ``rollout``); ``K`` ``(nenv, T, nu,
        2nv)`` and ``k`` ``(nenv, T, nu)`` (None: zero) are ``batched_tvlqr``'s gains; ``qpos`` ``(nenv, T or T+1, nq)`` and
        ``qvel`` ``(nenv, T or T+1, nv)`` the nominal states -- ``linearize_rollout``'s ``"qpos"`` / ``"qvel"`` as they are;
        ``alpha`` a float or an ``(nenv,)`` tensor (per-env line search; None: 1).  All on the batch's device, in its
        dtype; views of env-fastest storage are handed over without a copy.

        ``data.time`` and the step counter advance by T as in ``rollout``; ``data.ctrl`` holds the last applied control.
        ``record=True`` returns ``rollout``'s dict plus ``"ctrl": (nenv, T, nu)``, the applied controls (NaN from the step
        an env is frozen at).  Otherwise returns None."""
        import torch

        m, n = self.model, self.nenv
        seq, T = self._control_sequence("rollout_feedback", controls, None)
        if seq is None:
            raise ConfigError("rollout_feedback: controls (the nominal control sequence) are required")
        ref = self.data.qpos
        nx = 2 * m.nv

        def layout(name, t, shapes):
            if not isinstance(t, torch.Tensor) or tuple(t.shape) not in shapes:
                got = tuple(t.shape) if isinstance(t, torch.Tensor) else type(t).__name__
                raise ConfigError(f"rollout_feedback: {name} must have shape {' or '.join(map(str, shapes))}, got {got}")
            if t.device != ref.device or t.dtype != ref.dtype:
                raise ConfigError(f"rollout_feedback: {name}: expected {ref.dtype} on {ref.device}, got {t.dtype} on {t.device}")
            return t.permute(*range(1, t.dim()), 0).contiguous()  # env fastest; no copy for a view of such storage

        Ks = layout("K", K, [(n, T, m.nu, nx)])
        ks = None if k is None else layout("k", k, [(n, T, m.nu)])
        qs = layout("qpos", qpos, [(n, T, m.nq), (n, T + 1, m.nq)])
        vs = layout("qvel", qvel, [(n, T, m.nv), (n, T + 1, m.nv)])
        if alpha is None:
            a = None
        elif isinstance(alpha, torch.Tensor):
            if tuple(alpha.shape) != (n,) or alpha.device != ref.device or alpha.dtype != ref.dtype:
                raise ConfigError(f"rollout_feedback: alpha must be a float or a ({n},) {ref.dtype} tensor on {ref.device}")
            a = alpha.contiguous()
        else:
            a = torch.full((n,), float(alpha), dtype=ref.dtype, device=ref.device)
        out = self.data.backend.rollout_feedback(seq, qs, vs, Ks, ks, a, T, record)
        self._advance_time(T)
        self._substep += T
        if not record:
            return None
        traj = {"qpos": out[1].permute(2, 0, 1), "qvel": out[2].permute(2, 0, 1), "ctrl": out[0].permute(2, 0, 1)}
        if out[3] is not None:
            traj["sensordata"] = out[3].permute(2, 0, 1)
        return traj

    def traj_cost(self, qpos, qvel, ctrl, Q, R, Qf=None, *, qpos_ref, qvel_ref=None, ctrl_ref=None, grad: bool = False):
        """Tracking cost of every env's trajectory, in one kernel launch (``b2_traj_cost``):

            e_t = [q_t (-) qref_t ; v_t - vref_t]  (t = 0..T),   w_t = u_t - uref_t  (t < T)
            J   = sum_{t<T} (1/2 e_t'Q e_t + 1/2 w_t'R w_t) + 1/2 e_T'Qf e_T

        where (-) is ``mj_differentiatePos`` (the tangent space of ``linearize_rollout``'s ``A``: a quaternion log for a free
        joint).  ``qpos`` ``(nenv, T+1, nq)`` and ``qvel`` ``(nenv, T+1, nv)`` are ``linearize_rollout``'s ``"qpos"`` /
        ``"qvel"`` as they are, ``ctrl`` a ``(nenv, T, nu)`` control tensor; ``qpos_ref`` (required), ``qvel_ref`` and
        ``ctrl_ref`` (None: zero) are ``(nenv, rows, dim)``, ``(rows, dim)`` or ``(dim,)`` tensors -- the last two are
        broadcast over envs (and steps) once per call.  All on the batch's device, in its dtype.  ``Q``, ``R`` and ``Qf``
        (default ``Q``) are exactly symmetric host matrices.

        Returns ``J`` ``(nenv,)``; with ``grad=True`` ``(J, q, r)``, where ``q`` ``(nenv, T+1, 2nv)`` is the gradient with
        respect to the tangent deviation of ``A`` and ``rollout_feedback`` (``x = xbar (+) dx``; it differs from ``Q e`` on
        free joints' rotations by ``Jr^-1``) and ``r`` ``(nenv, T, nu)`` is ``R w``: ``batched_tvlqr``'s ``q`` / ``r``, read
        without a copy.  A NaN row makes its own env's results NaN only.  Neither the state, ``data.time`` nor the step
        counter moves."""
        import torch

        m, n = self.model, self.nenv
        if m.nu == 0:
            raise ConfigError("traj_cost: the model has no actuators (nu=0)")
        ref = self.data.qpos
        nx = 2 * m.nv

        def check(name, t, shapes):
            if not isinstance(t, torch.Tensor) or tuple(t.shape) not in shapes:
                got = tuple(t.shape) if isinstance(t, torch.Tensor) else type(t).__name__
                raise ConfigError(f"traj_cost: {name} must have shape {' or '.join(map(str, shapes))}, got {got}")
            if t.device != ref.device or t.dtype != ref.dtype:
                raise ConfigError(f"traj_cost: {name}: expected {ref.dtype} on {ref.device}, got {t.dtype} on {t.device}")

        if not isinstance(ctrl, torch.Tensor) or ctrl.dim() != 3 or ctrl.shape[1] < 1:
            raise ConfigError(f"traj_cost: ctrl must be a (nenv={n}, T, nu={m.nu}) tensor with T >= 1")
        T = int(ctrl.shape[1])
        rows = {"qpos": T + 1, "qvel": T + 1, "ctrl": T}
        dims = {"qpos": m.nq, "qvel": m.nv, "ctrl": m.nu}

        def traj(name, t):  # (nenv, rows, dim) -> (rows, dim, nenv) env fastest; no copy for a view of such storage
            check(name, t, [(n, rows[name], dims[name])])
            return t.permute(1, 2, 0).contiguous()

        def reference(name, t):
            if t is None:
                return None
            r, d = rows[name], dims[name]
            check(f"{name}_ref", t, [(n, r, d), (r, d), (d,)])
            if t.dim() == 3:
                return t.permute(1, 2, 0).contiguous()
            return (t[:, :, None] if t.dim() == 2 else t[None, :, None]).expand(r, d, n).contiguous()

        def host(name, M, k):
            M = np.asarray(M.cpu() if hasattr(M, "cpu") else M, dtype=float)
            if M.shape != (k, k):
                raise ConfigError(f"traj_cost: {name} must be ({k}, {k}), got {M.shape}")
            return np.ascontiguousarray(M).reshape(-1)

        qs, vs, us = traj("qpos", qpos), traj("qvel", qvel), traj("ctrl", ctrl)
        if qpos_ref is None:
            raise ConfigError("traj_cost: qpos_ref is required")
        qr, vr, ur = reference("qpos", qpos_ref), reference("qvel", qvel_ref), reference("ctrl", ctrl_ref)
        Qh, Rh = host("Q", Q, nx), host("R", R, m.nu)
        Qfh = Qh if Qf is None else host("Qf", Qf, nx)
        J, q, r = self.data.backend.traj_cost(qs, vs, us, qr, vr, ur, Qh, Rh, Qfh, T, bool(grad))
        if not grad:
            return J
        return J, q.permute(2, 0, 1), r.permute(2, 0, 1)

    def _control_sequence(self, what: str, controls, nsteps):
        """Validates a ``(nenv, T, nu)`` control tensor and ``nsteps``; returns the controls as a ``(T, nu, nenv)`` layout
        (None without controls) and T."""
        m = self.model
        seq = None
        if controls is not None:
            import torch

            if m.nu == 0:
                raise ConfigError(f"{what}(controls=...): the model has no actuators (nu=0)")
            if not isinstance(controls, torch.Tensor) or controls.dim() != 3 or controls.shape[0] != self.nenv or controls.shape[2] != m.nu:
                raise ConfigError(f"{what}(controls=...): expected a (nenv={self.nenv}, T, nu={m.nu}) tensor, got "
                                  f"{tuple(controls.shape) if isinstance(controls, torch.Tensor) else type(controls).__name__}")
            ref = self.data.qpos
            if controls.device != ref.device or controls.dtype != ref.dtype:
                raise ConfigError(f"{what}(controls=...): expected {ref.dtype} on {ref.device}, got {controls.dtype} on {controls.device}")
            if nsteps is not None and int(nsteps) != controls.shape[1]:
                raise ConfigError(f"{what}: nsteps={nsteps} disagrees with the {controls.shape[1]} rows of controls")
            nsteps = controls.shape[1]
            seq = controls.permute(1, 2, 0).contiguous()  # (T, nu, nenv); no copy for a permuted (T, nu, nenv) buffer
        if nsteps is None or int(nsteps) < 1:
            raise ConfigError("nsteps must be >= 1")
        return seq, int(nsteps)

    def linearize_rollout(self, controls=None, nsteps: int | None = None, *, eps: float | None = None, centered: bool = True,
                          sensors: bool = False):
        """Transition Jacobians at every step of an open-loop control sequence (iLQR / DDP, time-varying LQR about a
        nominal trajectory): the loop ``ctrl <- controls[:, t]; linearize(); step(1)`` run on a copy of the state, in two
        kernel launches on the lane engine for any T.  ``controls`` and ``nsteps`` as in ``rollout`` (without controls the
        current ones are held).  The controller is not called, and neither the state, ``data.time`` nor the
        control-decimation counter moves (only flags are OR-ed in, as the loop would).

        Returns a dict of ``(nenv, ...)`` views of fresh buffers: ``"qpos": (nenv, T+1, nq)`` and ``"qvel": (nenv, T+1, nv)``
        -- the nominal trajectory, row 0 the current state and row t+1 the state after step t -- and ``"A": (nenv, T, 2nv,
        2nv)``, ``"B": (nenv, T, 2nv, nu)``, the Jacobians about row t.  ``sensors=True`` on a model with sensors adds
        ``"C": (nenv, T, nsensordata, 2nv)``, ``"D": (nenv, T, nsensordata, nu)`` and the nominal readings
        ``"sensordata": (nenv, T, nsensordata)``.  An env that diverges is frozen as in ``rollout``."""
        seq, nsteps = self._control_sequence("linearize_rollout", controls, nsteps)
        eps = self.lin_eps if eps is None else float(eps)
        A, B, C, D, qpos, qvel, _, sd = self.data.backend.linearize_rollout(seq, nsteps, eps, centered, sensors)
        out = {"qpos": qpos.permute(2, 0, 1), "qvel": qvel.permute(2, 0, 1), "A": A.permute(3, 0, 1, 2), "B": B.permute(3, 0, 1, 2)}
        if C is not None:
            out.update(C=C.permute(3, 0, 1, 2), D=D.permute(3, 0, 1, 2), sensordata=sd.permute(2, 0, 1))
        return out

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
