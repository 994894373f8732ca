"""MuJoCo-shaped facade over the B200 C-ABI.

The reference calls a small set of ``mujoco`` symbols on its hot path (enumerated in the
reference stub ``mujoco_template/mujoco.pyi:60-75``).  This module provides those names with
the same argument meaning, backed by ``libb2mj.so`` instead of ``libmujoco``:

``MjModel.from_xml_path/from_xml_string``, ``MjData``, ``mj_step``, ``mj_forward``,
``mj_resetData``, ``mj_resetDataKeyframe``, ``mj_name2id``, ``mj_id2name``,
``mjd_transitionFD``, ``mj_integratePos``, ``mj_differentiatePos``,
``mj_jacSite/Body/BodyCom/SubtreeCom``, ``mj_subtreeCoM``, ``mjtObj``, ``mjtJoint``.

State lives in SoA ``(dim, nenv)`` buffers.  ``MjData`` (one env) keeps them in page-locked,
device-mapped host memory, so ``data.qpos`` etc. are ordinary NumPy views that the kernels
read and write in place (zero-copy, like the reference's views of ``mjData``).
``BatchData`` (N envs) keeps them as CUDA ``torch`` tensors.
"""

from __future__ import annotations

import ctypes as C
import os
from types import SimpleNamespace
from typing import Any

import numpy as np

from . import _capi, _layout, mjcf
from .exceptions import ConfigError, TemplateError


class mjtObj:
    mjOBJ_UNKNOWN = 0
    mjOBJ_BODY = 1
    mjOBJ_XBODY = 2
    mjOBJ_JOINT = 3
    mjOBJ_DOF = 4
    mjOBJ_GEOM = 5
    mjOBJ_SITE = 6
    mjOBJ_TENDON = 18
    mjOBJ_ACTUATOR = 19
    mjOBJ_SENSOR = 20
    mjOBJ_KEY = 25


class mjtJoint:
    mjJNT_FREE = 0
    mjJNT_BALL = 1
    mjJNT_SLIDE = 2
    mjJNT_HINGE = 3


_OBJ_KIND = {
    mjtObj.mjOBJ_BODY: "body", mjtObj.mjOBJ_XBODY: "body", mjtObj.mjOBJ_JOINT: "joint", mjtObj.mjOBJ_GEOM: "geom",
    mjtObj.mjOBJ_SITE: "site", mjtObj.mjOBJ_TENDON: "tendon", mjtObj.mjOBJ_ACTUATOR: "actuator", mjtObj.mjOBJ_KEY: "key",
    mjtObj.mjOBJ_SENSOR: "sensor",
}


class _Opt:
    """``model.opt``: read-only physics options plus the writable ``disableactuator`` bit mask."""

    def __init__(self, model: "MjModel", c: dict):
        object.__setattr__(self, "_model", model)
        object.__setattr__(self, "_disableactuator", 0)
        for k in ("timestep", "gravity", "wind", "density", "viscosity", "tolerance", "ls_tolerance", "impratio",
                  "integrator", "iterations", "ls_iterations"):
            object.__setattr__(self, k, c[k])

    @property
    def disableactuator(self) -> int:
        return self._disableactuator

    @disableactuator.setter
    def disableactuator(self, mask: int) -> None:
        object.__setattr__(self, "_disableactuator", int(mask))
        self._model._apply_disable_mask()

    def __setattr__(self, key, value):
        if key == "disableactuator":
            type(self).disableactuator.fset(self, value)
        else:
            raise ConfigError(f"model.opt.{key} is read-only on the B200 path (recompile the model to change it)")


class _Named:
    def __init__(self, idx: int, name: str | None):
        self.id = idx
        self.name = name if name is not None else ""


class MjModel:
    """Compiled model (``mj.MjModel``'s role; reference ``mujoco_template/model.py:14-43``)."""

    def __init__(self, compiled: dict):
        self._c = compiled
        self.names: dict[str, list[str | None]] = compiled["names"]
        for key in ("nq", "nv", "nu", "nbody", "njnt", "ngeom", "nsite", "ntendon", "nkey", "nsensor", "nsensordata"):
            setattr(self, key, int(compiled[key]))
        self.na = 0
        for key, val in compiled.items():
            if isinstance(val, np.ndarray) and not key.startswith("_") and not hasattr(self, key):
                setattr(self, key, val)
        nu = self.nu
        self.actuator_trnid = np.stack([compiled["actuator_trnid"], np.full(nu, -1, np.int32)], axis=1) if nu else np.zeros((0, 2), np.int32)
        self.actuator_actlimited = np.zeros(nu, dtype=bool)
        self.actuator_actrange = np.zeros((nu, 2))
        self.opt = _Opt(self, compiled)
        self.stat = SimpleNamespace(meaninertia=float(compiled["meaninertia"]))
        self.blob = _layout.pack(compiled)
        self._native: _capi.NativeModel | None = None

    # -- construction (reference model.py:22-31)
    @classmethod
    def from_xml_path(cls, path: str) -> "MjModel":
        return cls(mjcf.compile_xml_path(str(path)))

    @classmethod
    def from_xml_string(cls, text: str) -> "MjModel":
        return cls(mjcf.compile_xml_string(text))

    # -- compiled-model files (the role MJB files play upstream; reference model.py:33-51)
    def save_compiled(self, path: str) -> None:
        import json

        arrays = {k: v for k, v in self._c.items() if isinstance(v, np.ndarray) and not k.startswith("_")}
        scalars = {k: (v if isinstance(v, (int, float, str)) else float(v)) for k, v in self._c.items()
                   if isinstance(v, (int, float, str, np.integer, np.floating))}
        meta = json.dumps(dict(names=self.names, scalars=scalars))
        with open(path, "wb") as fh:
            np.savez_compressed(fh, __meta__=np.frombuffer(meta.encode(), dtype=np.uint8), **arrays)

    @classmethod
    def from_compiled(cls, path: str) -> "MjModel":
        import json

        try:
            with np.load(path, allow_pickle=False) as z:
                meta = json.loads(bytes(z["__meta__"]).decode())
                compiled = {k: z[k] for k in z.files if k != "__meta__"}
        except (OSError, KeyError, ValueError) as exc:
            raise ConfigError(f"cannot load compiled model {path}: {exc}") from exc
        compiled.update(meta["scalars"])
        compiled["names"] = meta["names"]
        if "nsensor" not in compiled:  # files written before sensors were compiled
            compiled.update(nsensor=0, nsensordata=0, sensor_cutoff=np.zeros(0),
                            **{k: np.zeros(0, np.int32) for k in ("sensor_type", "sensor_objtype", "sensor_objid", "sensor_adr", "sensor_dim")})
            compiled["names"].setdefault("sensor", [])
        return cls(compiled)

    @property
    def native(self) -> _capi.NativeModel:
        if self._native is None:
            if os.environ.get("B2_JIT_SPEC") == "1":  # opt-in: compile register-resident kernels for this model first
                from ._specialize import jit_specialize

                jit_specialize(self)
            self._native = _capi.NativeModel(self.blob)
            self._apply_disable_mask()
        return self._native

    def specialize(self, name: str | None = None) -> str | None:
        """Compile and register model-specialised kernels for this model (``_specialize.jit_specialize``).  Call it
        before the first env / batch of the model is created; returns the cached shared object or None (nv > 8)."""
        from ._specialize import jit_specialize

        if self._native is not None:
            raise ConfigError("MjModel.specialize(): call it before the model is first used on the device")
        return jit_specialize(self, name)

    def _apply_disable_mask(self) -> None:
        if self._native is None or self.nu == 0:
            return
        mask = int(self.opt.disableactuator)
        self._native.set_actuator_disabled([(mask >> int(g)) & 1 for g in self.actuator_group])

    # -- named accessors used by reference code (model.body(name).id, model.joint(i).name)
    def _named(self, kind: str, key: Any) -> _Named:
        names = self.names[kind]
        if isinstance(key, str):
            if key not in names:
                raise KeyError(f"Invalid name '{key}' for {kind}")
            return _Named(names.index(key), key)
        idx = int(key)
        if not 0 <= idx < len(names):
            raise IndexError(f"{kind} index {idx} out of range")
        return _Named(idx, names[idx])

    def body(self, key): return self._named("body", key)
    def joint(self, key): return self._named("joint", key)
    def geom(self, key): return self._named("geom", key)
    def site(self, key): return self._named("site", key)
    def actuator(self, key): return self._named("actuator", key)
    def key(self, key): return self._named("key", key)


# ----------------------------------------------------------------------------- buffers
_STATE_FIELDS = ("qpos", "qvel", "ctrl", "qacc_warmstart")


def _field_dims(m: MjModel) -> dict[str, int]:
    return dict(qpos=m.nq, qvel=m.nv, ctrl=m.nu, qacc_warmstart=m.nv, xpos=3 * m.nbody, xquat=4 * m.nbody,
                xipos=3 * m.nbody, geom_xpos=3 * m.ngeom, site_xpos=3 * m.nsite, subtree_com=3 * m.nbody,
                qacc=m.nv, qfrc_bias=m.nv, qfrc_inverse=m.nv, actuator_moment=m.nu * m.nv,
                sensordata=m.nsensordata)


_INT_FIELDS = ("flags", "ncon", "nefc", "solver_iter")


class NativeBackend:
    """Executes the hot path on a B200 through the C-ABI; owns the SoA buffers."""

    def __init__(self, model: MjModel, nenv: int, *, device: int | None = None, precision: int = 64,
                 host_mapped: bool = False):
        import torch

        if not torch.cuda.is_available():
            raise TemplateError("no CUDA device available: the physics path is B200-only and has no CPU fallback")
        self.torch = torch
        self.model = model
        self.nenv = int(nenv)
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.precision = int(precision)
        self.host_mapped = bool(host_mapped)
        self.dtype = torch.float64 if precision == 64 else torch.float32
        self.batch = _capi.NativeBatch(model.native, nenv, self.device, precision)
        self.buffers: dict[str, Any] = {}
        for name, dim in _field_dims(model).items():
            self.buffers[name] = self._alloc(dim, self.dtype)
        for name in _INT_FIELDS:
            self.buffers[name] = self._alloc(1, torch.int32)
        self._scratch: dict[str, Any] = {}
        self.derived_stale = False  # a control tick deferred the derived arrays (see ensure_derived)
        self.stream = 0  # legacy default stream; device batches launch on torch's current stream (see _pre)
        self.profile: dict[str, list] | None = None  # name -> [(start_event, end_event)], filled when enabled

    def _alloc(self, dim: int, dtype):
        torch = self.torch
        shape = (max(dim, 0), self.nenv)
        if self.host_mapped:
            t = torch.zeros(shape, dtype=dtype).pin_memory()
        else:
            t = torch.zeros(shape, dtype=dtype, device=f"cuda:{self.device}")
        return t

    def array(self, name: str):
        """NumPy view (host-mapped) or torch tensor (device) of a buffer."""
        t = self.buffers[name]
        return t.numpy() if self.host_mapped else t

    def _ptr(self, name: str) -> int | None:
        t = self.buffers[name]
        return t.data_ptr() if t.numel() else None

    def state_struct(self) -> _capi.State:
        return _capi.State(self._ptr("qpos"), self._ptr("qvel"), self._ptr("ctrl"), self._ptr("qacc_warmstart"), self._ptr("flags"))

    def derived_struct(self) -> _capi.Derived:
        p = self._ptr
        return _capi.Derived(p("xpos"), p("xquat"), p("xipos"), p("geom_xpos"), p("site_xpos"), p("subtree_com"), p("qacc"),
                             p("qfrc_bias"), p("ncon"), p("nefc"), p("solver_iter"), p("sensordata"))

    def _pre(self) -> None:
        # device tensors may have pending work on torch's current stream (controllers); order after it
        if not self.host_mapped:
            s = self.torch.cuda.current_stream(self.device)
            self.stream = s.cuda_stream

    def _post(self) -> None:
        if self.host_mapped:
            self.batch.synchronize(self.stream)

    def _launch(self, name: str, fn, *args) -> None:
        """Run one C-ABI launch; when profiling, bracket it with CUDA events on the launch stream."""
        self._pre()
        if self.profile is None or self.host_mapped or self.torch.cuda.is_current_stream_capturing():
            fn(*args, self.stream)
        else:
            torch = self.torch
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(torch.cuda.current_stream(self.device))
            fn(*args, self.stream)
            e1.record(torch.cuda.current_stream(self.device))
            self.profile.setdefault(name, []).append((e0, e1))
        self._post()

    def kernel_ms(self, name: str) -> list[float]:
        """Per-launch device times (ms) collected while ``profile`` was enabled."""
        return [a.elapsed_time(b) for a, b in (self.profile or {}).get(name, [])]

    def step_lazy(self) -> None:
        """One step without derived outputs (``b2_step_lazy``); ``ensure_derived()`` produces them if someone reads one."""
        self._launch("step", self.batch.step_lazy, self.state_struct())
        self.derived_stale = True

    def step(self, nsteps: int = 1, derived: bool = True) -> None:
        self.derived_stale = False
        self._launch("step", self.batch.step, self.state_struct(), nsteps, self.derived_struct() if derived else None)

    def rollout(self, ctrl_seq, nsteps: int, record: bool, out=None, derived: bool = True):
        """Open-loop rollout (``b2_rollout``): ``nsteps`` steps, control row t of ``ctrl_seq`` applied at step t.
        ``ctrl_seq``: a tensor laid out as (nsteps, nu, nenv) -- row-contiguous blocks, env fastest -- or None (the
        controls held).  With ``record`` returns (qpos_traj, qvel_traj, sensor_traj), of shapes (nsteps, nq, nenv),
        (nsteps, nv, nenv) and (nsteps, nsensordata, nenv) (None without sensors): the state, and the sensordata mj_step
        leaves, after every step.  Fresh buffers unless ``out`` gives them; an entry of ``out`` may be None (not
        recorded).  The derived arrays are those of the last step (``derived=False``: not written)."""
        torch, m = self.torch, self.model
        T = int(nsteps)
        if out is None and record:
            mk = ((lambda dim: torch.zeros((T, dim, self.nenv), dtype=self.dtype).pin_memory()) if self.host_mapped else
                  (lambda dim: torch.empty((T, dim, self.nenv), device=f"cuda:{self.device}", dtype=self.dtype)))
            out = (mk(m.nq), mk(m.nv), mk(m.nsensordata) if m.nsensordata else None)
        bufs = tuple(out) if out is not None else (None, None, None)
        ptr = lambda t: t.data_ptr() if t is not None and t.numel() else None  # noqa: E731
        self.derived_stale = False
        self._launch("rollout", self.batch.rollout, self.state_struct(), T, ptr(ctrl_seq) if m.nu else None, *map(ptr, bufs),
                     self.derived_struct() if derived else None)
        return bufs if out is not None else None

    def rollout_feedback(self, ctrl_nom, qpos_nom, qvel_nom, K, k, alpha, nsteps: int, record: bool, out=None, derived: bool = True):
        """Closed-loop rollout (``b2_rollout_feedback``): ``nsteps`` steps under the time-varying LQR law
        ``u_t = clip(ctrl_nom[t] + alpha k[t] - K[t] [q (-) qpos_nom[t] ; v - qvel_nom[t]], ctrlrange)``.  Tensors in the
        library's layouts: ``ctrl_nom`` (nsteps, nu, nenv), ``qpos_nom`` / ``qvel_nom`` (>= nsteps, dim, nenv), ``K``
        (nsteps, nu, 2nv, nenv), ``k`` (nsteps, nu, nenv) or None, ``alpha`` (nenv,) or None (1).  With ``record`` returns
        (ctrl_traj, qpos_traj, qvel_traj, sensor_traj) of shapes (nsteps, nu, nenv), (nsteps, nq, nenv), (nsteps, nv, nenv)
        and (nsteps, nsensordata, nenv) (None without sensors); fresh buffers unless ``out`` gives them."""
        torch, m = self.torch, self.model
        T = int(nsteps)
        if out is None and record:
            mk = ((lambda dim: torch.zeros((T, dim, self.nenv), dtype=self.dtype).pin_memory()) if self.host_mapped else
                  (lambda dim: torch.empty((T, dim, self.nenv), device=f"cuda:{self.device}", dtype=self.dtype)))
            out = (mk(m.nu), mk(m.nq), mk(m.nv), mk(m.nsensordata) if m.nsensordata else None)
        bufs = tuple(out) if out is not None else (None, None, None, None)
        ptr = lambda t: t.data_ptr() if t is not None and t.numel() else None  # noqa: E731
        self.derived_stale = False
        self._launch("rollout_feedback", self.batch.rollout_feedback, self.state_struct(), T, ptr(ctrl_nom), ptr(qpos_nom), ptr(qvel_nom),
                     ptr(K), ptr(k), ptr(alpha), *map(ptr, bufs), self.derived_struct() if derived else None)
        return bufs if out is not None else None

    def forward(self) -> None:
        self.derived_stale = False
        self._launch("forward", self.batch.forward, self.state_struct(), self.derived_struct())

    def ensure_derived(self) -> None:
        """Materialise the derived arrays of the last control tick that deferred them (``b2_refresh_derived``)."""
        if self.derived_stale:
            self.derived_stale = False
            self._launch("refresh_derived", self.batch.refresh_derived, self.derived_struct())

    def control_tick(self, eps: float, centered: bool, use_lqr: bool, out=None, derived: bool = True):
        """LQR law (optional) -> (A, B) -> one step (``b2_control_tick``).  ``derived=False`` defers the derived arrays:
        the step then rides in the FD launch, and ``ensure_derived()`` produces them later if someone reads them."""
        torch, m = self.torch, self.model
        nx = 2 * m.nv
        if out is not None:
            A, B = out
        else:
            A = torch.empty((nx, nx, self.nenv), device=f"cuda:{self.device}", dtype=self.dtype)
            B = torch.empty((nx, m.nu, self.nenv), device=f"cuda:{self.device}", dtype=self.dtype)
        defer = not derived and int(m.opt.integrator) == 0  # the library defers only for Euler models
        self._launch("control_tick", self.batch.control_tick, self.state_struct(), None if defer else self.derived_struct(),
                     use_lqr, eps, centered, A.data_ptr(), B.data_ptr() if m.nu else None)
        self.derived_stale = defer
        return A, B

    def linearize(self, eps: float, centered: bool, out=None):
        """Returns (A, B) as SoA buffers of shape (2nv, 2nv, nenv) and (2nv, nu, nenv).

        Fresh buffers by default (the reference returns fresh arrays, linearization.py:24-27);
        pass ``out=(A, B)`` to overwrite existing ones."""
        torch, m = self.torch, self.model
        nx = 2 * m.nv
        kw = dict(dtype=self.dtype)
        if out is not None:
            A, B = out
        elif self.host_mapped:
            A = torch.zeros((nx, nx, self.nenv), **kw).pin_memory()
            B = torch.zeros((nx, m.nu, self.nenv), **kw).pin_memory()
        else:
            A = torch.empty((nx, nx, self.nenv), device=f"cuda:{self.device}", **kw)  # every entry is written
            B = torch.empty((nx, m.nu, self.nenv), device=f"cuda:{self.device}", **kw)
        self._launch("linearize", self.batch.linearize, self.state_struct(), eps, centered, A.data_ptr(),
                     B.data_ptr() if m.nu else None)
        return A, B

    def linearize_sensors(self, eps: float, centered: bool, out=None):
        """(A, B, C, D) from one FD launch (``b2_linearize_sensors``): ``linearize``'s (A, B) plus the sensor Jacobians
        C = d sensordata / dx of shape (nsensordata, 2nv, nenv) and D = d sensordata / du of shape (nsensordata, nu, nenv).
        ``out=(A, B, C, D)`` overwrites existing buffers; an entry that is None gets a fresh one."""
        torch, m = self.torch, self.model
        nx, ns = 2 * m.nv, m.nsensordata
        shapes = ((nx, nx, self.nenv), (nx, m.nu, self.nenv), (ns, nx, self.nenv), (ns, m.nu, self.nenv))
        bufs = list(out) if out is not None else [None] * 4
        for k, shape in enumerate(shapes):
            if bufs[k] is None:
                bufs[k] = (torch.zeros(shape, dtype=self.dtype).pin_memory() if self.host_mapped
                           else torch.empty(shape, device=f"cuda:{self.device}", dtype=self.dtype))  # every entry is written
        self._launch("linearize_sensors", self.batch.linearize_sensors, self.state_struct(), eps, centered,
                     *[t.data_ptr() if t.numel() else None for t in bufs])
        return tuple(bufs)

    def linearize_rollout(self, ctrl_seq, nsteps: int, eps: float, centered: bool, sensors: bool, out=None):
        """(A, B) -- and with ``sensors`` (C, D) -- at every step of the open-loop rollout under ``ctrl_seq``
        (``b2_linearize_rollout``): the loop ``ctrl <- ctrl_seq[t]; linearize_sensors; step(1)`` on a copy of the state,
        which is left as it is (flags apart).  ``ctrl_seq``: a (nsteps, nu, nenv) tensor, or None (the controls held).

        Returns (A, B, C, D, qpos, qvel, warm, sensordata) of shapes (T, 2nv, 2nv, nenv), (T, 2nv, nu, nenv),
        (T, nsensordata, 2nv, nenv), (T, nsensordata, nu, nenv), (T+1, nq, nenv), (T+1, nv, nenv), (T+1, nv, nenv) and
        (T, nsensordata, nenv): the Jacobians of step t and the nominal trajectory they linearise about (row 0 is the
        state, row t+1 the state after step t, warm the warm start each step starts from).  C, D and sensordata are None
        unless ``sensors`` and the model has sensors; warm is None when the state has no warm start.  Fresh buffers unless
        ``out`` gives all eight (fixed addresses under graph capture); an entry of ``out`` may be None (not written)."""
        torch, m = self.torch, self.model
        T, nx, ns = int(nsteps), 2 * m.nv, m.nsensordata
        if out is None:
            mk = ((lambda *shape: torch.zeros(shape, dtype=self.dtype).pin_memory()) if self.host_mapped else
                  (lambda *shape: torch.empty(shape, device=f"cuda:{self.device}", dtype=self.dtype)))
            sens = bool(sensors) and ns > 0
            out = (mk(T, nx, nx, self.nenv), mk(T, nx, m.nu, self.nenv),
                   mk(T, ns, nx, self.nenv) if sens else None, mk(T, ns, m.nu, self.nenv) if sens else None,
                   mk(T + 1, m.nq, self.nenv), mk(T + 1, m.nv, self.nenv),
                   mk(T + 1, m.nv, self.nenv) if self._ptr("qacc_warmstart") else None, mk(T, ns, self.nenv) if sens else None)
        ptr = lambda t: t.data_ptr() if t is not None and t.numel() else None  # noqa: E731
        A, B, C_, D_, q, v, w, s = out
        self._launch("linearize_rollout", self.batch.linearize_rollout, self.state_struct(), T, ptr(ctrl_seq) if m.nu else None,
                     eps, centered, ptr(A), ptr(B), ptr(C_), ptr(D_), ptr(q), ptr(v), ptr(w), ptr(s))
        return tuple(out)

    def jacobian(self, kind: int, objid: int, want_rot: bool):
        torch, m = self.torch, self.model
        mk = (lambda: torch.zeros((3, m.nv, self.nenv), dtype=self.dtype).pin_memory()) if self.host_mapped else (
            lambda: torch.zeros((3, m.nv, self.nenv), dtype=self.dtype, device=f"cuda:{self.device}"))
        jp = mk()
        jr = mk() if want_rot else None
        self._launch("jacobian", self.batch.jacobian, self.state_struct(), kind, objid, jp.data_ptr(),
                     jr.data_ptr() if jr is not None else None)
        return jp, jr

    def inverse(self) -> None:
        """mj_inverse for the acceleration in the ``qacc`` buffer -> ``qfrc_inverse``, ``actuator_moment`` buffers."""
        self._launch("inverse", self.batch.inverse, self.state_struct(), self._ptr("qacc"), self._ptr("qfrc_inverse"),
                     self._ptr("actuator_moment"))

    def _tmp(self, key: str, dim: int):
        t = self._scratch.get(key)
        if t is None:
            t = self._alloc(dim, self.dtype)
            self._scratch[key] = t
        return t

    def integrate_pos_host(self, qpos: np.ndarray, qvel: np.ndarray, dt: float) -> None:
        """In-place mj_integratePos on caller-owned NumPy vectors (single env)."""
        m = self.model
        tq, tv = self._tmp("ip_q", m.nq), self._tmp("ip_v", m.nv)
        tq[:, 0] = self.torch.as_tensor(np.asarray(qpos, dtype=float), dtype=self.dtype)
        tv[:, 0] = self.torch.as_tensor(np.asarray(qvel, dtype=float), dtype=self.dtype)
        self._pre()
        self.batch.integrate_pos(tq.data_ptr(), tv.data_ptr(), dt, self.stream)
        self.batch.synchronize(self.stream)
        qpos[:] = tq[:, 0].cpu().numpy()

    def differentiate_pos_host(self, out: np.ndarray, dt: float, qpos1: np.ndarray, qpos2: np.ndarray) -> None:
        m = self.model
        t1, t2, to = self._tmp("dp_1", m.nq), self._tmp("dp_2", m.nq), self._tmp("dp_o", m.nv)
        t1[:, 0] = self.torch.as_tensor(np.asarray(qpos1, dtype=float), dtype=self.dtype)
        t2[:, 0] = self.torch.as_tensor(np.asarray(qpos2, dtype=float), dtype=self.dtype)
        self._pre()
        self.batch.differentiate_pos(to.data_ptr(), dt, t1.data_ptr(), t2.data_ptr(), self.stream)
        self.batch.synchronize(self.stream)
        out[:] = to[:, 0].cpu().numpy()


# ----------------------------------------------------------------------------- data facades
class _DataBase:
    model: MjModel
    backend: Any
    time: float

    def _reset_from(self, qpos, qvel, ctrl, time: float) -> None:
        b = self.backend
        q, v, u, w = b.array("qpos"), b.array("qvel"), b.array("ctrl"), b.array("qacc_warmstart")
        if isinstance(q, np.ndarray):
            q[:] = np.asarray(qpos, dtype=q.dtype)[:, None]
            v[:] = np.asarray(qvel, dtype=v.dtype)[:, None]
            if self.model.nu:
                u[:] = np.asarray(ctrl, dtype=u.dtype)[:, None]
            w[:] = 0
            b.array("qacc")[:] = 0
            b.array("flags")[:] = 0
        else:
            torch = b.torch
            q.copy_(torch.as_tensor(qpos, dtype=q.dtype, device=q.device)[:, None].expand_as(q))
            v.copy_(torch.as_tensor(qvel, dtype=v.dtype, device=v.device)[:, None].expand_as(v))
            if self.model.nu:
                u.copy_(torch.as_tensor(ctrl, dtype=u.dtype, device=u.device)[:, None].expand_as(u))
            w.zero_()
            b.array("qacc").zero_()
            b.array("flags").zero_()
        self.time = float(time)


class MjData(_DataBase):
    """One env (``mj.MjData``'s role).  Arrays are NumPy views of device-mapped host memory."""

    def __init__(self, model: MjModel, backend: Any = None):
        self.model = model
        self.backend = backend if backend is not None else NativeBackend(model, 1, host_mapped=True)
        b = self.backend
        m = model
        self.qpos = b.array("qpos")[:, 0]
        self.qvel = b.array("qvel")[:, 0]
        self.ctrl = b.array("ctrl")[:, 0]
        self.qacc_warmstart = b.array("qacc_warmstart")[:, 0]
        self.qacc = b.array("qacc")[:, 0]
        self.qfrc_bias = b.array("qfrc_bias")[:, 0]
        self.xpos = b.array("xpos")[:, 0].reshape(m.nbody, 3)
        self.xquat = b.array("xquat")[:, 0].reshape(m.nbody, 4)
        self.xipos = b.array("xipos")[:, 0].reshape(m.nbody, 3)
        self.geom_xpos = b.array("geom_xpos")[:, 0].reshape(m.ngeom, 3)
        self.site_xpos = b.array("site_xpos")[:, 0].reshape(m.nsite, 3)
        self.subtree_com = b.array("subtree_com")[:, 0].reshape(m.nbody, 3)
        self.qfrc_inverse = b.array("qfrc_inverse")[:, 0]
        self.actuator_moment = b.array("actuator_moment")[:, 0].reshape(m.nu, m.nv)  # dense nu x nv
        # MuJoCo >= 3.2 stores the moment matrix row-compressed; callers densify it with mju_sparse2dense (reference
        # setpoints.py:37-47, examples/humanoid/controllers/lqr.py:76-82).  Here every row is stored in full.
        self.moment_rownnz = np.full(m.nu, m.nv, dtype=np.int32)
        self.moment_rowadr = np.arange(m.nu, dtype=np.int32) * m.nv
        self.moment_colind = np.tile(np.arange(m.nv, dtype=np.int32), m.nu)
        self.act = np.zeros(0)
        self.sensordata = b.array("sensordata")[:, 0]
        self.time = 0.0
        # data-less calls (mj_integratePos / mj_differentiatePos) reuse this env's backend scratch
        _HELPERS.setdefault(id(model), self.backend)
        mj_resetData(model, self)

    @property
    def ncon(self) -> int:
        return int(self.backend.array("ncon")[0, 0])

    @property
    def nefc(self) -> int:
        return int(self.backend.array("nefc")[0, 0])

    @property
    def solver_iter(self) -> int:
        return int(self.backend.array("solver_iter")[0, 0])

    @property
    def flags(self) -> int:
        return int(self.backend.array("flags")[0, 0])


class BatchData(_DataBase):
    """N envs: every array is a ``(dim, nenv)`` CUDA tensor the kernels update in place."""

    def __init__(self, model: MjModel, nenv: int, *, device: int | None = None, precision: int = 64, backend: Any = None):
        self.model = model
        self.nenv = int(nenv)
        self.backend = backend if backend is not None else NativeBackend(model, nenv, device=device, precision=precision)
        b = self.backend
        for name in list(_field_dims(model)) + list(_INT_FIELDS):
            if name not in _LAZY_DERIVED:
                setattr(self, name, b.array(name))
        self.time = 0.0
        mj_resetData(model, self)


# Derived arrays of a batch are properties: a control tick may have deferred them (b2_control_tick without derived
# outputs), in which case the first read materialises them -- with the values mj_step leaves in mjData -- in place.
_LAZY_DERIVED = ("xpos", "xquat", "xipos", "geom_xpos", "site_xpos", "subtree_com", "qacc", "qfrc_bias", "sensordata",
                 "ncon", "nefc", "solver_iter")


def _lazy_derived(name: str):
    def get(self):
        self.backend.ensure_derived()
        return self.backend.array(name)
    return property(get)


for _name in _LAZY_DERIVED:
    setattr(BatchData, _name, _lazy_derived(_name))


# ----------------------------------------------------------------------------- mujoco-shaped functions
def mj_name2id(model: MjModel, objtype: int, name: str) -> int:
    kind = _OBJ_KIND.get(int(objtype))
    if kind is None:
        return -1
    try:
        return model.names[kind].index(name)
    except ValueError:
        return -1


def mj_id2name(model: MjModel, objtype: int, idx: int) -> str | None:
    kind = _OBJ_KIND.get(int(objtype))
    if kind is None or not 0 <= idx < len(model.names[kind]):
        return None
    return model.names[kind][idx]


def mj_resetData(model: MjModel, data: _DataBase) -> None:
    data._reset_from(model.qpos0, np.zeros(model.nv), np.zeros(model.nu), 0.0)


def mj_resetDataKeyframe(model: MjModel, data: _DataBase, key: int) -> None:
    if not 0 <= key < model.nkey:
        raise ConfigError(f"Keyframe index out of range: {key}")
    data._reset_from(model.key_qpos[key], model.key_qvel[key], model.key_ctrl[key], float(model.key_time[key]))


def mj_forward(model: MjModel, data: _DataBase) -> None:
    data.backend.forward()


def mj_step(model: MjModel, data: _DataBase, nstep: int = 1) -> None:
    data.backend.step(int(nstep))
    h = float(model.opt.timestep)
    for _ in range(int(nstep)):
        data.time += h  # repeated addition, exactly as upstream accumulates mjData.time


def mj_inverse(model: MjModel, data: _DataBase) -> None:
    """Inverse dynamics for ``data.qacc`` at the current state: fills ``data.qfrc_inverse`` and the dense
    ``data.actuator_moment`` (reference ``mujoco_template/setpoints.py:28-48``)."""
    data.backend.inverse()


def _to_host_matrix(t, nenv: int) -> np.ndarray:
    a = t.numpy() if t.device.type == "cpu" else t.cpu().numpy()
    return a


def mjd_transitionFD(model: MjModel, data: MjData, eps: float, flg_centered: bool, A, B, C_=None, D_=None) -> None:
    """Single-env signature of upstream: fills row-major ``A (2nv,2nv)`` and ``B (2nv,nu)`` in place, and with ``C_`` /
    ``D_`` the sensor Jacobians ``C (nsensordata,2nv)`` and ``D (nsensordata,nu)`` from the same rollouts."""
    if C_ is not None or D_ is not None:
        At, Bt, Ct, Dt = data.backend.linearize_sensors(float(eps), bool(flg_centered))
        if C_ is not None and model.nsensordata:
            C_[...] = _to_host_matrix(Ct, 1)[:, :, 0]
        if D_ is not None and model.nsensordata and model.nu:
            D_[...] = _to_host_matrix(Dt, 1)[:, :, 0]
    else:
        At, Bt = data.backend.linearize(float(eps), bool(flg_centered))
    if A is not None:
        A[...] = _to_host_matrix(At, 1)[:, :, 0]
    if B is not None and model.nu:
        B[...] = _to_host_matrix(Bt, 1)[:, :, 0]


def mj_integratePos(model: MjModel, qpos: np.ndarray, qvel: np.ndarray, dt: float, *, data: _DataBase | None = None) -> None:
    _host_helper(model, data).integrate_pos_host(qpos, qvel, float(dt))


def mj_differentiatePos(model: MjModel, qvel: np.ndarray, dt: float, qpos1: np.ndarray, qpos2: np.ndarray, *,
                        data: _DataBase | None = None) -> None:
    _host_helper(model, data).differentiate_pos_host(qvel, float(dt), qpos1, qpos2)


_HELPERS: dict[int, Any] = {}


def _host_helper(model: MjModel, data: _DataBase | None):
    if data is not None and getattr(data.backend, "nenv", 0) == 1:
        return data.backend
    h = _HELPERS.get(id(model))
    if h is None:
        h = NativeBackend(model, 1, host_mapped=True)
        _HELPERS[id(model)] = h
    return h


def _jac(model: MjModel, data: MjData, kind: int, objid: int, jacp, jacr) -> None:
    jp, jr = data.backend.jacobian(kind, int(objid), jacr is not None)
    if jacp is not None:
        jacp[...] = _to_host_matrix(jp, 1)[:, :, 0]
    if jacr is not None:
        jacr[...] = _to_host_matrix(jr, 1)[:, :, 0]


def mj_jacSite(model, data, jacp, jacr, site): _jac(model, data, _capi.JAC_SITE, site, jacp, jacr)
def mj_jacBody(model, data, jacp, jacr, body): _jac(model, data, _capi.JAC_BODY, body, jacp, jacr)
def mj_jacBodyCom(model, data, jacp, jacr, body): _jac(model, data, _capi.JAC_BODYCOM, body, jacp, jacr)
def mj_jacSubtreeCom(model, data, jacp, body): _jac(model, data, _capi.JAC_SUBTREECOM, body, jacp, None)


def mju_sparse2dense(res: np.ndarray, mat: np.ndarray, rownnz: np.ndarray, rowadr: np.ndarray, colind: np.ndarray) -> None:
    """Expand a row-compressed matrix into the dense ``res`` (nr x nc), as mujoco.mju_sparse2dense does."""
    res[...] = 0.0
    mat = np.asarray(mat).reshape(-1)
    colind = np.asarray(colind).reshape(-1)
    for r in range(res.shape[0]):
        a, n = int(rowadr[r]), int(rownnz[r])
        res[r, colind[a:a + n]] = mat[a:a + n]


def mj_subtreeCoM(model: MjModel, data: _DataBase) -> None:
    """``data.subtree_com`` is already produced by every forward pass; nothing to recompute."""
    return None


__all__ = [
    "MjModel", "MjData", "BatchData", "NativeBackend", "mjtObj", "mjtJoint", "mj_name2id", "mj_id2name", "mj_resetData",
    "mj_resetDataKeyframe", "mj_forward", "mj_step", "mj_inverse", "mjd_transitionFD", "mj_integratePos", "mj_differentiatePos",
    "mj_jacSite", "mj_jacBody", "mj_jacBodyCom", "mj_jacSubtreeCom", "mj_subtreeCoM", "mju_sparse2dense",
]
