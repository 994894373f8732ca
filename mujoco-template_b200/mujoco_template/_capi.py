"""ctypes binding of the C-ABI in ``include/b2mj.h`` (``libb2mj.so``).

This is the only place Python touches native code.  There is no CPU fallback: if the
library is missing, or a compute call is made without a CUDA device, the call raises.
Status codes map 1:1 onto the reference's exception hierarchy
(reference ``mujoco_template/exceptions.py:4-21``).
"""

from __future__ import annotations

import ctypes as C
import os

from .exceptions import ConfigError, LinearizationError, TemplateError, error_for_status  # noqa: F401

B2_F64, B2_F32 = 64, 32
JAC_SITE, JAC_BODY, JAC_BODYCOM, JAC_SUBTREECOM = 0, 1, 2, 3
FLAG_BAD_QPOS, FLAG_BAD_QVEL, FLAG_BAD_QACC, FLAG_OVERFLOW = 1, 2, 4, 8

_LIB_PATH = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "libb2mj.so"))
_lib: C.CDLL | None = None

# every symbol include/b2mj.h declares (tests check the shared object exports all of them)
EXPORTED_SYMBOLS = (
    "b2_model_create", "b2_model_destroy", "b2_model_set_actuator_disabled", "b2_batch_create",
    "b2_batch_destroy", "b2_step", "b2_rollout", "b2_forward", "b2_linearize", "b2_linearize_sensors", "b2_linearize_rollout", "b2_jacobian", "b2_integrate_pos",
    "b2_differentiate_pos", "b2_inverse", "b2_lqr_set_gain", "b2_lqr_control", "b2_control_tick", "b2_refresh_derived", "b2_step_lazy", "b2_step_host", "b2_step_host_wait", "b2_stream_synchronize", "b2_launch_count",
    "b2_batch_size_class", "b2_last_error", "b2_version", "b2_fp_peak", "b2_batch_kernel_variant",
    "b2_recorder_create", "b2_recorder_record", "b2_recorder_destroy", "b2_dlqr", "b2_random_controls", "b2_warp_queue_histogram", "b2_lqr_control_env",
    "b2_tvlqr", "b2_rollout_feedback", "b2_traj_cost",
)


class RecordCol(C.Structure):
    """One column of the batched recorder (include/b2mj.h b2_record_col): kind 0 array row, 1 time, 2 NaN."""
    _fields_ = [("base", C.c_void_p), ("row", C.c_int), ("kind", C.c_int)]


class State(C.Structure):
    _fields_ = [("qpos", C.c_void_p), ("qvel", C.c_void_p), ("ctrl", C.c_void_p),
                ("qacc_warmstart", C.c_void_p), ("flags", C.c_void_p)]


class Derived(C.Structure):
    _fields_ = [("xpos", C.c_void_p), ("xquat", C.c_void_p), ("xipos", C.c_void_p), ("geom_xpos", C.c_void_p),
                ("site_xpos", C.c_void_p), ("subtree_com", C.c_void_p), ("qacc", C.c_void_p),
                ("qfrc_bias", C.c_void_p), ("ncon", C.c_void_p), ("nefc", C.c_void_p), ("solver_iter", C.c_void_p),
                ("sensordata", C.c_void_p)]


def library_path() -> str:
    return _LIB_PATH


def lib() -> C.CDLL:
    """Load libb2mj.so (built in-tree by ``__graft_entry__.build()`` / ``csrc/Makefile``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise TemplateError(
            f"native library not found: {_LIB_PATH}. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C mujoco-template_b200/csrc). There is no CPU fallback for the physics path.")
    L = C.CDLL(_LIB_PATH, mode=C.RTLD_GLOBAL)  # global: run-time specialisations (jit_specialize) link against it
    vp, i, d = C.c_void_p, C.c_int, C.c_double
    L.b2_last_error.restype = C.c_char_p
    L.b2_version.restype = C.c_char_p
    L.b2_launch_count.restype = C.c_longlong
    L.b2_model_create.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(vp)]
    L.b2_model_destroy.argtypes = [vp]
    L.b2_model_destroy.restype = None
    L.b2_model_set_actuator_disabled.argtypes = [vp, C.POINTER(i), i]
    L.b2_batch_create.argtypes = [vp, i, i, i, C.POINTER(vp)]
    L.b2_batch_destroy.argtypes = [vp]
    L.b2_batch_destroy.restype = None
    L.b2_batch_size_class.argtypes = [vp]
    L.b2_batch_kernel_variant.argtypes = [vp]
    L.b2_batch_kernel_variant.restype = C.c_char_p
    L.b2_step.argtypes = [vp, C.POINTER(State), i, C.POINTER(Derived), vp]
    L.b2_rollout.argtypes = [vp, C.POINTER(State), i, vp, vp, vp, vp, C.POINTER(Derived), vp]
    L.b2_forward.argtypes = [vp, C.POINTER(State), C.POINTER(Derived), vp]
    L.b2_linearize.argtypes = [vp, C.POINTER(State), d, i, vp, vp, vp]
    L.b2_linearize_sensors.argtypes = [vp, C.POINTER(State), d, i, vp, vp, vp, vp, vp]
    L.b2_linearize_rollout.argtypes = [vp, C.POINTER(State), i, vp, d, i, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.b2_jacobian.argtypes = [vp, C.POINTER(State), i, i, vp, vp, vp]
    L.b2_inverse.argtypes = [vp, C.POINTER(State), vp, vp, vp, vp]
    L.b2_lqr_set_gain.argtypes = [vp, C.POINTER(d), C.POINTER(d), C.POINTER(d)]
    L.b2_lqr_control.argtypes = [vp, C.POINTER(State), vp]
    L.b2_control_tick.argtypes = [vp, C.POINTER(State), C.POINTER(Derived), i, C.c_double, i, vp, vp, vp]
    L.b2_refresh_derived.argtypes = [vp, C.POINTER(Derived), vp]
    L.b2_step_lazy.argtypes = [vp, C.POINTER(State), vp]
    L.b2_integrate_pos.argtypes = [vp, vp, vp, d, vp]
    L.b2_differentiate_pos.argtypes = [vp, vp, d, vp, vp, vp]
    L.b2_step_host.argtypes = [vp, C.POINTER(State), i, i, d, vp, vp, vp]
    L.b2_step_host_wait.argtypes = [vp]
    L.b2_stream_synchronize.argtypes = [vp, vp]
    L.b2_lqr_control_env.argtypes = [vp, C.POINTER(State), vp, vp]
    L.b2_random_controls.argtypes = [vp, C.POINTER(State), C.c_double, C.c_double, C.c_ulonglong, C.c_int, C.c_double, vp, vp, vp]
    L.b2_warp_queue_histogram.argtypes = [vp, C.POINTER(C.c_int), vp]
    L.b2_dlqr.argtypes = [C.c_int, C.c_int, vp, vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int, C.c_int, C.c_int, C.c_int,
                          C.c_double, vp, vp, vp, vp]
    L.b2_tvlqr.argtypes = [i, i, i, i, i, i, vp, vp, C.POINTER(d), C.POINTER(d), C.POINTER(d), vp, vp, d, vp, vp, vp, vp, vp, vp]
    L.b2_rollout_feedback.argtypes = [vp, C.POINTER(State), i, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.POINTER(Derived), vp]
    L.b2_traj_cost.argtypes = [vp, i, vp, vp, vp, vp, vp, vp, C.POINTER(d), C.POINTER(d), C.POINTER(d), vp, vp, vp, vp]
    L.b2_recorder_create.argtypes = [vp, C.POINTER(RecordCol), C.c_int, C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]
    L.b2_recorder_record.argtypes = [vp, C.c_double, vp, vp]
    L.b2_recorder_destroy.argtypes = [vp]
    L.b2_recorder_destroy.restype = None
    L.b2_fp_peak.argtypes = [i, i, C.POINTER(d)]
    _lib = L
    return L


def check(rc: int) -> None:
    """Translate a C status code into the reference's exception types."""
    if rc == 0:
        return
    raise error_for_status(rc, lib().b2_last_error().decode("utf-8", "replace"))


def fp_peak(precision: int = B2_F64, device: int = 0) -> float:
    """Measured CUDA-core FMA peak in TFLOP/s (roofline denominator for the FP-bound kernels)."""
    out = C.c_double()
    check(lib().b2_fp_peak(int(precision), int(device), C.byref(out)))
    return float(out.value)


def launch_count() -> int:
    return int(lib().b2_launch_count())


class NativeModel:
    """Owns a ``b2_model*``."""

    def __init__(self, blob: bytes):
        self._L = lib()
        h = C.c_void_p()
        check(self._L.b2_model_create(blob, len(blob), C.byref(h)))
        self.handle = h

    def set_actuator_disabled(self, disabled) -> None:
        arr = (C.c_int * len(disabled))(*[int(bool(x)) for x in disabled])
        check(self._L.b2_model_set_actuator_disabled(self.handle, arr, len(disabled)))

    def __del__(self):
        h = getattr(self, "handle", None)
        if h:
            self._L.b2_model_destroy(h)
            self.handle = None


class NativeBatch:
    """Owns a ``b2_batch*`` (nenv envs of one model on one device)."""

    def __init__(self, model: NativeModel, nenv: int, device: int = 0, precision: int = B2_F64):
        self._L = lib()
        self.model = model
        h = C.c_void_p()
        check(self._L.b2_batch_create(model.handle, int(nenv), int(device), int(precision), C.byref(h)))
        self.handle = h
        self.nenv = int(nenv)

    @property
    def size_class(self) -> int:
        return int(self._L.b2_batch_size_class(self.handle))

    @property
    def kernel_variant(self) -> str:
        return self._L.b2_batch_kernel_variant(self.handle).decode()

    def step(self, state: State, nsteps: int, derived: Derived | None, stream: int = 0) -> None:
        check(self._L.b2_step(self.handle, C.byref(state), int(nsteps), C.byref(derived) if derived is not None else None, stream))

    def rollout(self, state: State, nsteps: int, ctrl_seq: int | None, qpos_traj: int | None, qvel_traj: int | None,
                sensor_traj: int | None, derived: Derived | None, stream: int = 0) -> None:
        """``b2_rollout``: ``nsteps`` steps with control row t of ``ctrl_seq`` (nsteps, nu, nenv) applied at step t (None: held
        controls), recording the state (and sensordata) after every step into the (nsteps, dim, nenv) trajectory arrays."""
        check(self._L.b2_rollout(self.handle, C.byref(state), int(nsteps), ctrl_seq, qpos_traj, qvel_traj, sensor_traj,
                                 C.byref(derived) if derived is not None else None, stream))

    def rollout_feedback(self, state: State, nsteps: int, ctrl_nom: int, qpos_nom: int, qvel_nom: int, K: int, k: int | None,
                         alpha: int | None, ctrl_traj: int | None, qpos_traj: int | None, qvel_traj: int | None, sensor_traj: int | None,
                         derived: Derived | None, stream: int = 0) -> None:
        """``b2_rollout_feedback``: ``nsteps`` steps under ``u = clip(ctrl_nom[t] + alpha k[t] - K[t] [q (-) qpos_nom[t] ;
        v - qvel_nom[t]])``, recording the applied controls and the state (and sensordata) after every step."""
        check(self._L.b2_rollout_feedback(self.handle, C.byref(state), int(nsteps), ctrl_nom, qpos_nom, qvel_nom, K, k, alpha, ctrl_traj,
                                          qpos_traj, qvel_traj, sensor_traj, C.byref(derived) if derived is not None else None, stream))

    def traj_cost(self, nsteps: int, qpos: int, qvel: int, ctrl: int, qpos_ref: int, qvel_ref: int | None, ctrl_ref: int | None, Q, R, Qf,
                  J: int | None, q: int | None, r: int | None, stream: int = 0) -> None:
        """``b2_traj_cost``: the tracking cost ``J`` of every env's trajectory and its tangent-space gradients ``q`` / ``r``
        (device pointers in the env-fastest layout; Q, R, Qf host arrays)."""
        import numpy as np

        # flattened row-major float64 arrays, handed over without a per-element conversion (the humanoid's Q has 2,916)
        W = [np.ascontiguousarray(M, dtype=np.float64).reshape(-1) for M in (Q, R, Qf)]
        check(self._L.b2_traj_cost(self.handle, int(nsteps), qpos, qvel, ctrl, qpos_ref, qvel_ref, ctrl_ref,
                                   *[M.ctypes.data_as(C.POINTER(C.c_double)) for M in W], J, q, r, stream))

    def forward(self, state: State, derived: Derived | None, stream: int = 0) -> None:
        check(self._L.b2_forward(self.handle, C.byref(state), C.byref(derived) if derived is not None else None, stream))

    def linearize(self, state: State, eps: float, centered: bool, A: int, B: int, stream: int = 0) -> None:
        check(self._L.b2_linearize(self.handle, C.byref(state), float(eps), int(bool(centered)), A, B, stream))

    def linearize_sensors(self, state: State, eps: float, centered: bool, A: int | None, B: int | None, C_: int | None,
                          D_: int | None, stream: int = 0) -> None:
        """``b2_linearize_sensors``: (A, B) and the sensor Jacobians C = d sensordata / dx, D = d sensordata / du."""
        check(self._L.b2_linearize_sensors(self.handle, C.byref(state), float(eps), int(bool(centered)), A, B, C_, D_, stream))

    def linearize_rollout(self, state: State, nsteps: int, ctrl_seq: int | None, eps: float, centered: bool, A: int | None,
                          B: int | None, C_: int | None, D_: int | None, qpos_traj: int, qvel_traj: int, warm_traj: int | None,
                          sensor_traj: int | None, stream: int = 0) -> None:
        """``b2_linearize_rollout``: (A, B, C, D) at every step of the open-loop rollout under ``ctrl_seq`` (nsteps, nu, nenv)
        (None: held controls), about the nominal trajectory it records into the (nsteps+1, dim, nenv) arrays."""
        check(self._L.b2_linearize_rollout(self.handle, C.byref(state), int(nsteps), ctrl_seq, float(eps), int(bool(centered)), A, B,
                                           C_, D_, qpos_traj, qvel_traj, warm_traj, sensor_traj, stream))

    def jacobian(self, state: State, kind: int, objid: int, jacp: int, jacr: int | None, stream: int = 0) -> None:
        check(self._L.b2_jacobian(self.handle, C.byref(state), int(kind), int(objid), jacp, jacr, stream))

    def inverse(self, state: State, qacc: int | None, qfrc: int, moment: int | None, stream: int = 0) -> None:
        check(self._L.b2_inverse(self.handle, C.byref(state), qacc, qfrc, moment, stream))

    def lqr_set_gain(self, K, qpos_ref, ctrl_ref) -> None:
        import numpy as np

        K = np.ascontiguousarray(K, dtype=np.float64); q = np.ascontiguousarray(qpos_ref, dtype=np.float64)
        u = np.ascontiguousarray(ctrl_ref, dtype=np.float64)
        dp = C.POINTER(C.c_double)
        check(self._L.b2_lqr_set_gain(self.handle, K.ctypes.data_as(dp), q.ctypes.data_as(dp), u.ctypes.data_as(dp)))

    def lqr_control(self, state: State, stream: int = 0) -> None:
        check(self._L.b2_lqr_control(self.handle, C.byref(state), stream))

    def lqr_control_env(self, state: State, K_env: int, stream: int = 0) -> None:
        check(self._L.b2_lqr_control_env(self.handle, C.byref(state), K_env, stream))

    def control_tick(self, state: State, derived: Derived | None, use_lqr: bool, eps: float, centered: bool, A: int, B: int,
                     stream: int = 0) -> None:
        check(self._L.b2_control_tick(self.handle, C.byref(state), C.byref(derived) if derived is not None else None,
                                      int(bool(use_lqr)), float(eps), int(bool(centered)), A, B, stream))

    def step_lazy(self, state: State, stream: int = 0) -> None:
        check(self._L.b2_step_lazy(self.handle, C.byref(state), stream))

    def refresh_derived(self, derived: Derived, stream: int = 0) -> None:
        check(self._L.b2_refresh_derived(self.handle, C.byref(derived), stream))

    def integrate_pos(self, qpos: int, qvel: int, dt: float, stream: int = 0) -> None:
        check(self._L.b2_integrate_pos(self.handle, qpos, qvel, float(dt), stream))

    def differentiate_pos(self, out: int, dt: float, qpos1: int, qpos2: int, stream: int = 0) -> None:
        check(self._L.b2_differentiate_pos(self.handle, out, float(dt), qpos1, qpos2, stream))

    def step_host(self, state: State, nsteps: int, linearize: bool, eps: float, A: int | None, B: int | None, stream: int = 0,
                  device_lqr: bool = False, wait: bool = True) -> None:
        """Host-buffer step; ``device_lqr`` evaluates the ``lqr_set_gain`` law on the device (``state.ctrl`` becomes an output).
        ``wait=False`` queues the step and returns (B2_HOST_ASYNC); ``step_host_wait`` completes it."""
        flags = (1 if linearize else 0) | (2 if device_lqr else 0) | (0 if wait else 4)
        check(self._L.b2_step_host(self.handle, C.byref(state), int(nsteps), flags, float(eps), A, B, stream))

    def step_host_wait(self) -> None:
        """Completes a ``step_host(..., wait=False)``: the host buffers hold the step's results when this returns."""
        check(self._L.b2_step_host_wait(self.handle))

    def random_controls(self, state: State, lo: float, hi: float, seed: int, watch_row: int = -1, watch_min: float = 0.0,
                        reset_qpos: int | None = None, reset_qvel: int | None = None, stream: int = 0) -> None:
        check(self._L.b2_random_controls(self.handle, C.byref(state), float(lo), float(hi), int(seed), int(watch_row), float(watch_min),
                                         reset_qpos, reset_qvel, stream))

    def warp_queue_histogram(self, stream: int = 0) -> list[int]:
        out = (C.c_int * 16)()
        check(self._L.b2_warp_queue_histogram(self.handle, out, stream))
        return list(out)

    def synchronize(self, stream: int = 0) -> None:
        check(self._L.b2_stream_synchronize(self.handle, stream))

    def __del__(self):
        h = getattr(self, "handle", None)
        if h:
            self._L.b2_batch_destroy(h)
            self.handle = None


def dlqr(device: int, precision: int, A_ptr: int, B_ptr: int, Q, R, nx: int, nu: int, nenv: int, K_ptr: int, P_ptr: int,
         status_ptr: int | None, max_doublings: int = 40, tol: float = 1e-13, stream: int = 0) -> None:
    """``b2_dlqr``: batched DARE + gain on the device (A, B, K, P device pointers in the SoA layout; Q, R host arrays)."""
    q = (C.c_double * (nx * nx))(*[float(x) for x in Q])
    r = (C.c_double * (nu * nu))(*[float(x) for x in R])
    check(lib().b2_dlqr(int(device), int(precision), A_ptr, B_ptr, q, r, int(nx), int(nu), int(nenv), int(max_doublings), float(tol),
                        K_ptr, P_ptr, status_ptr, stream))


def tvlqr(device: int, precision: int, nsteps: int, nx: int, nu: int, nenv: int, A_ptr: int, B_ptr: int, Q, R, Qf, q_ptr: int | None,
          r_ptr: int | None, reg: float, K_ptr: int, k_ptr: int | None, P0_ptr: int | None, dV_ptr: int | None, status_ptr: int | None,
          stream: int = 0) -> None:
    """``b2_tvlqr``: batched finite-horizon Riccati backward pass on the device (device pointers in the env-fastest layout;
    Q, R, Qf host arrays)."""
    arr = lambda x, n: (C.c_double * n)(*[float(v) for v in x])  # noqa: E731
    check(lib().b2_tvlqr(int(device), int(precision), int(nsteps), int(nx), int(nu), int(nenv), A_ptr, B_ptr, arr(Q, nx * nx), arr(R, nu * nu),
                         arr(Qf, nx * nx), q_ptr, r_ptr, float(reg), K_ptr, k_ptr, P0_ptr, dV_ptr, status_ptr, stream))


class NativeRecorder:
    """Owns a ``b2_recorder*``: column table + env selection on the device, one gather launch per recorded step."""

    def __init__(self, batch: "NativeBatch", cols: list[tuple[int | None, int, int]], env_index: list[int]):
        self._L = lib()
        self.batch = batch  # keeps the batch alive
        table = (RecordCol * len(cols))(*[RecordCol(base, int(row), int(kind)) for base, row, kind in cols])
        idx = (C.c_int * len(env_index))(*[int(i) for i in env_index])
        h = C.c_void_p()
        check(self._L.b2_recorder_create(batch.handle, table, len(cols), idx, len(env_index), C.byref(h)))
        self.handle = h

    def record(self, time: float, out_ptr: int, stream: int = 0) -> None:
        check(self._L.b2_recorder_record(self.handle, float(time), out_ptr, stream))

    def __del__(self):
        h = getattr(self, "handle", None)
        if h:
            self._L.b2_recorder_destroy(h)
            self.handle = None
