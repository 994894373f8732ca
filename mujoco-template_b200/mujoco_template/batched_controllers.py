"""Vectorised controllers for ``BatchedEnv`` written against the reference ``Controller`` protocol.

``BatchedLQRController`` is the controller BASELINE config #2 needs and the reference does not
ship for the cartpole (its cartpole uses PID, reference ``examples/cartpole/controllers/pid.py``):
a discrete LQR about a fixed setpoint whose gain comes from the FD linearisation at that
setpoint -- the same recipe as the reference's drone / humanoid LQRs
(``examples/drone/controllers/lqr.py:120-133``: ``linearize_discrete`` once in ``prepare`` then a
DARE) -- and which declares ``needs_linearization=True`` so that every control tick also
produces the time-varying ``(A, B)`` of all envs in ``StepResult.info``.
"""

from __future__ import annotations

from typing import Any

import numpy as np

from .control import ControlSpace, ControllerCapabilities
from .exceptions import ConfigError


def dlqr_gain(A: np.ndarray, B: np.ndarray, Q: np.ndarray, R: np.ndarray, device: int | None = None) -> np.ndarray:
    """Infinite-horizon discrete LQR gain K (u = -K x) of ONE system: the library's DARE kernel (``b2_dlqr``) on a
    one-env batch.  The reference recipe is ``scipy.linalg.solve_discrete_are`` + a solve (reference
    ``examples/drone/controllers/lqr.py:350-378``); the two agree to ~1e-9 relative (tests/test_gpu_parity.py)."""
    import torch

    dev = torch.device("cuda", torch.cuda.current_device() if device is None else int(device)) if torch.cuda.is_available() else None
    if dev is None:
        from .exceptions import TemplateError

        raise TemplateError("dlqr_gain: no CUDA device (this path has no CPU fallback)")
    K, _ = batched_dlqr_gain(torch.as_tensor(np.asarray(A, dtype=float), device=dev)[None],
                             torch.as_tensor(np.asarray(B, dtype=float), device=dev)[None], Q, R)
    return K[0].cpu().numpy()


def batched_dlqr_gain(A, B, Q, R, max_doublings: int = 40, tol: float = 1e-13, return_status: bool = False):
    """Infinite-horizon discrete LQR gains of a whole batch on the device (SURVEY.md section 8f, row 2): ``b2_dlqr``, one
    warp per env, every env from its own ``(A, B)``.

    ``A`` (N, nx, nx) and ``B`` (N, nx, nu) are CUDA tensors -- ``StepResult.info['A'/'B']`` of a ``BatchedEnv`` have
    exactly this shape, as permuted views of the ``(nx, nx, N)`` arrays ``b2_linearize`` writes, which the kernel reads
    in place -- ``Q`` (nx, nx) and ``R`` (nu, nu) are shared.  Returns ``(K, P)`` with ``u = -K x``, ``K`` (N, nu, nx),
    ``P`` (N, nx, nx) the stabilising DARE solutions (views of env-fastest storage).  The DARE is solved by the
    structure-preserving doubling iteration (k doublings = a Riccati recursion over 2**k steps, quadratic convergence):

        W = I + G H;  A <- A W^-1 A;  G <- G + A W^-1 G A';  H <- H + A' H W^-1 A      (G0 = B R^-1 B', H0 = Q)

    The single-system reference recipe is ``scipy.linalg.solve_discrete_are`` (reference
    ``examples/drone/controllers/lqr.py:350-378``, ``examples/humanoid/controllers/lqr.py:114-115``)."""
    import torch

    from . import _capi
    from .exceptions import TemplateError

    A = torch.as_tensor(A)
    B = torch.as_tensor(B, dtype=A.dtype, device=A.device)
    if A.dim() == 2:
        A, B = A[None], B[None]
    if A.device.type != "cuda":
        raise TemplateError("batched_dlqr_gain: A and B must be CUDA tensors (this path has no CPU fallback)")
    if A.dtype not in (torch.float64, torch.float32):
        raise ConfigError("batched_dlqr_gain: float64 or float32 tensors expected")
    n, nx, nu = A.shape[0], A.shape[1], B.shape[2]
    if A.shape != (n, nx, nx) or B.shape != (n, nx, nu) or nu > nx:
        raise ConfigError("batched_dlqr_gain: A must be (N, nx, nx) and B (N, nx, nu) with nu <= nx")
    Q = np.ascontiguousarray(np.asarray(Q.cpu() if hasattr(Q, "cpu") else Q, dtype=float)).reshape(nx * nx)
    R = np.ascontiguousarray(np.asarray(R.cpu() if hasattr(R, "cpu") else R, dtype=float)).reshape(nu * nu)
    # env-fastest storage: a permuted view of the (nx, nx, N) array costs nothing, anything else is copied once
    As, Bs = A.permute(1, 2, 0), B.permute(1, 2, 0)
    As = As if As.is_contiguous() else As.contiguous()
    Bs = Bs if Bs.is_contiguous() else Bs.contiguous()
    Ks = torch.empty((nu, nx, n), dtype=A.dtype, device=A.device)
    Ps = torch.empty((nx, nx, n), dtype=A.dtype, device=A.device)
    status = torch.zeros(n, dtype=torch.int32, device=A.device)
    with torch.cuda.device(A.device):
        _capi.dlqr(A.device.index, 64 if A.dtype == torch.float64 else 32, As.data_ptr(), Bs.data_ptr(), Q, R, nx, nu, n,
                   Ks.data_ptr(), Ps.data_ptr(), status.data_ptr(), max_doublings, tol, torch.cuda.current_stream(A.device).cuda_stream)
    K, P = Ks.permute(2, 0, 1), Ps.permute(2, 0, 1)
    return (K, P, status) if return_status else (K, P)


def batched_tvlqr(A, B, Q, R, Qf=None, q=None, r=None, reg: float = 0.0):
    """Finite-horizon time-varying LQR about a trajectory for a whole batch on the device (``b2_tvlqr``): the Riccati
    backward pass of TV-LQR and iLQR, every env from its own ``(A_t, B_t)``.

    ``A`` (N, T, nx, nx) and ``B`` (N, T, nx, nu) are CUDA tensors -- ``BatchedEnv.linearize_rollout``'s ``"A"`` / ``"B"``
    are read in place; ``Q``, ``R`` and ``Qf`` (default ``Q``) are shared host matrices; ``q`` (N, T+1, nx) and ``r``
    (N, T, nu) optional linear cost terms; ``reg`` >= 0 is added to the diagonal of Quu before its Cholesky factorisation.
    With ``dx = [q (-) qbar ; v - vbar]`` and ``du = u - ubar`` the cost is

        J = sum_t [1/2 dx'Q dx + q_t'dx + 1/2 du'R du + r_t'du] + 1/2 dx_T'Qf dx_T + q_T'dx_T

    Returns ``(K, k, P0, dV, status)``: ``K`` (N, T, nu, nx) and ``k`` (N, T, nu) with ``u_t = ubar_t + alpha k_t - K_t
    dx_t`` (``BatchedEnv.rollout_feedback``), ``P0`` (N, nx, nx) the cost-to-go Hessian at t = 0, ``dV`` (N, 2) the
    expected cost change ``alpha dV[:, 0] + alpha**2 dV[:, 1]`` and ``status`` (N,) int32: 0, or -(t+1) when
    ``Quu_t + reg I`` is not positive definite (that env's rows <= t, ``P0`` and ``dV`` are NaN).  All are views of
    env-fastest storage.  See ``include/b2mj.h`` for the recursion."""
    import torch

    from . import _capi
    from .exceptions import TemplateError

    if not isinstance(A, torch.Tensor) or not isinstance(B, torch.Tensor):
        raise ConfigError("batched_tvlqr: A and B must be tensors")
    if A.device.type != "cuda":
        raise TemplateError("batched_tvlqr: A and B must be CUDA tensors (this path has no CPU fallback)")
    if A.dtype not in (torch.float64, torch.float32):
        raise ConfigError("batched_tvlqr: float64 or float32 tensors expected")
    if A.dim() != 4 or B.dim() != 4:
        raise ConfigError("batched_tvlqr: A must be (N, T, nx, nx) and B (N, T, nx, nu)")
    n, T, nx, nu = A.shape[0], A.shape[1], A.shape[2], B.shape[3]
    if A.shape != (n, T, nx, nx) or B.shape != (n, T, nx, nu) or min(n, T, nx, nu) < 1:
        raise ConfigError(f"batched_tvlqr: A must be (N, T, nx, nx) and B (N, T, nx, nu), got {tuple(A.shape)} and {tuple(B.shape)}")

    def env_fastest(name, t, shape):
        if not isinstance(t, torch.Tensor) or tuple(t.shape) != shape:
            raise ConfigError(f"batched_tvlqr: {name} must be a tensor of shape {shape}")
        if t.device != A.device or t.dtype != A.dtype:
            raise ConfigError(f"batched_tvlqr: {name}: expected {A.dtype} on {A.device}, got {t.dtype} on {t.device}")
        return t.permute(*range(1, t.dim()), 0).contiguous()  # no copy for a view of env-fastest storage

    def host(name, M, k):
        M = np.asarray(M.cpu() if hasattr(M, "cpu") else M, dtype=float)
        if M.shape != (k, k):
            raise ConfigError(f"batched_tvlqr: {name} must be ({k}, {k}), got {M.shape}")
        return np.ascontiguousarray(M).reshape(-1)

    As, Bs = env_fastest("A", A, (n, T, nx, nx)), env_fastest("B", B, (n, T, nx, nu))
    qs = None if q is None else env_fastest("q", q, (n, T + 1, nx))
    rs = None if r is None else env_fastest("r", r, (n, T, nu))
    Qh, Rh = host("Q", Q, nx), host("R", R, nu)
    Qfh = Qh if Qf is None else host("Qf", Qf, nx)
    if not float(reg) >= 0:
        raise ConfigError("batched_tvlqr: reg must be >= 0")
    mk = lambda *shape: torch.empty(shape, dtype=A.dtype, device=A.device)  # noqa: E731
    Ks, ks, Ps, dVs = mk(T, nu, nx, n), mk(T, nu, n), mk(nx, nx, n), mk(2, n)
    status = torch.zeros(n, dtype=torch.int32, device=A.device)
    ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
    with torch.cuda.device(A.device):
        _capi.tvlqr(A.device.index, 64 if A.dtype == torch.float64 else 32, T, nx, nu, n, As.data_ptr(), Bs.data_ptr(), Qh, Rh, Qfh,
                    ptr(qs), ptr(rs), float(reg), Ks.data_ptr(), ks.data_ptr(), Ps.data_ptr(), dVs.data_ptr(), status.data_ptr(),
                    torch.cuda.current_stream(A.device).cuda_stream)
    return Ks.permute(3, 0, 1, 2), ks.permute(2, 0, 1), Ps.permute(2, 0, 1), dVs.permute(1, 0), status


def batched_ilqr(env, controls, Q, R, Qf=None, *, qpos_ref, qvel_ref=None, ctrl_ref=None, iters: int = 20,
                 alphas=tuple(0.5 ** i for i in range(10)), reg: float = 1e-6, eps: float | None = None):
    """iLQR for every env of a ``BatchedEnv`` from its current state, on the device: minimises ``BatchedEnv.traj_cost``
    over the control sequence.  Each iteration runs

        1. ``linearize_rollout(ubar)``: the nominal trajectory and its ``(A_t, B_t)``;
        2. ``traj_cost(grad=True)``: its cost ``J`` and the gradients ``q_t`` / ``r_t``;
        3. ``batched_tvlqr(A, B, Q, R, Qf, q, r, reg)``: the gains ``K_t``, ``k_t``;
        4. a backtracking line search over ``alphas``: per trial one ``rollout_feedback`` with the step size of each env and
           one ``traj_cost``.  An env accepts the first step size whose cost is finite and below its current ``J`` and then
           keeps that result; an env whose backward pass failed (``status != 0``) rejects every trial.  The trials stop once
           every env with a valid backward pass has accepted.

    ``controls`` ``(nenv, T, nu)`` is the initial control sequence; ``Q``, ``R``, ``Qf`` and the references are those of
    ``traj_cost``; ``eps`` is the FD step of ``linearize_rollout`` (None: the env's ``lin_eps``).  The iterations stop early
    when one leaves every env where it was (the next would repeat it).  The env's state, warm start, controls, flags,
    ``data.time`` and step counter are left as they were.

    Returns a dict: ``"ctrl"`` ``(nenv, T, nu)``, ``"qpos"`` ``(nenv, T+1, nq)`` and ``"qvel"`` ``(nenv, T+1, nv)`` (the
    final nominal trajectory, row 0 the current state), ``"J"`` ``(nenv,)``, ``"J_history"`` ``(iterations + 1, nenv)``
    (the cost before the first iteration and after each) and ``"status"`` ``(nenv,)``, the last backward pass's status."""
    import torch

    data, b, m, n = env.data, env.data.backend, env.model, env.nenv
    if not isinstance(controls, torch.Tensor) or controls.dim() != 3 or tuple(controls.shape[::2]) != (n, m.nu) or controls.shape[1] < 1:
        raise ConfigError(f"batched_ilqr: controls must be a (nenv={n}, T, nu={m.nu}) tensor")
    alphas = [float(a) for a in alphas]
    if not alphas or not all(a > 0 for a in alphas) or int(iters) < 1:
        raise ConfigError("batched_ilqr: iters must be >= 1 and alphas a non-empty sequence of positive step sizes")
    T = int(controls.shape[1])
    cost = dict(qpos_ref=qpos_ref, qvel_ref=qvel_ref, ctrl_ref=ctrl_ref)
    saved = {k: b.buffers[k].clone() for k in ("qpos", "qvel", "ctrl", "qacc_warmstart", "flags") if b.buffers[k].numel()}
    stale = b.derived_stale
    x0 = saved["qpos"], saved["qvel"]
    # trial trajectories: rollout_feedback records rows 1..T of (T+1)-row buffers whose row 0 is x0
    mk = lambda *shape: torch.empty(shape, dtype=data.qpos.dtype, device=data.qpos.device)  # noqa: E731
    tq, tv, tu = mk(T + 1, m.nq, n), mk(T + 1, m.nv, n), mk(T, m.nu, n)
    tq[0], tv[0] = x0
    trial = tq.permute(2, 0, 1), tv.permute(2, 0, 1), tu.permute(2, 0, 1)

    def restore(keys):
        for k in keys:
            if k in saved:
                b.buffers[k].copy_(saved[k])

    try:
        ubar = controls.detach().clone()
        lin = env.linearize_rollout(ubar, eps=eps)
        J, q, r = env.traj_cost(lin["qpos"], lin["qvel"], ubar, Q, R, Qf, grad=True, **cost)
        xq, xv = lin["qpos"].clone(), lin["qvel"].clone()
        history = [J.clone()]
        status = torch.zeros(n, dtype=torch.int32, device=J.device)
        for it in range(int(iters)):
            K, k, _, _, status = batched_tvlqr(lin["A"], lin["B"], Q, R, Qf, q, r, reg)
            Ks, ks = K.permute(1, 2, 3, 0), k.permute(1, 2, 0)
            seq, qn, vn = ubar.permute(1, 2, 0).contiguous(), lin["qpos"].permute(1, 2, 0), lin["qvel"].permute(1, 2, 0)
            accepted = torch.zeros(n, dtype=torch.bool, device=J.device)
            done = status != 0  # NaN gains: never accepted, whatever the clip makes of them
            for a in alphas:
                restore(("qpos", "qvel", "qacc_warmstart", "flags"))
                alpha = torch.full((n,), a, dtype=J.dtype, device=J.device)
                b.rollout_feedback(seq, qn, vn, Ks, ks, alpha, T, False, out=(tu, tq[1:], tv[1:], None), derived=False)
                Jn = env.traj_cost(*trial, Q, R, Qf, **cost)
                take = ~done & torch.isfinite(Jn) & (Jn < J)
                J = torch.where(take, Jn, J)
                ubar = torch.where(take[:, None, None], trial[2], ubar)
                xq, xv = torch.where(take[:, None, None], trial[0], xq), torch.where(take[:, None, None], trial[1], xv)
                accepted |= take
                done |= take
                if bool(done.all()):
                    break
            history.append(J.clone())
            if not bool(accepted.any()) or it == int(iters) - 1:
                break
            restore(("qpos", "qvel", "qacc_warmstart", "flags"))
            lin = env.linearize_rollout(ubar, eps=eps)
            _, q, r = env.traj_cost(lin["qpos"], lin["qvel"], ubar, Q, R, Qf, grad=True, **cost)
    finally:
        restore(saved)
        b.derived_stale = stale
    return {"ctrl": ubar, "qpos": xq, "qvel": xv, "J": J, "J_history": torch.stack(history), "status": status}


class BatchedLQRController:
    def __init__(self, qpos_ref: np.ndarray | None = None, ctrl_ref: np.ndarray | None = None,
                 Q: np.ndarray | None = None, R: np.ndarray | None = None, eps: float = 1e-6,
                 needs_linearization: bool = True, fused: bool = True):
        self.qpos_ref = None if qpos_ref is None else np.asarray(qpos_ref, dtype=float)
        self.ctrl_ref = None if ctrl_ref is None else np.asarray(ctrl_ref, dtype=float)
        self.Q, self.R, self.eps = Q, R, float(eps)
        self.capabilities = ControllerCapabilities(control_space=ControlSpace.TORQUE,
                                                   needs_linearization=bool(needs_linearization))
        self.fused = bool(fused)  # False: the same tick as a handful of torch ops (reference-style arithmetic)
        self._gain_uploaded = False
        self.K: np.ndarray | None = None
        self._dev: dict[str, Any] = {}

    def prepare(self, model: Any, data: Any) -> None:
        from . import _mj as mj

        nv, nu = model.nv, model.nu
        if nu == 0:
            raise ConfigError("BatchedLQRController requires nu>0")
        qref = np.array(model.qpos0) if self.qpos_ref is None else self.qpos_ref
        uref = np.zeros(nu) if self.ctrl_ref is None else self.ctrl_ref
        if self.K is None:
            probe = mj.MjData(model)  # one env in device-mapped host memory
            probe.qpos[:] = qref
            probe.qvel[:] = 0.0
            probe.ctrl[:] = uref
            A = np.zeros((2 * nv, 2 * nv))
            B = np.zeros((2 * nv, nu))
            mj.mjd_transitionFD(model, probe, self.eps, True, A, B, None, None)
            Q = np.eye(2 * nv) if self.Q is None else np.asarray(self.Q, dtype=float)
            R = np.eye(nu) if self.R is None else np.asarray(self.R, dtype=float)
            self.A0, self.B0 = A, B
            self.K = dlqr_gain(A, B, Q, R)
        if hasattr(data.qpos, "device"):
            import torch

            dev, dt = data.qpos.device, data.qpos.dtype
            self._dev = dict(
                K=torch.as_tensor(self.K, device=dev, dtype=dt), qref=torch.as_tensor(qref, device=dev, dtype=dt)[:, None],
                uref=torch.as_tensor(uref, device=dev, dtype=dt)[:, None],
                lo=torch.as_tensor(model.actuator_ctrlrange[:, 0], device=dev, dtype=dt)[:, None],
                hi=torch.as_tensor(model.actuator_ctrlrange[:, 1], device=dev, dtype=dt)[:, None],
                limited=torch.as_tensor(np.asarray(model.actuator_ctrllimited, dtype=bool), device=dev)[:, None],
                qref_full=None, dq=torch.zeros((nv, data.qpos.shape[1]), device=dev, dtype=dt))
        self._gain_uploaded = False
        self._free = bool(np.any(model.jnt_type == 0))
        self._qref_np, self._uref_np = qref, uref

    def device_law_ready(self, data: Any) -> bool:
        """True when the control law lives on the device (b2_lqr_set_gain done): ``BatchedEnv`` may then fold this
        controller's tick, the (A, B) linearisation and the step into one ``b2_control_tick`` launch."""
        b = data.backend
        if not (self.fused and hasattr(b, "batch") and hasattr(data.qpos, "device")):
            return False
        if not self._gain_uploaded:
            b.batch.lqr_set_gain(self.K, self._qref_np, self._uref_np)
            self._gain_uploaded = True
        return True

    def __call__(self, model: Any, data: Any, t: float) -> None:
        b = data.backend
        if self.device_law_ready(data):
            # one kernel: tangent-space state error, gain product, ctrlrange clamp (b2_lqr_control)
            b._launch("lqr_control", b.batch.lqr_control, b.state_struct())
            return
        import torch

        d = self._dev
        if self._free:
            if d["qref_full"] is None:
                d["qref_full"] = d["qref"].expand_as(data.qpos).contiguous()
            b._pre()
            b.batch.differentiate_pos(d["dq"].data_ptr(), 1.0, d["qref_full"].data_ptr(), data.qpos.data_ptr(), b.stream)
            dq = d["dq"]
        else:
            dq = data.qpos - d["qref"]
        x = torch.cat([dq, data.qvel], dim=0)
        u = d["uref"] - d["K"] @ x
        u = torch.where(d["limited"], torch.minimum(torch.maximum(u, d["lo"]), d["hi"]), u)
        data.ctrl.copy_(u)


class BatchedTVLQRController(BatchedLQRController):
    """Time-varying LQR: every control tick re-synthesises the gain of EVERY env from that env's latest FD linearisation
    ``(A_e, B_e)`` (``b2_dlqr``: DARE + gain on the device, one thread or warp per env) and applies it
    (``b2_lqr_control_env``) -- BASELINE config #2 read literally: "per-step FD (A, B) linearisation for LQR".

    The ``(A, B)`` are the ones the env computed for the previous tick (``needs_linearization=True``: ``BatchedEnv`` linearises
    after every controller call, reference ``env.py:178-190``), so the gain lags the state by one step; the first tick uses the
    setpoint gain of ``BatchedLQRController``.  No host round trip: three launches per tick (DARE, control law, FD) plus the
    step."""

    def __init__(self, *args, max_doublings: int = 40, tol: float = 1e-12, **kwargs):
        kwargs["fused"] = False
        super().__init__(*args, **kwargs)
        self.max_doublings, self.tol = int(max_doublings), float(tol)
        self._bufs = None
        self.lin_out = None   # (A, B) buffers BatchedEnv.linearize writes into: fixed addresses (CUDA-graph replay)
        self._have_lin = False

    def prepare(self, model: Any, data: Any) -> None:
        super().prepare(model, data)
        if hasattr(data.qpos, "device"):
            import torch

            nx, n = 2 * model.nv, data.qpos.shape[1]
            self.lin_out = (torch.zeros((nx, nx, n), dtype=data.qpos.dtype, device=data.qpos.device),
                            torch.zeros((nx, model.nu, n), dtype=data.qpos.dtype, device=data.qpos.device))
        self._have_lin = False

    def device_law_ready(self, data: Any) -> bool:  # the gain differs per env: BatchedEnv must not fold the tick
        return False

    def __call__(self, model: Any, data: Any, t: float) -> None:
        import torch

        from . import _capi

        b = data.backend
        if not (hasattr(b, "batch") and hasattr(data.qpos, "device")):
            raise ConfigError("BatchedTVLQRController drives a BatchedEnv (device tensors)")
        if not self._gain_uploaded:
            b.batch.lqr_set_gain(self.K, self._qref_np, self._uref_np)
            self._gain_uploaded = True
        if not self._have_lin or self.lin_out is None:   # first tick after prepare(): no linearisation yet
            self._have_lin = True
            b._launch("lqr_control", b.batch.lqr_control, b.state_struct())
            return
        A, B = self.lin_out
        nx, nu, n = A.shape[0], B.shape[1], A.shape[2]
        if self._bufs is None:
            self._bufs = (torch.empty((nu, nx, n), dtype=A.dtype, device=A.device), torch.empty((nx, nx, n), dtype=A.dtype, device=A.device),
                          torch.zeros(n, dtype=torch.int32, device=A.device))
            self._Q = np.ascontiguousarray(np.eye(nx) if self.Q is None else np.asarray(self.Q, dtype=float)).reshape(-1)
            self._R = np.ascontiguousarray(np.eye(nu) if self.R is None else np.asarray(self.R, dtype=float)).reshape(-1)
        K_env, P_env, status = self._bufs
        b._pre()
        _capi.dlqr(A.device.index, 64 if A.dtype == torch.float64 else 32, A.data_ptr(), B.data_ptr(), self._Q, self._R, nx, nu, n,
                   K_env.data_ptr(), P_env.data_ptr(), status.data_ptr(), self.max_doublings, self.tol, b.stream)
        b._launch("lqr_control_env", b.batch.lqr_control_env, b.state_struct(), K_env.data_ptr())

    @property
    def gains(self):
        """(K (N, nu, nx), P (N, nx, nx), status (N,)) of the last tick, or None before the first re-synthesis."""
        if self._bufs is None:
            return None
        K_env, P_env, status = self._bufs
        return K_env.permute(2, 0, 1), P_env.permute(2, 0, 1), status


class BatchedRandomController:
    """Random-rollout controller of BASELINE.json configs #3 / #4 ("batched random controls", drawn on the device every
    step): ``ctrl ~ U(lo, hi)`` i.i.d. per step, env and actuator, in ONE library launch (``b2_random_controls``, Philox
    keyed by ``(seed, env)``).  ``reset_below=(qpos_row, threshold)`` adds a rollout driver's episode reset to the same
    launch: an env whose ``qpos[qpos_row]`` has dropped below the threshold restarts from the state it had when
    ``prepare()`` (i.e. ``reset()``) last ran, or from ``set_reset_state(qpos, qvel)``."""

    def __init__(self, lo: float, hi: float, seed: int = 0, reset_below: tuple[int, float] | None = None):
        self.lo, self.hi, self.seed = float(lo), float(hi), int(seed)
        self.reset_below = reset_below
        self.capabilities = ControllerCapabilities(control_space=ControlSpace.TORQUE)
        self._reset = None

    def prepare(self, model: Any, data: Any) -> None:
        if model.nu == 0:
            raise ConfigError("BatchedRandomController requires nu>0")
        if not hasattr(data.qpos, "device"):
            raise ConfigError("BatchedRandomController drives a BatchedEnv (device tensors)")
        if self.reset_below is not None:
            self.set_reset_state(data.qpos, data.qvel)

    def set_reset_state(self, qpos: Any, qvel: Any) -> None:
        self._reset = (qpos.clone(), qvel.clone())

    def __call__(self, model: Any, data: Any, t: float) -> None:
        b = data.backend
        row, thr = self.reset_below if self.reset_below is not None else (-1, 0.0)
        rq = self._reset[0].data_ptr() if self._reset is not None else None
        rv = self._reset[1].data_ptr() if self._reset is not None else None
        b._launch("random_controls", b.batch.random_controls, b.state_struct(), self.lo, self.hi, self.seed, row, thr, rq, rv)


__all__ = ["BatchedLQRController", "BatchedTVLQRController", "BatchedRandomController", "batched_dlqr_gain", "batched_ilqr", "batched_tvlqr",
           "dlqr_gain"]
