"""Plain NumPy statement of b2_tvlqr's backward pass (include/b2mj.h) for one env, and the linear-quadratic problem it
solves, so that the recursion can be pinned independently of the kernels: the cost of a trajectory, a linear rollout of
the feedback policy, and the same problem written as one dense least-squares problem over all controls."""
import numpy as np


def tvlqr(A, B, Q, R, Qf=None, q=None, r=None, reg=0.0):
    """A (T, nx, nx), B (T, nx, nu); q (T+1, nx), r (T, nu) or None.  Returns K (T, nu, nx), k (T, nu), P0 (nx, nx),
    dV (2,) and status (0, or -(t+1) for the first step from the end whose Quu + reg I is not positive definite; rows <= t
    of K and k, P0 and dV are then NaN)."""
    T, nx, nu = A.shape[0], A.shape[1], B.shape[2]
    Qf = Q if Qf is None else Qf
    P = np.array(Qf, dtype=float)
    s = np.zeros(nx) if q is None else np.array(q[T], dtype=float)
    K, k = np.empty((T, nu, nx)), np.empty((T, nu))
    dV, status = np.zeros(2), 0
    for t in range(T - 1, -1, -1):
        At, Bt = A[t], B[t]
        Qx = (0 if q is None else q[t]) + At.T @ s
        Qu = (0 if r is None else r[t]) + Bt.T @ s
        Qxx, Quu, Qux = Q + At.T @ P @ At, R + Bt.T @ P @ Bt, Bt.T @ P @ At
        try:
            L = np.linalg.cholesky(Quu + reg * np.eye(nu))
            Kt = np.linalg.solve(L.T, np.linalg.solve(L, Qux))
            kt = -np.linalg.solve(L.T, np.linalg.solve(L, Qu))
        except np.linalg.LinAlgError:
            status = status or -(t + 1)
            Kt, kt = np.full((nu, nx), np.nan), np.full(nu, np.nan)
        K[t], k[t] = Kt, kt
        P = Qxx + Kt.T @ Quu @ Kt - Kt.T @ Qux - Qux.T @ Kt
        P = 0.5 * (P + P.T)
        s = Qx - Kt.T @ Qu - Kt.T @ Quu @ kt + Qux.T @ kt
        dV += (kt @ Qu, 0.5 * kt @ Quu @ kt)
    return K, k, P, dV, status


def cost(xs, us, Q, R, Qf=None, q=None, r=None):
    """J of deviations xs (T+1, nx), us (T, nu)."""
    Qf = Q if Qf is None else Qf
    T = us.shape[0]
    J = 0.5 * xs[T] @ Qf @ xs[T] + (0 if q is None else q[T] @ xs[T])
    for t in range(T):
        J += 0.5 * xs[t] @ Q @ xs[t] + 0.5 * us[t] @ R @ us[t]
        J += (0 if q is None else q[t] @ xs[t]) + (0 if r is None else r[t] @ us[t])
    return J


def rollout_linear(A, B, x0, K, k, alpha=1.0):
    """x_{t+1} = A_t x_t + B_t u_t under u_t = alpha k_t - K_t x_t.  Returns xs (T+1, nx), us (T, nu)."""
    T = A.shape[0]
    xs, us = [np.asarray(x0, dtype=float)], []
    for t in range(T):
        us.append(alpha * k[t] - K[t] @ xs[-1])
        xs.append(A[t] @ xs[-1] + B[t] @ us[-1])
    return np.array(xs), np.array(us)


def dense_minimiser(A, B, x0, Q, R, Qf=None, q=None, r=None):
    """The optimal open-loop controls (T, nu) of the same problem from x0, with x = F x0 + G u substituted: one dense
    least-squares problem over all controls."""
    T, nx, nu = A.shape[0], A.shape[1], B.shape[2]
    Qf = Q if Qf is None else Qf
    F = np.zeros(((T + 1) * nx, nx))
    G = np.zeros(((T + 1) * nx, T * nu))
    F[:nx] = np.eye(nx)
    for t in range(T):
        rows, prev = slice((t + 1) * nx, (t + 2) * nx), slice(t * nx, (t + 1) * nx)
        F[rows] = A[t] @ F[prev]
        G[rows] = A[t] @ G[prev]
        G[rows, t * nu:(t + 1) * nu] += B[t]
    Qbig = np.zeros(((T + 1) * nx, (T + 1) * nx))
    for t in range(T + 1):
        Qbig[t * nx:(t + 1) * nx, t * nx:(t + 1) * nx] = Qf if t == T else Q
    Rbig = np.kron(np.eye(T), R)
    qbig = np.zeros((T + 1) * nx) if q is None else np.asarray(q).reshape(-1)
    rbig = np.zeros(T * nu) if r is None else np.asarray(r).reshape(-1)
    H = G.T @ Qbig @ G + Rbig
    g = G.T @ (Qbig @ F @ x0 + qbig) + rbig
    return np.linalg.solve(H, -g).reshape(T, nu)


def random_system(rng, T, nx, nu, scale=0.3):
    """A time-varying linear system near the identity, with random positive-definite weights and linear terms."""
    A = np.eye(nx) + scale * rng.normal(size=(T, nx, nx))
    B = rng.normal(size=(T, nx, nu))
    M = rng.normal(size=(nx, nx))
    Q = M @ M.T / nx + 0.1 * np.eye(nx)
    N = rng.normal(size=(nu, nu))
    R = N @ N.T / nu + 0.1 * np.eye(nu)
    F = rng.normal(size=(nx, nx))
    Qf = F @ F.T / nx + np.eye(nx)
    return A, B, Q, R, Qf, rng.normal(size=(T + 1, nx)), rng.normal(size=(T, nu))
