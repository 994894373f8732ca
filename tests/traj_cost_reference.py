"""Plain NumPy statement of b2_traj_cost (include/b2mj.h) for one env: the tracking cost J of a trajectory and its
gradients q_t = G_t' M e_t, r_t = R w_t with respect to the tangent deviation x_t = xbar_t (+) dx_t, together with the
(-) and (+) operators of b2_differentiate_pos / b2_integrate_pos, so that the definition can be pinned against finite
differences independently of the kernels."""
import numpy as np

JNT_FREE = 0


def joints(model):
    """(type, qposadr, dofadr) of every joint of a model (anything with jnt_type / jnt_qposadr / jnt_dofadr)."""
    return [(int(t), int(a), int(d)) for t, a, d in zip(model.jnt_type, model.jnt_qposadr, model.jnt_dofadr)]


def quat_mul(a, b):
    return np.array([a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3],
                     a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2],
                     a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1],
                     a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0]])


def quat_log(q):
    """Rotation vector of a unit quaternion on the shortest path (angle in (-pi, pi], as quat_to_vel)."""
    s = np.linalg.norm(q[1:])
    if s == 0:
        return np.zeros(3)
    angle = 2 * np.arctan2(s, q[0])
    if angle > np.pi:
        angle -= 2 * np.pi
    return q[1:] / s * angle


def quat_exp(w):
    th = np.linalg.norm(w)
    if th == 0:
        return np.array([1.0, 0, 0, 0])
    return np.concatenate([[np.cos(th / 2)], w / th * np.sin(th / 2)])


def differentiate_pos(jnts, nv, qref, q):
    """q (-) qref: b2_differentiate_pos(dt = 1, qref -> q)."""
    out = np.zeros(nv)
    for typ, pa, va in jnts:
        if typ == JNT_FREE:
            out[va:va + 3] = q[pa:pa + 3] - qref[pa:pa + 3]
            conj = qref[pa + 3:pa + 7] * np.array([1, -1, -1, -1])
            out[va + 3:va + 6] = quat_log(quat_mul(conj, q[pa + 3:pa + 7]))
        else:
            out[va] = q[pa] - qref[pa]
    return out


def integrate_pos(jnts, q, v):
    """q (+) v: b2_integrate_pos(dt = 1); a free joint's rotation is normalize(q) (x) Exp(v_rot)."""
    q = np.array(q, dtype=float)
    for typ, pa, va in jnts:
        if typ == JNT_FREE:
            q[pa:pa + 3] += v[va:va + 3]
            quat = q[pa + 3:pa + 7] / np.linalg.norm(q[pa + 3:pa + 7])
            q[pa + 3:pa + 7] = quat_mul(quat, quat_exp(v[va + 3:va + 6]))
        else:
            q[pa] += v[va]
    return q


def jr_inv_coef(th):
    """c(th) of Jr^-1 = I + 1/2 [phi]x + c [phi]x^2: 1/th^2 - (1 + cos th) / (2 th sin th), its series below th = 0.1."""
    th2 = th * th
    if th2 < 1e-2:
        return 1 / 12 + th2 * (1 / 720 + th2 * (1 / 30240 + th2 / 1209600))
    return 1 / th2 - (1 + np.cos(th)) / (2 * th * np.sin(th))


def skew(p):
    return np.array([[0, -p[2], p[1]], [p[2], 0, -p[0]], [-p[1], p[0], 0]])


def jr_inv(phi):
    S = skew(phi)
    return np.eye(3) + 0.5 * S + jr_inv_coef(np.linalg.norm(phi)) * S @ S


def G(jnts, nv, e):
    """The chain-rule matrix of e with respect to the tangent deviation: identity but Jr^-1(phi) on free rotations."""
    g = np.eye(2 * nv)
    for typ, pa, va in jnts:
        if typ == JNT_FREE:
            g[va + 3:va + 6, va + 3:va + 6] = jr_inv(e[va + 3:va + 6])
    return g


def traj_cost(jnts, nv, qs, vs, us, qr, vr, ur, Q, R, Qf, exact=True):
    """qs, qr (T+1, nq), vs, vr (T+1, nv), us, ur (T, nu); vr / ur may be None.  Returns (J, q (T+1, 2nv), r (T, nu)).
    exact=False drops G (q_t = M e_t): what a caller who ignores the rotation's chain rule would compute."""
    T = us.shape[0]
    J, q, r = 0.0, np.empty((T + 1, 2 * nv)), np.empty((T, R.shape[0]))
    for t in range(T + 1):
        e = np.concatenate([differentiate_pos(jnts, nv, qr[t], qs[t]), vs[t] - (0 if vr is None else vr[t])])
        M = Q if t < T else Qf
        J += 0.5 * e @ M @ e
        q[t] = (G(jnts, nv, e).T if exact else np.eye(2 * nv)) @ (M @ e)
        if t < T:
            w = us[t] - (0 if ur is None else ur[t])
            J += 0.5 * w @ R @ w
            r[t] = R @ w
    return J, q, r


def perturb(jnts, nv, qs, vs, dx):
    """The trajectory xbar (+) dx: qs (T+1, nq), vs (T+1, nv), dx (T+1, 2nv)."""
    return np.stack([integrate_pos(jnts, qs[t], dx[t, :nv]) for t in range(qs.shape[0])]), vs + dx[:, nv:]


def random_spd(rng, n, cond=10.0):
    U, _ = np.linalg.qr(rng.normal(size=(n, n)))
    M = U @ np.diag(np.geomspace(1.0, cond, n)) @ U.T
    return 0.5 * (M + M.T)


def random_rotation_errors(rng, jnts, qs, max_angle):
    """qs with every free joint's quaternion rotated by a random rotation of angle up to max_angle (the reference qpos
    is then qs and the result differs from it by that rotation)."""
    out = np.array(qs, dtype=float)
    for typ, pa, _ in jnts:
        if typ == JNT_FREE:
            for t in range(out.shape[0]):
                axis = rng.normal(size=3)
                axis /= np.linalg.norm(axis)
                out[t, pa + 3:pa + 7] = quat_mul(out[t, pa + 3:pa + 7], quat_exp(axis * rng.uniform(0, max_angle)))
    return out
