"""Pins the NumPy statement of b2_traj_cost (tests/traj_cost_reference.py) without a GPU: its gradients are the central
differences of J under xbar (+) h d (also through large rotation errors of a free joint), G is the identity on hinge and
slide models and wherever the rotation weight is isotropic, and the small-angle series of Jr^-1 joins the closed form."""
import numpy as np
import pytest

import traj_cost_reference as ref
from conftest import load_model, random_states


def _problem(name, T, seed, max_angle=2.5, iso_rot=None):
    """A random trajectory, reference and non-diagonal SPD weights for a golden model."""
    model = load_model(name)
    rng = np.random.default_rng(seed)
    jnts, nv, nu = ref.joints(model), model.nv, model.nu
    qs = np.stack([random_states(model, name, T + 1, seed=seed)[0][t] for t in range(T + 1)])
    for typ, pa, _ in jnts:
        if typ != ref.JNT_FREE:
            qs[:, pa] += rng.normal(0, 0.5, T + 1)
    qr = ref.random_rotation_errors(rng, jnts, qs, max_angle) if max_angle else qs.copy()
    for typ, pa, _ in jnts:  # position errors too
        qr[:, pa:pa + (3 if typ == ref.JNT_FREE else 1)] += rng.normal(0, 0.3, (T + 1, 3 if typ == ref.JNT_FREE else 1))
    vs, vr = rng.normal(size=(T + 1, nv)), rng.normal(size=(T + 1, nv))
    us, ur = rng.normal(size=(T, nu)), rng.normal(size=(T, nu))
    Q, R, Qf = ref.random_spd(rng, 2 * nv), ref.random_spd(rng, nu), ref.random_spd(rng, 2 * nv, 30.0)
    if iso_rot is not None:  # rotation blocks of Q and Qf set to c I, decoupled from the rest
        for typ, _, va in jnts:
            if typ == ref.JNT_FREE:
                for M in (Q, Qf):
                    M[va + 3:va + 6, :] = 0
                    M[:, va + 3:va + 6] = 0
                    M[va + 3:va + 6, va + 3:va + 6] = iso_rot * np.eye(3)
    return model, jnts, (qs, vs, us, qr, vr, ur), (Q, R, Qf)


def _fd_residual(jnts, nv, traj, W, d, du, h):
    qs, vs, us, qr, vr, ur = traj
    J0, q, r = ref.traj_cost(jnts, nv, qs, vs, us, qr, vr, ur, *W)
    Jp = ref.traj_cost(jnts, nv, *ref.perturb(jnts, nv, qs, vs, h * d), us + h * du, qr, vr, ur, *W)[0]
    Jm = ref.traj_cost(jnts, nv, *ref.perturb(jnts, nv, qs, vs, -h * d), us - h * du, qr, vr, ur, *W)[0]
    analytic = float(np.sum(q * d) + np.sum(r * du))
    return abs((Jp - Jm) / (2 * h) - analytic), analytic


def test_rotation_errors_reach_the_requested_angles():
    model, jnts, traj, _ = _problem("drone", 24, 0)
    qs, qr = traj[0], traj[3]
    angles = [np.linalg.norm(ref.differentiate_pos(jnts, model.nv, qr[t], qs[t])[3:]) for t in range(qs.shape[0])]
    assert max(angles) > 2.0 and max(angles) <= 2.5 + 1e-12


@pytest.mark.parametrize("name", ["drone", "pendulum", "cartpole"])
def test_gradient_is_the_central_difference_of_J(name):
    """Halving h quarters the residual: the analytic gradient is exact, Jr^-1 included (anisotropic rotation weight)."""
    model, jnts, traj, W = _problem(name, 12, 1)
    rng = np.random.default_rng(2)
    d, du = rng.normal(size=(13, 2 * model.nv)), rng.normal(size=(12, model.nu))
    res = [_fd_residual(jnts, model.nv, traj, W, d, du, h)[0] for h in (2e-3, 1e-3)]
    ratio = res[0] / res[1]
    print(f"central-difference residual {name}: {res[0]:.2e} -> {res[1]:.2e}, ratio {ratio:.2f}")
    assert 3.5 <= ratio <= 4.5 or res[0] < 1e-9, res


def test_dropping_jr_inv_breaks_the_gradient_on_a_free_joint():
    model, jnts, traj, W = _problem("drone", 12, 3)
    rng = np.random.default_rng(4)
    d, du = rng.normal(size=(13, 2 * model.nv)), rng.normal(size=(12, model.nu))
    res, analytic = _fd_residual(jnts, model.nv, traj, W, d, du, 1e-4)
    qs, vs, us, qr, vr, ur = traj
    q_naive = ref.traj_cost(jnts, model.nv, qs, vs, us, qr, vr, ur, *W, exact=False)[1]
    naive = float(np.sum(q_naive * d) + np.sum(ref.traj_cost(jnts, model.nv, *traj, *W)[2] * du))
    assert abs(naive - analytic) > 1e4 * res, (naive, analytic, res)


@pytest.mark.parametrize("name", ["pendulum", "cartpole"])
def test_G_is_the_identity_without_free_joints(name):
    model, jnts, traj, W = _problem(name, 8, 5)
    exact = ref.traj_cost(jnts, model.nv, *traj, *W)
    naive = ref.traj_cost(jnts, model.nv, *traj, *W, exact=False)
    assert exact[0] == naive[0] and np.array_equal(exact[1], naive[1]) and np.array_equal(exact[2], naive[2])


def test_isotropic_rotation_weight_makes_G_vanish():
    """Jr^-1(phi)' phi = phi: with the rotation block c I (decoupled), G'Qe = Qe."""
    model, jnts, traj, W = _problem("drone", 8, 6, iso_rot=3.0)
    exact = ref.traj_cost(jnts, model.nv, *traj, *W)[1]
    naive = ref.traj_cost(jnts, model.nv, *traj, *W, exact=False)[1]
    assert np.max(np.abs(exact - naive)) <= 1e-12 * np.max(np.abs(naive))


def test_small_angle_series_joins_the_closed_form():
    th = 0.1
    below, above = ref.jr_inv_coef(np.nextafter(th, 0)), ref.jr_inv_coef(th)
    assert abs(below - above) <= 1e-14, (below, above)
    for t in (1e-8, 1e-4, 0.05, 0.0999):
        closed = 1 / t**2 - (1 + np.cos(t)) / (2 * t * np.sin(t))
        assert abs(ref.jr_inv_coef(t) - 1 / 12) <= t * t / 700 + 1e-16
        if t >= 0.05:  # where the closed form is still accurate
            assert abs(ref.jr_inv_coef(t) - closed) <= 1e-12
    assert ref.jr_inv_coef(0.0) == 1 / 12


def test_jr_inv_inverts_the_right_jacobian():
    """Jr(phi) = I - (1 - cos th)/th^2 [phi]x + (th - sin th)/th^3 [phi]x^2; Jr^-1 is its inverse."""
    rng = np.random.default_rng(7)
    for th in (0.01, 0.3, 1.5, 2.5, 3.0):
        phi = rng.normal(size=3)
        phi *= th / np.linalg.norm(phi)
        S = ref.skew(phi)
        Jr = np.eye(3) - (1 - np.cos(th)) / th**2 * S + (th - np.sin(th)) / th**3 * S @ S
        assert np.max(np.abs(ref.jr_inv(phi) @ Jr - np.eye(3))) <= 1e-12
