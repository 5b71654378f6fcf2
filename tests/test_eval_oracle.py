"""The numpy mirror of the scoring against the ground truth (oracle/eval_oracle.py) on its own, no device: its
Jacobians against central differences, a perfect estimate, the NEES of a seeded linear-Gaussian draw against its
degrees of freedom, and the skip / status rules."""
import math

import numpy as np

from oracle import eval_oracle as E


def _quat(rng):
    q = rng.normal(size=4)
    q /= np.linalg.norm(q)
    return q if q[0] > 0 else -q


def _spd(rng, n, scale):
    A = rng.normal(size=(n, n)) * scale
    return A @ A.T + np.eye(n) * scale * scale


def _invdepth_of(point, anchor, rho_scale=1.0):
    d = point - anchor
    th = math.atan2(d[0], d[2])
    ph = math.atan2(-d[1], math.sqrt(d[0] * d[0] + d[2] * d[2]))
    return np.array([anchor[0], anchor[1], anchor[2], th, ph, rho_scale / np.linalg.norm(d)])


def _state(rng, r_t, q_t, points, types):
    """x with the camera at the truth and every feature exactly at its point (inverse depth anchored at r_t)."""
    x = [r_t, q_t, rng.normal(size=6) * 0.01]
    for k, ty in enumerate(types):
        x.append(_invdepth_of(points[k], r_t) if ty == 1 else points[k].copy())
    return np.concatenate(x)


def test_orientation_jacobian_matches_central_differences():
    rng = np.random.RandomState(3)
    for _ in range(5):
        r_t, q_t = rng.normal(size=3), _quat(rng)
        x = np.concatenate([r_t + 0.1 * rng.normal(size=3), q_t + 0.05 * rng.normal(size=4)])
        P = np.eye(7)
        cam = E.camera(x, P, r_t, q_t)
        h = 1e-6
        Jfd = np.zeros((6, 7))
        for k in range(7):
            xp, xm = x.copy(), x.copy()
            xp[k] += h
            xm[k] -= h
            cp, cm = E.camera(xp, P, r_t, q_t), E.camera(xm, P, r_t, q_t)
            Jfd[:, k] = (np.concatenate([cp["e_r"], cp["e_theta"]]) - np.concatenate([cm["e_r"], cm["e_theta"]])) / (2 * h)
        assert np.abs(Jfd - cam["J"]).max() < 1e-8


def test_orientation_error_is_the_rotation_angle():
    rng = np.random.RandomState(4)
    r_t, q_t = np.zeros(3), _quat(rng)
    ang = 0.3
    axis = rng.normal(size=3)
    axis /= np.linalg.norm(axis)
    dq = np.concatenate([[math.cos(ang / 2)], math.sin(ang / 2) * axis])
    from oracle.ekf_oracle import dq3_by_dq1
    q_hat = dq3_by_dq1(q_t) @ dq                     # q_t * dq
    for sign in (1.0, -1.0):                         # q and -q are the same rotation
        cam = E.camera(np.concatenate([r_t, sign * q_hat]), np.eye(7), r_t, q_t)
        assert abs(cam["angle"] - ang) < 1e-12
        assert np.abs(cam["e_theta"] - 2 * math.sin(ang / 2) * axis).max() < 1e-12


def test_inverse_depth_jacobian_matches_central_differences():
    rng = np.random.RandomState(5)
    for _ in range(10):
        y = np.concatenate([rng.normal(size=3), rng.uniform(-1, 1, 2), [rng.uniform(0.1, 2.0)]])
        p, J = E.feature_cartesian(y, 1)
        Jfd = np.zeros((3, 6))
        for k in range(6):
            h = 1e-6 * max(1.0, abs(y[k]))
            yp, ym = y.copy(), y.copy()
            yp[k] += h
            ym[k] -= h
            Jfd[:, k] = (E.feature_cartesian(yp, 1)[0] - E.feature_cartesian(ym, 1)[0]) / (2 * h)
        assert np.abs(Jfd - J).max() / np.abs(J).max() < 1e-7
    p, J = E.feature_cartesian(np.array([1.0, 2.0, 3.0]), 2)
    assert np.array_equal(p, [1.0, 2.0, 3.0]) and np.array_equal(J, np.eye(3))


def test_perfect_estimate_scores_zero():
    rng = np.random.RandomState(6)
    r_t, q_t = rng.normal(size=3), _quat(rng)
    types = np.array([1, 2, 1, 2], dtype=np.uint8)
    pts = rng.normal(size=(4, 3)) * 3 + np.array([0, 0, 6.0])
    x = _state(rng, r_t, q_t, pts, types)
    P = _spd(rng, len(x), 0.1)
    rec, fe, fn = E.evaluate(x, P, types, 4, np.arange(4), pts, r_t, q_t)
    assert rec["pos_sq_err"] == 0.0 and rec["rot_sq_err"] == 0.0
    assert rec["nees_pos"] == 0.0 and rec["nees_pose"] == 0.0
    assert rec["n_map"] == 4 and rec["n_skip"] == 0 and rec["status"] == 0 and rec["frames"] == 1
    # inverse depth -> Cartesian rounds in the last bits of the point
    assert rec["map_sq_err"] < 1e-28 and rec["map_nees"] < 1e-24
    assert np.abs(fe).max() < 1e-14 and fn.max() < 1e-24


def test_linear_gaussian_mean_nees_is_the_dof():
    """x ~ N(truth, P): e = J (x - truth) exactly for the camera (e_theta is linear in q_hat), to first order for the
    features (small covariance), so each NEES is chi-square with its dof; 20 000 seeded draws put the mean within 3 %."""
    rng = np.random.RandomState(2024)
    r_t, q_t = np.array([0.3, -0.2, 0.1]), _quat(rng)
    types = np.array([1, 2], dtype=np.uint8)
    pts = np.array([[0.5, -0.4, 5.0], [-1.0, 0.7, 4.0]])
    x0 = _state(rng, r_t, q_t, pts, types)
    n = len(x0)
    P = _spd(rng, n, 0.01)
    P[13:, 13:] *= 0.1                                       # keep the inverse-depth block in its linear range
    P[:13, 13:] *= math.sqrt(0.1)
    P[13:, :13] *= math.sqrt(0.1)
    Lc = np.linalg.cholesky(P)
    S = 20000
    nees = np.zeros((S, 4))
    draws = rng.normal(size=(S, n))
    for k in range(S):
        x = x0 + Lc @ draws[k]
        rec, _, fn = E.evaluate(x, P, types, 2, np.arange(2), pts, r_t, q_t)
        assert rec["n_map"] == 2 and rec["status"] == 0
        nees[k] = rec["nees_pos"], rec["nees_pose"], fn[0], fn[1]
    mean = nees.mean(axis=0)
    dof = np.array([3.0, 6.0, 3.0, 3.0])
    print("mean NEES", mean, "dof", dof)
    assert (np.abs(mean / dof - 1.0) < 0.03).all(), mean


def test_skips_and_status_bits():
    rng = np.random.RandomState(8)
    r_t, q_t = np.zeros(3), np.array([1.0, 0, 0, 0])
    types = np.array([1, 1, 2, 2, 1, 0], dtype=np.uint8)
    pts = rng.normal(size=(3, 3)) + np.array([0, 0, 5.0])
    x = _state(rng, r_t, q_t, pts[[0, 1, 2, 0, 1]], types[:5])
    x = np.concatenate([x, np.zeros(6)])
    P = _spd(rng, len(x), 0.1)
    off = E.offsets(types, 5)
    tags = np.array([0, 1, 2, -1, 7, 0])
    x[off[1] + 5] = -0.2                                    # rho <= 0: not evaluable
    P[off[2]:off[2] + 3, :] = 0.0                           # Cartesian block with a zero pivot: not evaluable
    P[:, off[2]:off[2] + 3] = 0.0
    rec, fe, fn = E.evaluate(x, P, types, 5, tags, pts, r_t, q_t, N=6)
    # slot 0 ok; 1 rho <= 0; 2 zero covariance; 3 tag -1; 4 tag >= M; slot 5 beyond nfeat is empty
    assert rec["n_map"] == 1 and rec["n_skip"] == 4
    assert rec["status"] == E.NO_TRUTH | E.NOT_EVALUABLE
    assert np.isfinite(fn[0]) and np.isnan(fn[1:]).all() and np.isnan(fe[1:]).all()
    assert rec["map_nees"] == fn[0]
    # camera covariance not SPD: NaN NEES, status bit 0, the errors still reported
    P0 = P.copy()
    P0[:7, :] = 0.0
    P0[:, :7] = 0.0
    rec0, _, _ = E.evaluate(x, P0, types, 5, tags, pts, r_t, q_t, N=6)
    assert rec0["status"] & E.CAM_NOT_SPD and math.isnan(rec0["nees_pos"]) and math.isnan(rec0["nees_pose"])
    assert rec0["pos_sq_err"] == rec["pos_sq_err"]
    # the map export skips the same slots (it needs no truth: slots 3 and 4 are exported)
    p, C = E.map_cartesian(x, P, types, 5, 6)
    assert np.isnan(p[[1, 2, 5]]).all() and np.isfinite(p[[0, 3, 4]]).all()
    assert np.isnan(C[[1, 2, 5]]).all() and np.allclose(C[0], C[0].T)
