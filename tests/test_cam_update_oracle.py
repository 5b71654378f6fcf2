"""The statistical yardstick of the camera-state measurement update, on the numpy oracle alone (no device).

The filter's own motion model is linear and decoupled from (q, omega) on the (r, v) rows (fv, dfv_by_dxv, func_Q of
mc/): r' = r + (v + V) dt, v' = v + V, V ~ N(0, (std_a dt)^2 I), which is func_Q's G Pn G' on those rows.  A truth drawn
from that model and from the initial (x0, P0) makes a filter that only sees linear (r, v) fixes exactly consistent, so
the mean NIS of a fix with m rows is m.  tests/test_gpu_cam_update.py checks the device against the same number."""
import numpy as np

from oracle import ekf_oracle as O

STD_A = 0.007
DT = 1.0     # predict_state_and_covariance's delta_t


def initial_camera():
    """mc/initialize_x_and_p.m: the camera-only filter's x0 [13], P0 [13, 13]."""
    return O.initialize_x_and_p()


def draw_truth(rng, x0, P0, nb):
    """nb truth states [nb, 13] drawn from N(x0, P0) (P0 is diagonal)."""
    return x0 + rng.standard_normal((nb, 13)) * np.sqrt(np.diag(P0))


def truth_step(rng, xt):
    """One step of the (r, v) model on truth states [nb, 13] (in place); q and omega are not modelled."""
    V = rng.standard_normal((len(xt), 3)) * (STD_A * DT)
    xt[:, 0:3] += (xt[:, 7:10] + V) * DT
    xt[:, 7:10] += V
    return xt


def fix_model(m, sigma_r=0.05, sigma_v=0.01):
    """H [m, 13] and R [m, m] of a position fix (m = 3) or a position and velocity fix (m = 6)."""
    H = np.zeros((m, 13))
    H[0:3, 0:3] = np.eye(3)
    sig = [sigma_r] * 3
    if m == 6:
        H[3:6, 7:10] = np.eye(3)
        sig += [sigma_v] * 3
    return H, np.diag(np.square(sig))


def nis(P, H, R, nu):
    S = H @ P @ H.T + R
    return float(nu @ np.linalg.solve(S, nu))


def run_oracle(m, runs, frames, seed):
    """Mean NIS of `runs` camera-only filters x `frames` (predict, then an m-row fix) through the oracle."""
    rng = np.random.RandomState(seed)
    x0, P0 = initial_camera()
    H, R = fix_model(m)
    Lr = np.linalg.cholesky(R)
    xt = draw_truth(rng, x0, P0, runs)
    total = 0.0
    for b in range(runs):
        x, P = x0.copy(), P0.copy()
        t = xt[b:b + 1].copy()
        for _ in range(frames):
            x, P = O.predict_state_and_covariance(x, P, "constant_velocity", STD_A, STD_A)
            truth_step(rng, t)
            z = H @ t[0] + Lr @ rng.standard_normal(m)
            total += nis(P, H, R, z - H @ x)
            x, P, _ = O.update(x, P, H, R, z, H @ x)
    return total / (runs * frames)


def test_truth_model_is_func_Q():
    """The truth simulator's (r, v) increment covariance equals func_Q's G Pn G' on those rows."""
    x0, _ = initial_camera()
    la = (STD_A * DT) ** 2
    Q = O.func_Q(x0, np.zeros(6), np.diag([la] * 3 + [STD_A ** 2] * 3), DT, "constant_velocity")
    idx = np.r_[0:3, 7:10]
    # [dr; dv] = [V dt; V] given (r, v): covariance [[dt^2, dt], [dt, 1]] (x) la I
    C = np.kron(np.array([[DT * DT, DT], [DT, 1.0]]), la * np.eye(3))
    assert np.allclose(Q[np.ix_(idx, idx)], C, rtol=0, atol=1e-18)
    F = O.dfv_by_dxv(x0, np.zeros(6), DT, "constant_velocity")
    assert np.array_equal(F[np.ix_(idx, idx)], np.block([[np.eye(3), DT * np.eye(3)], [np.zeros((3, 3)), np.eye(3)]]))
    # (r, v) rows are decoupled from (q, omega) in F and Q
    other = np.r_[3:7, 10:13]
    assert not F[np.ix_(idx, other)].any() and not Q[np.ix_(idx, other)].any()


def test_mean_nis_is_m():
    """1500 runs x 20 frames = 30000 samples: the standard error of the mean NIS is sqrt(2/(m 30000)) relative
    (0.47 % for m = 3, 0.33 % for m = 6), so the 3 % band is more than 6 standard errors wide."""
    for m, seed in ((3, 11), (6, 12)):
        mean = run_oracle(m, runs=1500, frames=20, seed=seed)
        assert abs(mean / m - 1.0) < 0.03, (m, mean)


def test_inconsistent_filter_is_detected():
    """The yardstick has power: the same scenario with R understated four times gives a mean NIS far above m."""
    rng = np.random.RandomState(5)
    x0, P0 = initial_camera()
    H, R = fix_model(3)
    xt = draw_truth(rng, x0, P0, 200)
    total, cnt = 0.0, 0
    for b in range(200):
        x, P = x0.copy(), P0.copy()
        t = xt[b:b + 1].copy()
        for _ in range(10):
            x, P = O.predict_state_and_covariance(x, P, "constant_velocity", STD_A, STD_A)
            truth_step(rng, t)
            z = H @ t[0] + np.linalg.cholesky(R) @ rng.standard_normal(3)
            total += nis(P, H, R / 4, z - H @ x)
            cnt += 1
            x, P, _ = O.update(x, P, H, R / 4, z, H @ x)
    assert total / cnt > 1.5 * 3
