"""The known-landmark update's numpy mirror (oracle/landmark_oracle.py) and the synthetic landmark observations
(SynthWorld.landmark_obs), with no device: the landmark Jacobians against central differences of hi_cartesian, an exact
zero correction for a perfect observation, the statuses of landmarks that cannot be seen, the NIS statistics of the
update on a truth drawn from the filter's own covariance, and the observations against their definition.
tests/test_gpu_landmark_update.py checks the device against the mirror."""
import math

import numpy as np

import ekf_slam_b200.synth as synth
from oracle import ekf_oracle as O
from oracle import landmark_oracle as LO

CAM = O.initialize_cam()


def camera_state(r=(0.05, -0.02, 0.1), q=(1.0, 0.03, -0.02, 0.01)):
    """x [13]: a camera at r with the unit quaternion along q, at rest."""
    x = np.zeros(13)
    x[0:3] = r
    x[3:7] = np.asarray(q) / np.linalg.norm(q)
    return x


def camera_cov(sr=0.01, sq=0.002, sv=0.01):
    return np.diag([sr ** 2] * 3 + [sq ** 2] * 4 + [sv ** 2] * 6)


def world_point(xv, hrl):
    """The world point whose camera-frame ray (R' (p - r)) is hrl, for a unit quaternion."""
    return xv[0:3] + O.q2r(xv[3:7]) @ np.asarray(hrl, dtype=np.float64)


def pixel_ray(uv, depth):
    """Camera-frame point at `depth` along the ray of distorted pixel uv."""
    uu = O.undistort_fm(np.asarray(uv, dtype=np.float64), CAM)
    return np.array([(uu[0] - CAM.Cx) / (CAM.f / CAM.dx), (uu[1] - CAM.Cy) / (CAM.f / CAM.dy), 1.0]) * depth


def test_jacobians_central_differences():
    x = camera_state()
    for uv, depth in (((60.0, 50.0), 2.0), ((250.0, 190.0), 4.5), ((160.0, 120.0), 1.2)):
        p = world_point(x, pixel_ray(uv, depth))
        h = LO.predict(x, p, CAM)
        A, Jp = LO.jacobians(x, p, CAM, h)
        num_A, num_p = np.zeros((2, 7)), np.zeros((2, 3))
        for i in range(7):
            d = np.zeros(13)
            d[i] = 1e-6
            num_A[:, i] = (LO.predict(x + d, p, CAM) - LO.predict(x - d, p, CAM)) / 2e-6
        for i in range(3):
            d = np.zeros(3)
            d[i] = 1e-6
            num_p[:, i] = (LO.predict(x, p + d, CAM) - LO.predict(x, p - d, CAM)) / 2e-6
        assert np.abs(A - num_A).max() < 1e-5 * np.abs(A).max(), (uv, A, num_A)
        assert np.abs(Jp - num_p).max() < 1e-5 * np.abs(Jp).max(), (uv, Jp, num_p)
        assert np.allclose(Jp, -A[:, 0:3], rtol=0, atol=1e-12 * np.abs(Jp).max())   # d/dp = -d/dr


def test_zero_correction_for_a_perfect_observation():
    x, P = camera_state(), camera_cov()
    pts = np.array([world_point(x, pixel_ray(uv, 3.0)) for uv in ((80, 60), (240, 70), (150, 180))])
    uv = np.array([LO.predict(x, p, CAM) for p in pts])
    res = LO.landmark_update(x, P, CAM, pts, uv, np.ones(3, np.uint8), 3, std_px=1.0, gate=5.9915)
    assert res["status"] == LO.LMU_APPLIED and res["k"] == 6 and (res["lm_status"] == LO.LM_USED).all()
    assert res["nis"] == 0.0 and (res["lm_nis"] == 0.0).all()
    xe = x.copy()
    xe[3:7] = x[3:7] / np.linalg.norm(x[3:7])
    assert np.array_equal(res["x"], xe)
    assert (np.diag(res["P"])[0:3] < np.diag(P)[0:3]).all()


def test_statuses_of_unusable_landmarks():
    x, P = camera_state(), camera_cov()
    hrl = [(0.2, 0.1, 3.0),                       # used
           (0.2, 0.1, -3.0),                      # behind the camera
           (math.tan(math.radians(70)), 0, 1),    # outside the +-60 deg cone
           (0.0, 1.0, 1.0),                       # inside the cone (45 deg), outside the image
           (-0.3, 0.2, 2.0),                      # not observed
           (0.1, -0.2, 2.5),                      # gross outlier, gated out
           (0.0, 0.0, 4.0)]                       # absent (j >= nlm)
    pts = np.array([world_point(x, v) for v in hrl])
    uv = np.full((7, 2), 100.0)
    for j in (0, 4, 5):
        uv[j] = LO.predict(x, pts[j], CAM)
    uv[5] += 40.0
    has = np.ones(7, np.uint8)
    has[4] = 0
    res = LO.landmark_update(x, P, CAM, pts, uv, has, 6, std_px=1.0, gate=5.9915)
    exp = [LO.LM_USED, LO.LM_NOT_VISIBLE, LO.LM_NOT_VISIBLE, LO.LM_NOT_VISIBLE, LO.LM_NOT_OBSERVED, LO.LM_GATED,
           LO.LM_ABSENT]
    assert list(res["lm_status"]) == exp
    assert res["k"] == 2 and res["status"] == LO.LMU_APPLIED
    assert np.isnan(res["lm_h"][[1, 2, 3, 4, 6]]).all() and np.isfinite(res["lm_h"][[0, 5]]).all()
    assert res["lm_nis"][5] > 5.9915 and np.isnan(res["lm_nis"][[1, 2, 3, 4, 6]]).all()
    # nothing usable: the state comes back unchanged
    none = LO.landmark_update(x, P, CAM, pts[1:4], uv[1:4], has[1:4], 3, std_px=1.0)
    assert none["status"] == LO.LMU_NONE and none["k"] == 0 and np.isnan(none["nis"])
    assert np.array_equal(none["x"], x) and np.array_equal(none["P"], P)
    # a zero covariance with no pixel noise: S_j = 0 is not SPD
    zero = LO.landmark_update(x, np.zeros((13, 13)), CAM, pts[:1], uv[:1], has[:1], 1, std_px=0.0)
    assert zero["lm_status"][0] == LO.LM_NOT_SPD and zero["status"] == LO.LMU_NONE


def nis_samples(n, seed, std_px=1.0):
    """Mean NIS and mean k of the mirror over n truths drawn from the filter's own (r, q) covariance, landmark
    positions drawn from their C_j, and pixel noise std_px."""
    rng = np.random.RandomState(seed)
    x, P = camera_state(), camera_cov()
    pts = np.array([world_point(x, pixel_ray(uv, d)) for uv, d in (((70, 60), 2.5), ((250, 80), 3.0),
                                                                     ((120, 190), 2.0), ((230, 170), 4.0))])
    cov = np.zeros((4, 6))
    cov[1] = [0.02 ** 2, 0, 0.02 ** 2, 0, 0, 0.03 ** 2]
    cov[3] = [0.03 ** 2, 0.0002, 0.02 ** 2, 0.0001, 0.0, 0.04 ** 2]
    Lc = [np.linalg.cholesky(LO.unpack_cov(c)) if c.any() else np.zeros((3, 3)) for c in cov]
    Lp = np.linalg.cholesky(P[0:7, 0:7])
    has = np.ones(4, np.uint8)
    tot_nis = tot_k = 0.0
    for _ in range(n):
        xt = x.copy()
        xt[0:7] += Lp @ rng.standard_normal(7)
        uv = np.array([LO.predict(xt, pts[j] + Lc[j] @ rng.standard_normal(3), CAM) for j in range(4)])
        uv += std_px * rng.standard_normal((4, 2))
        res = LO.landmark_update(x, P, CAM, pts, uv, has, 4, std_px=std_px, cov=cov)
        assert res["status"] == LO.LMU_APPLIED
        tot_nis += res["nis"]
        tot_k += res["k"]
    return tot_nis / n, tot_k / n


def test_mean_nis_is_k():
    """20000 samples of k = 8: the standard error of the mean NIS is sqrt(2 / (8 * 20000)) = 0.25 % relative, so the
    3 % band is twelve standard errors wide."""
    mean_nis, mean_k = nis_samples(20000, 17)
    assert mean_k == 8.0
    assert abs(mean_nis / mean_k - 1.0) < 0.03, mean_nis


def test_understated_noise_is_detected():
    """The yardstick has power: the same samples drawn with 3 px noise but updated with 1 px give a mean NIS far
    above k."""
    rng = np.random.RandomState(4)
    x, P = camera_state(), camera_cov()
    pts = np.array([world_point(x, pixel_ray(uv, 3.0)) for uv in ((70, 60), (250, 80))])
    tot = 0.0
    for _ in range(300):
        uv = np.array([LO.predict(x, p, CAM) for p in pts]) + 3.0 * rng.standard_normal((2, 2))
        tot += LO.landmark_update(x, P, CAM, pts, uv, np.ones(2, np.uint8), 2, std_px=1.0)["nis"]
    assert tot / 300 > 2.0 * 4


def test_synthetic_landmark_obs_definition():
    B, M, L, T = 96, 300, 16, 6
    world = synth.SynthWorld(B=B, M=M, T=T, seed=9, p_outlier=0.2, p_flaky=0.8, flaky_mod=7, noise_px=0.5, gross_px=8.0)
    rng = np.random.RandomState(2)
    tags = rng.randint(-1, M + 3, (B, L)).astype(np.int32)          # some -1 and some >= M: no world point
    nlm = rng.randint(0, L + 1, B).astype(np.int32)
    n_out = n_exp = n_obs = 0.0
    res_in = []
    for t in range(T + 1):
        uv, has = world.landmark_obs(t, tags, nlm)
        zt, vis = world.truth_pixels(t)
        for b in range(B):
            for j in range(L):
                w = int(tags[b, j])
                ok = j < nlm[b] and 0 <= w < M and bool(vis[b, w])
                assert bool(has[b, j]) == ok, (t, b, j)
                if not ok:
                    assert (uv[b, j] == 0.0).all()
                    continue
                n_obs += 1
                p_out = world.p_flaky if w % 7 == 6 else world.p_outlier
                n_exp += p_out
                u8 = synth.world_uniform(world.seed, b, t, w, 8)
                d = uv[b, j] - zt[b, w]
                if u8 < p_out:
                    n_out += 1
                    assert (np.abs(d) <= world.gross_px).all()
                else:
                    res_in.append(d)
        # landmark noise is drawn on its own channels: never the candidate's noise of the same point
        zc, hc = world.candidates(t, tags.clip(0, M - 1), np.full(B, L))
        both = (has == 1) & (hc == 1) & (tags >= 0) & (tags < M)
        assert not (uv[both] == zc[both]).all(axis=1).any()
    res_in = np.array(res_in)
    assert n_obs > 1500
    sd = math.sqrt(n_exp * (1 - n_exp / n_obs))
    assert abs(n_out - n_exp) < 4 * sd, (n_out, n_exp)
    assert abs(res_in.std() / world.noise_px - 1.0) < 0.05 and abs(res_in.mean()) < 0.05
