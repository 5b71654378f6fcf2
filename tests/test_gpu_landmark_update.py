"""The known-landmark update (ekfslam_update_landmarks) on the device against its numpy mirror
(oracle/landmark_oracle.py) for one call: 1 to 16 landmarks (k = 2 .. 32), ragged landmark counts and ragged maps, both
`which`, landmarks behind the camera / outside the cone / outside the image / not observed, gross outliers under the
gate, exact and uncertain landmark positions, L = N_max at a small N_max.  Then the untouched-filter rules, batch
independence, determinism, the error codes, the device footprint, the launched kernels, the synthetic observations
against SynthWorld.landmark_obs, the NIS statistics at B = 4096 and a closed-loop diagnostic."""
import ctypes as C

import numpy as np
import pytest

from oracle import ekf_oracle as O
from oracle import landmark_oracle as LO
from tests.test_landmark_oracle import camera_state, pixel_ray, world_point

pytestmark = pytest.mark.gpu
TOL = 1e-9
CAM = O.initialize_cam()
GATE = 5.9915


@pytest.fixture(scope="module")
def pkg():
    import ekf_slam_b200 as pkg
    return pkg


def _state(B, N, seed, nfeat):
    """Host-built maps of SynthSequence, filter b keeping its first nfeat[b] inverse-depth features, a rotated and
    displaced camera and a camera block of P widened to (1 cm, 0.002)^2 so that landmarks move the pose."""
    import ekf_slam_b200.synth as synth
    seq = synth.SynthSequence(B=B, N=N, T=1, seed=seed)
    x, P, types = seq.initial_state()
    ns = 13 + 6 * np.asarray(nfeat)
    for b in range(B):
        n = ns[b]
        types[b, nfeat[b]:] = 0
        x[b, n:] = 0.0
        P[b, n:, :] = 0.0
        P[b, :, n:] = 0.0
    x[:, 0:13] = camera_state()
    P[:, 0:3, 0:3] += 1e-4 * np.eye(3)
    P[:, 3:7, 3:7] += 4e-6 * np.eye(4)
    return x, P, types, ns.astype(np.int32)


def _bank(pkg, B, N, x, P, types, ns):
    bank = pkg.FilterBank(B, N)
    bank.upload_feature_types(types)
    bank.upload_state(x, P, ns)
    bank.upload_state(x, nstate=ns, which=1)
    return bank


KINDS = ("ok", "behind", "cone", "image", "unobserved", "outlier")


def _landmarks(rng, x, L, nlm, kinds=False, cov=False, sigma=1.0):
    """pts [B,L,3], cov [B,L,6] or None, uv [B,L,2], has [B,L]: landmarks in front of each filter's camera seen from
    a perturbed true pose with pixel noise sigma; with kinds, slots also take the unusable kinds of KINDS."""
    B = len(x)
    pts, uv = np.zeros((B, L, 3)), np.zeros((B, L, 2))
    has = np.ones((B, L), dtype=np.uint8)
    C6 = np.zeros((B, L, 6)) if cov else None
    for b in range(B):
        xt = x[b, :13].copy()
        xt[0:3] += 0.005 * rng.standard_normal(3)
        xt[3:7] += 0.001 * rng.standard_normal(4)
        xt[3:7] /= np.linalg.norm(xt[3:7])
        for j in range(L):
            kind = rng.choice(KINDS, p=[0.5, 0.1, 0.1, 0.1, 0.1, 0.1]) if kinds else "ok"
            ray = pixel_ray((rng.uniform(30, 290), rng.uniform(30, 210)), rng.uniform(1.5, 6.0))
            if kind == "behind":
                ray = -ray
            elif kind == "cone":
                ray = np.array([2.9, 0.1, 1.0]) * rng.uniform(1, 3)
            elif kind == "image":
                ray = np.array([0.0, 1.0, 1.0]) * rng.uniform(1, 3)
            pts[b, j] = world_point(x[b], ray)
            if cov and rng.rand() < 0.5:
                s = rng.uniform(0.005, 0.03, 3)
                A = rng.standard_normal((3, 3)) * 0.3 + np.eye(3)
                Cj = (A * s) @ (A * s).T
                C6[b, j] = Cj[[0, 1, 1, 2, 2, 2], [0, 0, 1, 0, 1, 2]]
            h = LO.predict(xt, pts[b, j], CAM)
            uv[b, j] = (h if h is not None else np.array([100.0, 100.0])) + sigma * rng.standard_normal(2)
            if kind == "outlier":
                uv[b, j] += 40.0
            if kind == "unobserved":
                has[b, j] = 0
    return pts, C6, uv, has


def _snapshot(bank):
    x, P, ns = bank.download_state()
    xp, _, _ = bank.download_state(which=1, want_P=False)
    return dict(x=x, xp=xp, P=P, ns=ns, stats=np.stack(list(bank.download_stats().values()), axis=1),
                tags=bank.download_feature_tags(), types=bank.download_feature_types()[0], **bank.download_features())


def _scaled(a, b, d):
    """max |a - b| scaled by the prior: |dx_i| / sqrt(P_ii) for vectors, |dP_ij| / sqrt(P_ii P_jj) for matrices."""
    e = np.abs(a - b)
    return float(np.max(e / d if e.ndim == 1 else e / np.outer(d, d)))


def _run_case(pkg, B, N, L, nlm, nfeat, which, seed, kinds, cov, gate):
    rng = np.random.RandomState(seed)
    x, P, types, ns = _state(B, N, seed, nfeat)
    bank = _bank(pkg, B, N, x, P, types, ns)
    pts, C6, uv, has = _landmarks(rng, x, L, nlm, kinds=kinds, cov=cov)
    before = _snapshot(bank)
    bank.upload_landmarks(pts, C6, nlm=nlm)
    bank.upload_landmark_obs(uv, has)
    bank.update_landmarks(1.0, gate=gate, which=which)
    res = bank.download_landmark_update()
    after = _snapshot(bank)
    other = "x" if which else "xp"
    for k in before:
        if k not in ("x", "xp", "P"):
            assert np.array_equal(before[k].view(np.uint8), after[k].view(np.uint8)), k
    assert np.array_equal(before[other].view(np.uint8), after[other].view(np.uint8))
    xs = "xp" if which else "x"
    worst = dict(x=0.0, P=0.0, h=0.0, nis=0.0)
    for b in range(B):
        n = int(ns[b])
        xin = before[xs][b, :n]
        m = LO.landmark_update(xin, before["P"][b, :n, :n], CAM, pts[b], uv[b], has[b], nlm[b], 1.0, gate,
                               None if C6 is None else C6[b])
        ctx = (B, N, L, which, b)
        assert np.array_equal(res["lm_status"][b], m["lm_status"]), (ctx, res["lm_status"][b], m["lm_status"])
        assert res["status"][b] == m["status"] and res["k"][b] == m["k"], (ctx, res["status"][b], m["status"])
        assert np.array_equal(np.isnan(res["lm_h"][b]), np.isnan(m["lm_h"])), ctx
        assert np.array_equal(np.isnan(res["lm_nis"][b]), np.isnan(m["lm_nis"])), ctx
        f = ~np.isnan(m["lm_h"])
        if f.any():
            worst["h"] = max(worst["h"], float(np.max(np.abs(res["lm_h"][b][f] - m["lm_h"][f]) / np.abs(m["lm_h"][f]))))
        f = ~np.isnan(m["lm_nis"])
        if f.any():
            # relative to max(NIS, 1): a small NIS comes from a small nu = uv - h, whose last bits cancel
            worst["nis"] = max(worst["nis"], float(np.max(np.abs(res["lm_nis"][b][f] - m["lm_nis"][f])
                                                          / np.maximum(m["lm_nis"][f], 1.0))))
        Pg = after["P"][b]
        assert np.array_equal(Pg, Pg.T), ctx
        assert not Pg[n:].any() and not Pg[:, n:].any() and not after[xs][b, n:].any(), ctx
        if m["status"] != LO.LMU_APPLIED:
            assert np.isnan(res["nis"][b])
            for k in (xs, "P"):
                assert np.array_equal(before[k][b].view(np.uint8), after[k][b].view(np.uint8)), (ctx, k)
            continue
        d = np.sqrt(np.diag(before["P"][b, :n, :n]))
        worst["x"] = max(worst["x"], _scaled(after[xs][b, :n], m["x"], d))
        worst["P"] = max(worst["P"], _scaled(Pg[:n, :n], m["P"], d))
        assert abs(res["nis"][b] - m["nis"]) <= 1e-9 * m["nis"], ctx
    bank.close()
    assert worst["x"] < TOL and worst["P"] < TOL and worst["h"] < 1e-12 and worst["nis"] < 1e-12, worst
    return worst, res


def test_parity_k_2_to_32(pkg):
    """Every filter sees all of its nlm[b] landmarks: k = 2 nlm[b] for nlm = 1 .. 16, both which, ragged maps."""
    B, N, L = 48, 100, 16
    rng = np.random.RandomState(1)
    nlm = np.arange(B) % L + 1
    nfeat = rng.randint(0, N + 1, B)
    nfeat[:4] = [0, 8, 9, 100]            # n = 13, 61, 67, 613: both sides of the 64-column tile edge
    for which in (0, 1):
        w, res = _run_case(pkg, B, N, L, nlm, nfeat, which, 10 + which, kinds=False, cov=False, gate=0.0)
        assert np.array_equal(res["k"], 2 * nlm) and (res["status"] == 0).all()
        print("landmark parity k=2..32 which=%d: scaled err x %.2e P %.2e, rel h %.2e nis %.2e"
              % (which, w["x"], w["P"], w["h"], w["nis"]))


def test_parity_mixed_landmarks(pkg):
    """Ragged nlm (0 .. 16), every unusable kind, gross outliers under the gate, half the landmarks uncertain."""
    B, N, L = 64, 100, 16
    rng = np.random.RandomState(2)
    nlm = rng.randint(0, L + 1, B)
    nlm[:3] = [0, 16, 1]
    nfeat = rng.randint(0, N + 1, B)
    seen = set()
    for which in (0, 1):
        for cov in (False, True):
            w, res = _run_case(pkg, B, N, L, nlm, nfeat, which, 20 + 2 * which + cov, kinds=True, cov=cov, gate=GATE)
            seen |= set(np.unique(res["lm_status"]).tolist())
            print("landmark parity mixed which=%d cov=%d: scaled err x %.2e P %.2e, rel h %.2e nis %.2e"
                  % (which, cov, w["x"], w["P"], w["h"], w["nis"]))
    assert {LO.LM_USED, LO.LM_NOT_OBSERVED, LO.LM_NOT_VISIBLE, LO.LM_GATED, LO.LM_ABSENT} <= seen, seen


def test_parity_L_equals_N_max(pkg):
    B, N = 16, 4
    nlm = np.arange(B) % (N + 1)
    nfeat = np.arange(B) % (N + 1)
    for which in (0, 1):
        _run_case(pkg, B, N, N, nlm, nfeat, which, 30 + which, kinds=True, cov=True, gate=GATE)


def test_untouched_filters_and_independence(pkg):
    """Filters with nothing used (no landmark, none observed, none visible, all gated) keep every byte; a filter's
    result is the same in a batch of 32 and alone in a batch of 4; two runs are bit-identical."""
    B, N, L = 32, 40, 6
    rng = np.random.RandomState(5)
    nfeat = rng.randint(0, N + 1, B)
    x, P, types, ns = _state(B, N, 6, nfeat)
    pts, _, uv, has = _landmarks(rng, x, L, None)
    nlm = np.full(B, L)
    nlm[3] = 0                                              # no landmark
    has[7] = 0                                              # none observed
    pts[11] = [world_point(x[11], (0.1, 0.1, -2.0))] * L    # all behind the camera
    uv[15] += 50.0                                          # all gated out
    outs = []
    for _ in range(2):
        bank = _bank(pkg, B, N, x, P, types, ns)
        bank.ekf_prediction()
        before = _snapshot(bank)
        bank.upload_landmarks(pts, nlm=nlm)
        bank.upload_landmark_obs(uv, has)
        bank.update_landmarks(1.0, gate=GATE)
        res = bank.download_landmark_update()
        after = _snapshot(bank)
        for b in (3, 7, 11, 15):
            assert res["status"][b] == pkg.LMU_NONE and res["k"][b] == 0, (b, res["status"][b])
            for k in before:
                assert np.array_equal(np.atleast_1d(before[k][b]).view(np.uint8),
                                      np.atleast_1d(after[k][b]).view(np.uint8)), (b, k)
        assert (np.delete(res["status"], [3, 7, 11, 15]) == pkg.LMU_APPLIED).all()
        outs.append((after["x"], after["P"], res["nis"], res["lm_h"], res["lm_nis"]))
        bank.close()
    for a, b in zip(*outs):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    sl = slice(12, 16)
    bank = _bank(pkg, 4, N, x[sl], P[sl], types[sl], ns[sl])
    bank.ekf_prediction()
    bank.upload_landmarks(pts[sl], nlm=nlm[sl])
    bank.upload_landmark_obs(uv[sl], has[sl])
    bank.update_landmarks(1.0, gate=GATE)
    xs, Ps, _ = bank.download_state()
    assert np.array_equal(xs.view(np.uint8), outs[0][0][sl].view(np.uint8))
    assert np.array_equal(Ps.view(np.uint8), outs[0][1][sl].view(np.uint8))
    bank.close()


def test_errors_and_footprint(pkg):
    bank = pkg.FilterBank(4, 3)
    lib, h = bank.lib, bank._h
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    bytes0 = bank.device_bytes
    pts, uv = np.zeros((4, 3, 3)), np.zeros((4, 3, 2))
    nis = np.empty(4)
    assert lib.ekfslam_download_landmark_update(h, 0, 4, ptr(nis), None, None, None, None, None) == -4
    assert lib.ekfslam_update_landmarks(h, 1.0, 0.0, 0) == -4
    assert lib.ekfslam_upload_landmark_obs(h, 0, 4, ptr(uv), None) == -4
    for L in (0, 4, 17):                                   # L outside [1, min(16, N_max)]
        assert lib.ekfslam_upload_landmarks(h, 0, 4, L, ptr(np.zeros((4, 17, 3))), None, None, None) == -1
    for b0, nb in ((-1, 2), (0, 0), (3, 2)):
        assert lib.ekfslam_upload_landmarks(h, b0, nb, 3, ptr(pts), None, None, None) == -1
    assert lib.ekfslam_upload_landmarks(h, 0, 4, 3, None, None, None, None) == -1
    bad = np.array([0, 1, 4, 2], dtype=np.int32)           # nlm outside [0, L]
    assert lib.ekfslam_upload_landmarks(h, 0, 4, 3, ptr(pts), None, None, ptr(bad)) == -1
    assert bank.device_bytes == bytes0                     # nothing allocated until the first landmark upload
    bank.reset_filters()
    bytes0 = bank.device_bytes
    bank.upload_landmarks(np.tile(world_point(camera_state(0, (1, 0, 0, 0)), (0, 0, 3.0)), (4, 3, 1)))
    assert bank.device_bytes > bytes0
    assert lib.ekfslam_update_landmarks(h, 1.0, 0.0, 0) == -4          # no observations yet
    assert lib.ekfslam_world_landmark_obs(h, 0) == -4                  # no world
    assert lib.ekfslam_upload_landmark_obs(h, 0, 4, None, None) == -1
    assert lib.ekfslam_upload_landmark_obs(h, 2, 3, ptr(uv), None) == -1
    bank.upload_landmark_obs(np.full((4, 3, 2), 100.0))
    for args in ((-1.0, 0.0, 0), (float("nan"), 0.0, 0), (float("inf"), 0.0, 0), (1.0, 0.0, 2)):
        assert lib.ekfslam_update_landmarks(h, *args) == -1, args
    assert lib.ekfslam_download_landmark_update(h, 0, 4, ptr(nis), None, None, None, None, None) == -4
    bank.update_landmarks(1.0)
    res = bank.download_landmark_update()
    assert (res["status"] == pkg.LMU_APPLIED).all() and (res["k"] == 6).all()
    assert lib.ekfslam_download_landmark_update(h, 3, 2, ptr(nis), None, None, None, None, None) == -1
    import ekf_slam_b200.synth as synth
    world = synth.SynthWorld(4, M=10, T=2, seed=1)
    bank.world_upload(world)
    assert lib.ekfslam_world_landmark_obs(h, 3) == -1                  # t outside [0, T]
    bank.close()


def test_profiler_kernels(pkg):
    """Every update launches k_lm_update and then the short-K downdate k_downdate_ws2<2,2>.  Three updates are
    profiled after a warm-up one; the activity records of a profiling session are not guaranteed to hold a kernel
    launched right as the session starts (the session is given a moment before the first launch, and the first
    update's k_lm_update may still be missing from them)."""
    import time
    from torch.profiler import ProfilerActivity, profile
    B, N, L = 8, 20, 4
    rng = np.random.RandomState(8)
    x, P, types, ns = _state(B, N, 8, np.full(B, N))
    bank = _bank(pkg, B, N, x, P, types, ns)
    pts, _, uv, has = _landmarks(rng, x, L, None)
    bank.upload_landmarks(pts)
    bank.upload_landmark_obs(uv, has)
    bank.update_landmarks(1.0)
    bank.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        time.sleep(0.2)
        for _ in range(3):
            bank.update_landmarks(1.0)
        bank.synchronize()
    assert (bank.download_landmark_update()["status"] == pkg.LMU_APPLIED).all()
    names = [e.name.replace(" ", "") for e in sorted(prof.events(), key=lambda e: e.time_range.start)
             if "k_" in e.name]
    upd = [i for i, k in enumerate(names) if "k_lm_update" in k]
    assert len(upd) >= 2, names
    assert all(i + 1 < len(names) and "k_downdate_ws2<2,2>" in names[i + 1] for i in upd), names
    assert all("k_lm_update" in k or "k_downdate_ws2<2,2>" in k for k in names), names
    bank.close()


def test_world_landmark_obs_matches_synth(pkg):
    import ekf_slam_b200.synth as synth
    B, M, L, T = 32, 120, 16, 4
    world = synth.SynthWorld(B, M=M, T=T, seed=7, p_outlier=0.3)
    rng = np.random.RandomState(3)
    tags = rng.randint(-1, M + 2, (B, L)).astype(np.int32)
    nlm = rng.randint(0, L + 1, B).astype(np.int32)
    bank = pkg.FilterBank(B, 20)
    bank.world_upload(world)
    bank.upload_landmarks(np.zeros((B, L, 3)), tag=tags, nlm=nlm)
    worst = 0.0
    for t in range(T + 1):
        bank.world_landmark_obs(t)
        uv_m, has_m = world.landmark_obs(t, tags, nlm)
        uv, has = bank.download_landmark_obs()
        assert np.array_equal(has, has_m), t
        assert not uv[has == 0].any()
        worst = max(worst, float(np.abs(uv - uv_m).max()))
    print("world landmark observations vs SynthWorld.landmark_obs: has identical, worst |duv| %.3e px" % worst)
    assert worst < 1e-9
    bank.close()


def test_consistency_on_device():
    """B = 4096 camera-only filters with the (1 cm, 0.002)^2 camera covariance of tests/test_landmark_oracle.py, each
    with a static truth drawn from it and four exactly known landmarks; 20 frames of fresh 1 px observations, one
    update per frame.  Mean NIS within 3 % of the mean k = 8 (standard error 0.06 %)."""
    import ekf_slam_b200 as pkg
    import ekf_slam_b200.synth as synth
    from tests.test_landmark_oracle import camera_cov
    B, frames, L, sigma = 4096, 20, 4, 1.0
    rng = np.random.RandomState(41)
    x0, P0 = camera_state(), camera_cov()
    pts = np.array([world_point(x0, pixel_ray(uv, d)) for uv, d in (((70, 60), 2.5), ((250, 80), 3.0),
                                                                      ((120, 190), 2.0), ((230, 170), 4.0))])
    xt = np.tile(x0, (B, 1))
    xt[:, 0:7] += rng.standard_normal((B, 7)) @ np.linalg.cholesky(P0[0:7, 0:7]).T
    cam = synth.default_camera()
    zt, dep = synth.project(np.tile(pts, (B, 1, 1)), xt[:, 0:3], xt[:, 3:7], cam)
    assert (dep > 0).all()
    bank = pkg.FilterBank(B, 4)
    bank.reset_filters(xv=x0, Pxv=P0)
    bank.upload_landmarks(np.tile(pts, (B, 1, 1)))
    nis, ks = [], []
    for _ in range(frames):
        bank.upload_landmark_obs(zt + sigma * rng.standard_normal((B, L, 2)))
        bank.update_landmarks(sigma, which=0)
        res = bank.download_landmark_update()
        assert (res["status"] == pkg.LMU_APPLIED).all()
        nis.append(res["nis"])
        ks.append(res["k"])
    mean_nis, mean_k = float(np.mean(nis)), float(np.mean(ks))
    print("device landmark consistency: mean NIS %.4f, mean k %.2f" % (mean_nis, mean_k))
    assert abs(mean_nis / mean_k - 1.0) < 0.03, (mean_nis, mean_k)
    bank.close()


def _best_landmarks(world, frames, n=6):
    """Per filter the n world points (not flaky) visible in the most of frames 1..frames."""
    seen = np.zeros((world.B, world.M), dtype=np.int64)
    for t in range(1, frames + 1):
        seen += world.truth_pixels(t)[1]
    seen[:, np.arange(world.M) % world.flaky_mod == world.flaky_mod - 1] = -1
    return np.argsort(-seen, axis=1, kind="stable")[:, :n].astype(np.int32)


def test_closed_loop_diagnostic(pkg):
    """The 50-frame closed loop of test_gpu_eval with the device world: after every step an update with 6 tagged
    landmarks at their true positions, observed through ekfslam_world_landmark_obs (0.5 px pixel noise and the world's
    20 % of +-8 px outliers), fused with std_px = 1 (the filter's own pixel noise) and no gate.  The monocular filter
    starts with an exactly known pose and a 2.5 cm/frame velocity prior against a 5-8 cm/frame truth, so its first
    predictions are overconfident and the 5.9915 gate would reject most of the landmarks (1.4 of 6 used on average in
    the same run).  The camera-position and map errors are scored with ekfslam_evaluate after the step and before that
    frame's update.  Measured (seeded): camera-position RMSE 0.442 unaided, 0.025 aided; map RMSE 1.51 and 1.01."""
    from tests.test_gpu_eval import _closed_loop, _world
    frames = 50
    world = _world(4, frames)
    tags = _best_landmarks(world, frames)
    pts = world.points[np.arange(4)[:, None], tags]
    rmse = {}
    for aided in (False, True):
        pos, mp = [], []

        def on_frame(bank, t):
            bank.evaluate(t)
            rec = bank.download_eval(features=False)
            pos.append(rec["pos_sq_err"])
            mp.append(rec["map_sq_err"] / np.maximum(rec["n_map"], 1))
            if aided:
                if t == 1:
                    bank.upload_landmarks(pts, tag=tags)
                bank.world_landmark_obs(t)
                bank.update_landmarks(1.0, which=0)
                assert (bank.download_landmark_update()["status"] == pkg.LMU_APPLIED).all()

        _closed_loop(pkg, world, frames, on_frame).close()
        pos, mp = np.array(pos), np.array(mp)
        h = frames // 2
        rmse[aided] = (float(np.sqrt(pos[h:].mean())), float(np.sqrt(mp[h:].mean())))
    print("closed loop, last 25 of 50 frames: camera-position RMSE unaided %.4f aided %.4f; map RMSE unaided %.4f "
          "aided %.4f" % (rmse[False][0], rmse[True][0], rmse[False][1], rmse[True][1]))
    assert rmse[True][0] < 0.25 * rmse[False][0] and rmse[True][1] < 0.9 * rmse[False][1], rmse
