"""The camera-state measurement update (ekfslam_update_camera) on the device: parity with oracle.update for one call and
inside the visual step in both call orders, the untouched-filter rules, the tile-downdate fallback of a large map,
the NIS / NEES consistency of the device filter at B=4096, determinism, the error codes, and a closed-loop diagnostic."""
import ctypes as C

import numpy as np
import pytest

from oracle import ekf_oracle as O
from tests import helpers as T
from tests.test_cam_update_oracle import draw_truth, fix_model, initial_camera, truth_step

pytestmark = pytest.mark.gpu
TOL = 1e-9


@pytest.fixture(scope="module")
def pkg():
    import ekf_slam_b200 as pkg
    return pkg


def _full_H(H, n):
    Hf = np.zeros((H.shape[0], n))
    Hf[:, :13] = H
    return Hf


def _oracle(x, P, H, R, z):
    """oracle.update with [H | 0] and the NIS nu' inv(S) nu."""
    Hf = _full_H(H, len(x))
    nu = z - Hf @ x
    S = Hf @ P @ Hf.T + R
    xo, Po, _ = O.update(x, P, Hf, R, z, Hf @ x)
    return xo, Po, float(nu @ np.linalg.solve(S, nu))


def _cases(rng, nb):
    """(name, H [m,13] or [nb,m,13], R [m,m] or [nb,m,m]) for m in 1, 3, 6, 13."""
    H1 = np.zeros((1, 13)); H1[0, 7] = 1.0                         # forward speed
    H3, R3 = fix_model(3)
    H6, R6 = fix_model(6)
    H13 = rng.standard_normal((nb, 13, 13))
    A = rng.standard_normal((nb, 13, 13)) * 0.1
    R13 = A @ np.transpose(A, (0, 2, 1)) + 0.01 * np.eye(13)
    return [("m1", H1, np.array([[0.02 ** 2]])), ("m3", H3, R3), ("m6", H6, R6), ("m13", H13, R13)]


def _bench_maps(pkg, B, N, seed, nfeat):
    """Maps built on the device as bench.py builds them, filter b keeping its first nfeat[b] features."""
    import ekf_slam_b200.synth as synth
    seq = synth.SynthSequence(B=B, N=N, T=1, seed=seed)
    bank = pkg.FilterBank(B, N)
    bank.reset_filters()
    for k in range(N):
        bank.add_features_inverse_depth(np.ascontiguousarray(seq.zc[0, :, k]), add=(nfeat > k).astype(np.uint8))
    return bank


def _snapshot(bank):
    x, P, ns = bank.download_state()
    xp, _, _ = bank.download_state(which=1, want_P=False)
    d = bank.download_features()
    return dict(x=x, xp=xp, P=P, ns=ns, stats=np.stack(list(bank.download_stats().values())),
                tags=bank.download_feature_tags(), types=bank.download_feature_types()[0], **d)


def _draw_z(rng, H, R, x13):
    """z [nb, m] = H x + v with v ~ N(0, R), per filter."""
    nb = len(x13)
    Hb = np.broadcast_to(H, (nb,) + H.shape[-2:])
    Rb = np.broadcast_to(R, (nb,) + R.shape[-2:])
    m = Hb.shape[1]
    return np.einsum("bij,bj->bi", Hb, x13) + np.einsum("bij,bj->bi", np.linalg.cholesky(Rb), rng.standard_normal((nb, m)))


def test_parity_one_update(pkg):
    B, N = 64, 100
    rng = np.random.RandomState(3)
    nfeat = rng.randint(0, N + 1, B)
    nfeat[[0, 9, 33]] = 0                                         # camera-only filters
    nfeat[1] = N
    worst = dict(x=0.0, P=0.0, nis=0.0)
    for which in (0, 1):
        for name, H, R in _cases(rng, B):
            bank = _bench_maps(pkg, B, N, 77, nfeat)
            if which == 1:
                bank.ekf_prediction()                             # fills x_k_km1
            before = _snapshot(bank)
            xin = before["xp" if which else "x"]
            z = _draw_z(rng, H, R, xin[:, :13])
            bank.update_camera(H, z, R, which=which)
            res = bank.download_camera_update()
            after = _snapshot(bank)
            assert (res["status"] == pkg.CAM_APPLIED).all(), (name, which, res["status"])
            other = "x" if which else "xp"
            for k in before:
                if k not in ("x", "xp", "P"):
                    assert np.array_equal(before[k].view(np.uint8), after[k].view(np.uint8)), (name, which, k)
            assert np.array_equal(before[other].view(np.uint8), after[other].view(np.uint8)), (name, which, other)
            xg, Pg = after["xp" if which else "x"], after["P"]
            for b in range(B):
                n = int(before["ns"][b])
                Hb = H if H.ndim == 2 else H[b]
                Rb = R if R.ndim == 2 else R[b]
                xo, Po, nis = _oracle(xin[b, :n], before["P"][b, :n, :n], Hb, Rb, z[b])
                ex, eP = T.rel_err(xg[b, :n], xo), T.rel_err(Pg[b, :n, :n], Po)
                en = abs(res["nis"][b] - nis) / max(abs(nis), 1e-300)
                worst["x"], worst["P"], worst["nis"] = max(worst["x"], ex), max(worst["P"], eP), max(worst["nis"], en)
                assert ex < TOL and eP < TOL and en < TOL, (name, which, b, ex, eP, en)
                assert np.array_equal(Pg[b], Pg[b].T), (name, which, b)
            bank.close()
    print("camera update parity (B=%d, N=%d, ragged): worst rel err x %.2e, P %.2e, NIS %.2e"
          % (B, N, worst["x"], worst["P"], worst["nis"]))


def test_untouched_filters(pkg):
    B, N = 16, 20
    nfeat = np.full(B, N)
    rng = np.random.RandomState(4)
    bank = _bench_maps(pkg, B, N, 5, nfeat)
    bank.ekf_prediction()
    before = _snapshot(bank)
    H, R = fix_model(3)
    Rb = np.tile(R, (B, 1, 1))
    z = _draw_z(rng, H, R, before["x"][:, :13])
    on = np.ones(B, dtype=np.uint8)
    off, gated, bad = [1, 6], [2, 11], [3, 12]
    on[off] = 0
    z[gated] += 1.0                                               # 20 sigma: NIS in the hundreds
    Rb[bad] = -np.eye(3)                                          # S = H P H' - I is not SPD
    bank.update_camera(H, z, Rb, on=on, gate=50.0, which=0)
    res = bank.download_camera_update()
    after = _snapshot(bank)
    exp = np.zeros(B, dtype=np.int32)
    exp[off], exp[gated], exp[bad] = pkg.CAM_OFF, pkg.CAM_GATED, pkg.CAM_NOT_SPD
    assert np.array_equal(res["status"], exp), res["status"]
    assert np.isnan(res["nis"][off]).all() and np.isnan(res["nis"][bad]).all()
    assert (res["nis"][gated] > 50.0).all() and (res["nis"][exp == 0] <= 50.0).all()
    for b in range(B):
        same = all(np.array_equal(before[k][b].view(np.uint8), after[k][b].view(np.uint8)) for k in ("x", "xp", "P"))
        assert same == (exp[b] != 0), (b, exp[b])
        n = int(before["ns"][b])
        if exp[b] == 0:
            xo, Po, nis = _oracle(before["x"][b, :n], before["P"][b, :n, :n], H, R, z[b])
            assert T.rel_err(after["x"][b, :n], xo) < TOL and T.rel_err(after["P"][b, :n, :n], Po) < TOL
    # filters outside [b0, b0+nb) get status 1 for that call
    bank.update_camera(H, z[4:8], R, b0=4, which=0)
    res = bank.download_camera_update()
    assert (res["status"][4:8] == 0).all() and (np.delete(res["status"], range(4, 8)) == pkg.CAM_OFF).all()
    bank.close()


def _visual_run(pkg, order, frames=10, B=3, N=40, seed=300, n_u=64, sigma=0.02):
    """The N=40 free-running configuration of test_gpu_parity with a position fix every frame, against the oracle."""
    import ekf_slam_b200.synth as synth
    seq = synth.SynthSequence(B=B, N=N, T=frames, seed=seed, p_outlier=0.2, n_u=n_u, noise_px=0.5)
    x0, P0, types = seq.initial_state()
    cam = O.initialize_cam()
    bank = pkg.FilterBank(B, N)
    bank.upload_feature_types(types)
    bank.upload_state(x0, P0)
    filts = [T.oracle_filter(x0[b], P0[b]) for b in range(B)]
    feats = [T.oracle_features(types[b]) for b in range(B)]
    H = np.zeros((3, 13)); H[:, :3] = np.eye(3)
    R = sigma ** 2 * np.eye(3)
    rng = np.random.RandomState(seed + 1)
    worst = dict(x=0.0, P=0.0)
    for t in range(1, frames + 1):
        zc, has = seq.frame(t)
        u = seq.uniforms(t, n_u)
        z = seq.pose_r[:, t] + sigma * rng.standard_normal((B, 3))
        bank.upload_candidates(zc, has)
        bank.upload_uniforms(u)
        if order == "A":
            bank.step(reset=True, match_mode=1)
            bank.update_camera(H, z, R, which=0)
        else:
            bank.begin_frame()
            bank.ekf_prediction()
            bank.update_camera(H, z, R, which=1)
            bank.measure(1)
            bank.gate()
            bank.ransac_hypotheses()
            bank.ekf_update_li_inliers()
            bank.rescue_hi_inliers()
            bank.ekf_update_hi_inliers()
        assert (bank.download_camera_update()["status"] == 0).all()
        xg, Pg, _ = bank.download_state()
        fg = bank.download_flags()
        for b in range(B):
            f, fi = filts[b], O.update_features_info(feats[b])
            if order == "A":
                f, fi = O.filter_step(f, fi, cam, (zc[b], has[b]), u[b])
                f.x_k_k, f.p_k_k, _ = O.update(f.x_k_k, f.p_k_k, _full_H(H, len(f.x_k_k)), R, z[b],
                                               _full_H(H, len(f.x_k_k)) @ f.x_k_k)
            else:
                f, fi = O.ekf_prediction(f, fi)
                f.x_k_km1, f.p_k_km1, _ = O.update(f.x_k_km1, f.p_k_km1, _full_H(H, len(f.x_k_km1)), R, z[b],
                                                   _full_H(H, len(f.x_k_km1)) @ f.x_k_km1)
                fi = O.search_IC_matches(f, fi, cam, (zc[b], has[b]))
                fi = O.ransac_hypotheses(f, fi, cam, u[b])
                f = O.ekf_update_li_inliers(f, fi)
                fi = O.rescue_hi_inliers(f, fi, cam)
                f = O.ekf_update_hi_inliers(f, fi)
            filts[b], feats[b] = f, fi
            mask = T.F_HAS_H | T.F_HAS_Z | T.F_IC | T.F_LI | T.F_HI
            assert np.array_equal(fg[b] & mask, T.oracle_flags(fi, N)), (order, t, b)
            n = len(f.x_k_k)
            ex, eP = T.rel_err(xg[b, :n], f.x_k_k), T.rel_err(Pg[b, :n, :n], f.p_k_k)
            worst["x"], worst["P"] = max(worst["x"], ex), max(worst["P"], eP)
            assert ex < TOL and eP < TOL, (order, t, b, ex, eP)
    bank.close()
    return worst


def test_inside_visual_step_after_step(pkg):
    w = _visual_run(pkg, "A")
    print("order A (step, fix): worst rel err x %.2e P %.2e" % (w["x"], w["P"]))


def test_inside_visual_step_between_predict_and_measure(pkg):
    w = _visual_run(pkg, "B")
    print("order B (predict, fix, measure, ...): worst rel err x %.2e P %.2e" % (w["x"], w["P"]))


def test_large_map_tile_downdate(pkg):
    """N_max = 767 (n_max = 4615 > 4608): the tile table of the short-K downdate no longer fits, so the update's
    downdate runs on k_downdate_tile."""
    import ekf_slam_b200.synth as synth
    from torch.profiler import ProfilerActivity, profile
    B, N = 2, 767
    seq = synth.SynthSequence(B=B, N=N, T=1, seed=720)
    x0, P0, types = seq.initial_state()
    bank = pkg.FilterBank(B, N)
    bank.upload_feature_types(types)
    bank.upload_state(x0, P0)
    x, P, ns = bank.download_state()
    H, R = fix_model(6)
    z = _draw_z(np.random.RandomState(8), H, R, x[:, :13])
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        bank.update_camera(H, z, R, which=0)
        bank.synchronize()
    kernels = {e.name for e in prof.events()}
    assert any("k_downdate_tile" in k for k in kernels), sorted(kernels)
    assert any("k_cam_update" in k for k in kernels), sorted(kernels)
    xg, Pg, _ = bank.download_state()
    nis = bank.download_camera_update()["nis"]
    for b in range(B):
        n = int(ns[b])
        xo, Po, ni = _oracle(x[b, :n], P[b, :n, :n], H, R, z[b])
        assert T.rel_err(xg[b, :n], xo) < TOL and T.rel_err(Pg[b, :n, :n], Po) < TOL, b
        assert abs(nis[b] - ni) <= TOL * abs(ni)
        assert np.array_equal(Pg[b], Pg[b].T)
    bank.close()


def test_consistency_on_device(pkg):
    """The scenario of tests/test_cam_update_oracle.py at B=4096 camera-only filters, 20 frames of predict and a fix
    (which=1, then the li update with no features carries x_k_km1 into x_k_k).  Mean NIS within 3 % of m (standard
    error 0.29 % / 0.20 % for m = 3 / 6), and for m = 3 the mean posterior position NEES of ekfslam_evaluate within 3 %
    of 3."""
    from types import SimpleNamespace
    B, frames = 4096, 20
    x0, P0 = initial_camera()
    for m, seed in ((3, 21), (6, 22)):
        rng = np.random.RandomState(seed)
        H, R = fix_model(m)
        xt = draw_truth(rng, x0, P0, B)
        pose_r = np.zeros((B, frames + 1, 3))
        pose_q = np.zeros((B, frames + 1, 4)); pose_q[..., 0] = 1.0
        zs = []
        for t in range(1, frames + 1):
            truth_step(rng, xt)
            pose_r[:, t] = xt[:, 0:3]
            zs.append(_draw_z(rng, H, R, xt))
        world = SimpleNamespace(points=np.zeros((B, 1, 3)), pose_r=pose_r, pose_q=pose_q, M=1, T=frames, seed=0,
                                b_offset=0, flaky_mod=1, noise_px=0.0, gross_px=0.0, p_outlier=0.0, p_flaky=0.0, BAND=22)
        bank = pkg.FilterBank(B, 4)                               # 2 N_max = 8 >= m rows of W; no feature is added
        bank.reset_filters(xv=x0, Pxv=P0)
        bank.world_upload(world)
        nis = []
        for t in range(1, frames + 1):
            bank.ekf_prediction()
            bank.update_camera(H, zs[t - 1], R, which=1)
            bank.ekf_update_li_inliers()
            bank.evaluate(t)
            res = bank.download_camera_update()
            assert (res["status"] == 0).all()
            nis.append(res["nis"])
        mean_nis = float(np.mean(nis))
        tot = bank.download_eval(totals=True)
        mean_nees = float(tot["nees_pos"].sum() / tot["frames"].sum())
        print("device consistency m=%d: mean NIS %.4f (m=%d), mean position NEES %.4f (3)" % (m, mean_nis, m, mean_nees))
        assert abs(mean_nis / m - 1.0) < 0.03, (m, mean_nis)
        if m == 3:
            assert abs(mean_nees / 3.0 - 1.0) < 0.03, mean_nees
        bank.close()


def test_determinism(pkg):
    B, N = 64, 100
    nfeat = np.random.RandomState(6).randint(0, N + 1, B)
    outs = []
    for _ in range(2):
        rng = np.random.RandomState(9)
        _, H, R = _cases(rng, B)[3]
        bank = _bench_maps(pkg, B, N, 77, nfeat)
        x, _, _ = bank.download_state(want_P=False)
        bank.update_camera(H, _draw_z(rng, H, R, x[:, :13]), R, which=0)
        xg, Pg, _ = bank.download_state()
        outs.append((xg, Pg, bank.download_camera_update()["nis"]))
        bank.close()
    for a, b in zip(outs[0], outs[1]):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))


def test_errors(pkg):
    bank = pkg.FilterBank(4, 2)                                   # 2 N_max = 4 rows of W
    lib, h = bank.lib, bank._h
    P = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    bytes0 = bank.device_bytes
    nis, st = np.empty(4), np.empty(4, dtype=np.int32)
    assert lib.ekfslam_download_camera_update(h, 0, 4, P(nis), P(st)) == -4     # ERR_STATE before the first call
    Hm, zm, Rm = np.zeros((4, 13, 13)), np.zeros((4, 13)), np.tile(np.eye(13), (4, 1, 1))
    for m in (0, 5, 14):                                          # m outside [1, min(13, 2 N_max)]
        assert lib.ekfslam_update_camera(h, 0, 4, m, P(Hm), P(zm), P(Rm), None, 0.0, 0) == -1
    assert lib.ekfslam_update_camera(h, 0, 4, 3, P(Hm), P(zm), P(Rm), None, 0.0, 2) == -1      # which
    for b0, nb in ((-1, 2), (0, 0), (3, 2)):                      # bad [b0, b0+nb)
        assert lib.ekfslam_update_camera(h, b0, nb, 3, P(Hm), P(zm), P(Rm), None, 0.0, 0) == -1
    assert lib.ekfslam_update_camera(h, 0, 4, 3, None, P(zm), P(Rm), None, 0.0, 0) == -1
    assert lib.ekfslam_update_camera(h, 0, 4, 3, P(Hm), None, P(Rm), None, 0.0, 0) == -1
    assert lib.ekfslam_update_camera(h, 0, 4, 3, P(Hm), P(zm), None, None, 0.0, 0) == -1
    assert bank.device_bytes == bytes0                            # nothing allocated by a refused call
    bank.reset_filters()
    H, R = fix_model(3)
    bank.update_camera(H, np.zeros((4, 3)), R)
    assert bank.device_bytes > bytes0
    assert (bank.download_camera_update()["status"] == 0).all()
    bank.update_camera(H[:1], np.zeros((4, 1)), R[:1, :1], which=0)   # m = 1 <= 2 N_max
    assert (bank.download_camera_update()["status"] == 0).all()
    with pytest.raises(ValueError):
        bank.update_camera(np.zeros((3, 12)), np.zeros((4, 3)), R)
    bank.close()


def test_closed_loop_diagnostic(pkg):
    """The 50-frame closed loop of test_gpu_eval with a seeded position fix (sigma = 0.01) from the true pose after every
    step.  The camera-position error is taken after the step and before that frame's fix."""
    from tests.test_gpu_eval import _closed_loop, _world
    frames, sigma = 50, 0.01
    world = _world(4, frames)
    H, R = fix_model(3, sigma_r=sigma)
    rmse = {}
    for aided in (False, True):
        rng = np.random.RandomState(31)
        err = []

        def on_frame(bank, t):
            x, _, _ = bank.download_state(want_P=False)
            err.append(np.sum((x[:, 0:3] - world.pose_r[:, t]) ** 2, axis=1))
            if aided:
                z = world.pose_r[:, t] + sigma * rng.standard_normal((bank.B, 3))
                bank.update_camera(H, z, R, which=0)
                assert (bank.download_camera_update()["status"] == 0).all()

        _closed_loop(pkg, world, frames, on_frame).close()
        err = np.array(err)
        rmse[aided] = (float(np.sqrt(err.mean())), float(np.sqrt(err[frames // 2:].mean())))
    print("closed loop camera-position RMSE (all frames / last 25): unaided %.4f / %.4f, aided %.4f / %.4f"
          % (rmse[False] + rmse[True]))
    assert rmse[True][1] < rmse[False][1], rmse
