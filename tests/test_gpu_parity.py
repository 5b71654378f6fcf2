"""CUDA path vs the CPU oracle on identical seeded inputs, through the C ABI.

Bar (BASELINE.json north_star): inlier sets and feature indices bit-exact, state and
covariance within 1e-9 relative.  Checked teacher-forced (every step restarted from the oracle's
state) and free-running (device state carried across frames).
"""
import numpy as np
import pytest

from oracle import ekf_oracle as O
from tests import helpers as T

pytestmark = pytest.mark.gpu

TOL = 1e-9


@pytest.fixture(scope="module")
def ekf():
    import ekf_slam_b200 as pkg
    import ekf_slam_b200.synth as synth
    return pkg, synth


def _run_sequence(ekf, B, N, frames, seed, fixed=0, n_u=64, p_outlier=0.2, teacher_forced=False, cart=None, noise_px=0.5,
                  nfeat=None, behind=None):
    pkg, synth = ekf
    seq = synth.SynthSequence(B=B, N=N, T=frames, seed=seed, p_outlier=p_outlier, n_u=n_u, noise_px=noise_px)
    x0, P0, types = seq.initial_state()
    n_max = 13 + 6 * N
    if behind:
        # features whose ray points away from the camera: never predicted (h stays empty), never matched
        for (b, i) in behind:
            x0[b, 13 + 6 * i + 3] += np.pi
    if nfeat is not None:
        # ragged batch: filter b keeps its first nfeat[b] features (0 = a camera-only filter)
        types = types.copy()
        for b in range(B):
            nb_ = 13 + 6 * nfeat[b]
            types[b, nfeat[b]:] = 0
            x0[b, nb_:] = 0.0
            P0[b, nb_:, :] = 0.0
            P0[b, :, nb_:] = 0.0
            seq.has[:, b, nfeat[b]:] = 0
    if cart:
        xs, Ps, ts = [], [], []
        for b in range(B):
            xb, Pb, tb = synth.convert_to_cartesian(x0[b], P0[b], types[b], cart)
            xs.append(np.pad(xb, (0, n_max - len(xb))))
            Ps.append(np.pad(Pb, ((0, n_max - len(xb)), (0, n_max - len(xb)))))
            ts.append(tb)
        x0, P0, types = np.stack(xs), np.stack(Ps), np.stack(ts)
    cam = O.initialize_cam()
    bank = pkg.FilterBank(B, N, n_max)
    bank.set_params(fixed_hyp=fixed)
    bank.upload_feature_types(types)
    bank.upload_state(x0, P0)
    _, _, nstate = bank.download_state(want_P=False)
    filts = [T.oracle_filter(x0[b, :nstate[b]], P0[b, :nstate[b], :nstate[b]]) for b in range(B)]
    feats = [T.oracle_features(types[b]) for b in range(B)]
    worst = dict(x=0.0, P=0.0)
    totals = dict(li=0, hi=0, ic=0, iters=0)
    for t in range(1, frames + 1):
        zc, has = seq.frame(t)
        u = seq.uniforms(t, n_u)
        if teacher_forced and t > 1:
            xs = np.zeros((B, n_max))
            Ps = np.zeros((B, n_max, n_max))
            for b in range(B):
                xs[b, :nstate[b]] = filts[b].x_k_k
                Ps[b, :nstate[b], :nstate[b]] = filts[b].p_k_k
            bank.upload_state(xs, Ps)
        bank.upload_candidates(zc, has)
        bank.upload_uniforms(u)
        bank.step(reset=True, match_mode=1)
        xg, Pg, _ = bank.download_state()
        fg = bank.download_flags()
        st = bank.download_stats()
        for b in range(B):
            filts[b], feats[b], info = T.oracle_step(filts[b], feats[b], cam, zc[b], has[b], u[b], fixed)
            n = nstate[b]
            fo = T.oracle_flags(feats[b], N)
            mask = T.F_HAS_H | T.F_HAS_Z | T.F_IC | T.F_LI | T.F_HI
            assert np.array_equal(fg[b] & mask, fo), "flag mismatch: frame %d filter %d" % (t, b)
            assert st["ransac_iters"][b] == info["iterations"], (t, b)
            assert st["status"][b] == 0
            ex = T.rel_err(xg[b, :n], filts[b].x_k_k)
            eP = T.rel_err(Pg[b, :n, :n], filts[b].p_k_k)
            worst["x"] = max(worst["x"], ex)
            worst["P"] = max(worst["P"], eP)
            assert ex < TOL and eP < TOL, "frame %d filter %d: x %.2e P %.2e" % (t, b, ex, eP)
            assert np.array_equal(Pg[b], Pg[b].T)
            totals["li"] += int(st["n_li"][b])
            totals["hi"] += int(st["n_hi"][b])
            totals["ic"] += int(st["n_ic"][b])
            totals["iters"] += int(st["ransac_iters"][b])
    bank.close()
    return worst, totals


def test_teacher_forced_small(ekf):
    worst, tot = _run_sequence(ekf, B=4, N=12, frames=6, seed=100, teacher_forced=True)
    assert tot["li"] > 0 and tot["ic"] > 0


def test_free_running_small(ekf):
    worst, tot = _run_sequence(ekf, B=4, N=12, frames=8, seed=200)
    assert tot["li"] > 0


def test_free_running_n40(ekf):
    """BASELINE config 1 shape (~40 features), adaptive RANSAC."""
    worst, tot = _run_sequence(ekf, B=3, N=40, frames=6, seed=300)
    assert tot["hi"] >= 0 and tot["li"] > 40


def test_n100_fixed_256(ekf):
    """BASELINE config 2 shape: N=100, 256 hypotheses per frame."""
    worst, tot = _run_sequence(ekf, B=2, N=100, frames=3, seed=400, fixed=256, n_u=256)
    assert tot["iters"] == 2 * 3 * 256


def test_heavy_outliers(ekf):
    worst, tot = _run_sequence(ekf, B=3, N=30, frames=5, seed=500, p_outlier=0.5, n_u=200)
    assert tot["li"] > 0


def test_mixed_cartesian(ekf):
    """BASELINE config 5 shape: mixed inverse-depth / Cartesian maps."""
    worst, tot = _run_sequence(ekf, B=3, N=20, frames=5, seed=600, cart=[0, 3, 4, 9, 15, 19])
    assert tot["li"] > 0


def test_no_matches_is_passthrough(ekf):
    pkg, synth = ekf
    seq = synth.SynthSequence(B=2, N=8, T=2, seed=7)
    x0, P0, types = seq.initial_state()
    bank = pkg.FilterBank(2, 8)
    bank.upload_feature_types(types)
    bank.upload_state(x0, P0)
    zc, has = seq.frame(1)
    bank.upload_candidates(zc, np.zeros_like(has))   # no candidate at all
    bank.upload_uniforms(seq.uniforms(1, 16))
    bank.step()
    xg, Pg, _ = bank.download_state()
    st = bank.download_stats()
    assert (st["n_ic"] == 0).all() and (st["n_li"] == 0).all() and (st["ransac_iters"] == 0).all()
    cam = O.initialize_cam()
    for b in range(2):
        f = T.oracle_filter(x0[b], P0[b])
        f, _ = O.ekf_prediction(f, [])
        assert T.rel_err(xg[b], f.x_k_km1) < 1e-12
        assert T.rel_err(Pg[b], f.p_k_km1) < 1e-12
    bank.close()


def test_large_map_n500(ekf):
    """BASELINE config 4 shape: N=500 features (n=3013), dense covariance update on the DMMA path."""
    worst, tot = _run_sequence(ekf, B=1, N=500, frames=2, seed=700, n_u=64)
    assert tot["li"] > 200


def test_large_map_n724_tile_downdate(ekf):
    """N=724 features (n=4357): the per-CTA tile table of the li downdate no longer fits the persistent kernel's shared
    memory, so it falls back to one CTA per tile (k_downdate_tile), while the hi downdate stays on k_downdate_ws2 and the
    Cholesky takes the lock-step blocked-64 path.  Same bar as N=500; the profiler confirms that the fallback ran."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        worst, tot = _run_sequence(ekf, B=1, N=724, frames=2, seed=710, n_u=64)
    kernels = {e.name for e in prof.events()}
    assert any("k_downdate_tile" in k for k in kernels), sorted(kernels)
    assert any("k_downdate_ws2" in k for k in kernels), sorted(kernels)
    assert tot["li"] > 200


def test_ragged_batch_and_unpredicted_features(ekf):
    """Filters of one batch with different map sizes (24, 17, 5 and 0 features: n = 157, 115, 43, 13) and features that
    are never predicted (ray pointing away from the camera: h / H / S stay empty, mc/predict_camera_measurements.m:14-16)."""
    nf = [24, 17, 5, 0]
    worst, tot = _run_sequence(ekf, B=4, N=24, frames=4, seed=840, nfeat=nf, behind=[(0, 3), (0, 11), (1, 0), (2, 4)])
    assert tot["li"] > 20 and tot["ic"] > 40


def test_downdate_filter_groups(ekf, monkeypatch):
    """The persistent downdate keeps its per-CTA tile metadata in shared memory and therefore processes very large
    batches in groups of filters (one launch per group); EKFSLAM_DD_GROUP forces tiny groups so that the
    group offset path is exercised at test sizes.  Same parity bar."""
    monkeypatch.setenv("EKFSLAM_DD_GROUP", "2")
    worst, tot = _run_sequence(ekf, B=5, N=24, frames=3, seed=810)
    assert tot["li"] > 20


def test_n100_many_inliers_large_k(ekf):
    """No gross outliers and little pixel noise at N=100: the li update stacks more than 144 rows, i.e. the Cholesky runs in the
    200-row resident variant (512 threads, second side stream) and the W GEMM spans three row tiles."""
    worst, tot = _run_sequence(ekf, B=2, N=100, frames=3, seed=820, p_outlier=0.0, noise_px=0.15)
    assert tot["li"] > 2 * 3 * 72, tot


def test_n120_more_than_200_stacked_rows(ekf):
    """N=120 without gross outliers: 106-113 li inliers per filter (oracle), i.e. k = 212-226 stacked rows - beyond the largest
    shared-memory resident Cholesky variant (200 rows), so the factorisation runs in the global-memory kernel (k_chol) behind
    the resident ones, and the W GEMM spans four row tiles."""
    worst, tot = _run_sequence(ekf, B=2, N=120, frames=2, seed=830, p_outlier=0.0, noise_px=0.15)
    assert tot["li"] > 2 * 2 * 100, tot


def test_row_pitch_256_bytes(ekf):
    """Row pitch of x / P / G: a multiple of 256 bytes (ld % 32 == 0); at n = 85 (ld = 96) the last 64-wide tile column of the
    covariance downdate is partial, results must not differ from the oracle."""
    pkg, _ = ekf
    bank = pkg.FilterBank(1, 12, 85)
    assert bank.ld % 32 == 0 and bank.ld >= 85
    bank.close()
    worst, tot = _run_sequence(ekf, B=3, N=12, frames=3, seed=860)
    assert tot["li"] > 30, tot


def test_blocked64_cholesky_ragged_k(ekf):
    """Few filters with N_max >= 128 take the 64-wide blocked DMMA factorisation (k_chol_big.cu): three filters with
    different map sizes, so the stacked innovation sizes differ per filter and are not multiples of 64."""
    nf = [140, 97, 33]
    worst, tot = _run_sequence(ekf, B=3, N=140, frames=3, seed=850, nfeat=nf, p_outlier=0.1)
    assert tot["li"] > 300, tot


def test_innovation_gather_mixed_ragged_map(ekf):
    """S_i = H_i P H_i' + R_i from 13x13 / 10x10 gathers of P (k_innov_gather; mc/search_IC_matches.m:6-10) on a mixed
    inverse-depth / Cartesian, ragged batch with a fully dense covariance, against the oracle's dense
    H P H' + R: h, the compact Jacobian and S to 1e-12; the G rows are never formed on this path."""
    pkg, synth = ekf
    B, N = 4, 30
    seq = synth.SynthSequence(B=B, N=N, T=2, seed=321, n_u=16)
    x0, P0, types = seq.initial_state()
    n_max = 13 + 6 * N
    nfeat = [30, 30, 11, 1]
    cart = [0, 3, 4, 9, 17, 29]
    xs, Ps, ts, ns = [], [], [], []
    rng = np.random.RandomState(7)
    for b in range(B):
        tb = types[b].copy()
        nb_ = 13 + 6 * nfeat[b]
        tb[nfeat[b]:] = 0
        xb, Pb = x0[b, :nb_].copy(), P0[b, :nb_, :nb_].copy()
        A = rng.normal(0, 1e-3, (nb_, nb_))           # fill in every cross-covariance block
        Pb = Pb + A @ A.T
        if b < 2:
            xb, Pb, tb2 = synth.convert_to_cartesian(np.pad(xb, (0, n_max - nb_)), np.pad(Pb, ((0, n_max - nb_),) * 2),
                                                     np.pad(tb[:N], (0, 0)), cart)
            tb = tb2
            nb_ = 13 + 6 * int((tb == 1).sum()) + 3 * int((tb == 2).sum())
            xb, Pb = xb[:nb_], Pb[:nb_, :nb_]
        xs.append(np.pad(xb, (0, n_max - nb_)))
        Ps.append(np.pad(Pb, ((0, n_max - nb_), (0, n_max - nb_))))
        ts.append(tb)
        ns.append(nb_)
    xs, Ps, ts = np.stack(xs), np.stack(Ps), np.stack(ts)
    bank = pkg.FilterBank(B, N, n_max)
    bank.upload_feature_types(ts)
    bank.upload_state(xs, Ps)
    bank.begin_frame()
    bank.ekf_prediction()
    bank.measure(1)
    d = bank.download_features()
    cam = O.initialize_cam()
    checked = 0
    for b in range(B):
        f = T.oracle_filter(xs[b, :ns[b]], Ps[b, :ns[b], :ns[b]])
        fi = T.oracle_features(ts[b])
        f, fi = O.ekf_prediction(f, fi)
        fi = O.predict_and_derive(f, fi, cam)
        Hc = T.compact_H(fi)
        for i, a in enumerate(fi):
            has_h = bool(d["flags"][b, i] & T.F_HAS_H)
            assert has_h == (a.h is not None), (b, i)
            if a.h is None:
                continue
            np.testing.assert_allclose(d["h"][b, i], a.h, rtol=1e-12, atol=1e-12)
            np.testing.assert_allclose(d["Hc"][b, i], Hc[i], rtol=1e-11, atol=1e-11 * np.abs(Hc[i]).max())
            np.testing.assert_allclose(d["S"][b, i], a.S, rtol=1e-12, atol=1e-12 * np.abs(a.S).max())
            checked += 1
    assert checked >= 60
    bank.close()
