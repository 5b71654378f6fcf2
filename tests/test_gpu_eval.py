"""Scoring against the resident ground truth on the device (ekfslam_evaluate / ekfslam_map_cartesian) against its numpy
mirror (oracle/eval_oracle.py) on the downloaded state: the closed loop of test_gpu_map_ref (map growth, Cartesian
conversions, deletions), read-only-ness, run-to-run determinism, the map export, the error codes, and the full bench
shape on a seeded sample of filters."""
import numpy as np
import pytest

from oracle import eval_oracle as E

pytestmark = pytest.mark.gpu
FLOAT = ["pos_sq_err", "rot_sq_err", "nees_pos", "nees_pose", "map_sq_err", "map_nees"]
ERR = ["pos_sq_err", "rot_sq_err", "map_sq_err"]
NEES = ["nees_pos", "nees_pose", "map_nees"]
INT = ["n_map", "n_skip", "frames", "status"]


@pytest.fixture(scope="module")
def pkg():
    import ekf_slam_b200 as pkg
    return pkg


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    assert np.array_equal(np.isnan(a), np.isnan(b))
    m = ~np.isnan(b)
    if not m.any():
        return 0.0
    return float(np.max(np.abs(a[m] - b[m])) / max(np.max(np.abs(b[m])), 1e-300))


def _world(B, frames, seed=2):
    import ekf_slam_b200.synth as synth
    from tests.golden.make_ref_steps import MAP_WORLD
    return synth.SynthWorld(B, T=frames, seed=seed, **MAP_WORLD)


def _closed_loop(pkg, world, frames, on_frame=None):
    """The schedule of test_closed_loop_on_device_50_frames: B=4, N=64, K=20, min 20 features, n_u=64."""
    B, N, K, minf, n_u = 4, 64, 20, 20, 64
    bank = pkg.FilterBank(B, N)
    bank.reset_filters()
    bank.world_upload(world)
    for step in range(1, frames + 1):
        bank.world_detect(step - 1, K)
        bank.map_management(minf)
        bank.world_candidates(step)
        bank.world_uniforms(step, n_u)
        bank.step(reset=False, match_mode=1)
        if on_frame is not None:
            on_frame(bank, step)
    return bank


def _mirror(bank, world, t, b0=0, nb=None):
    nb = bank.B - b0 if nb is None else nb
    x, P, _ = bank.download_state(b0=b0, nb=nb)
    ty, nf = bank.download_feature_types(b0=b0, nb=nb)
    tg = bank.download_feature_tags(b0=b0, nb=nb)
    out = []
    for k in range(nb):
        b = b0 + k
        out.append(E.evaluate(x[k], P[k], ty[k], nf[k], tg[k], world.points[b], world.pose_r[b, t], world.pose_q[b, t],
                              N=bank.N) + (E.map_cartesian(x[k], P[k], ty[k], nf[k], bank.N),))
    return out, ty, nf


def _compare(got, mirror, worst, b0=0):
    for k, (rec, fe, fn, _) in enumerate(mirror):
        b = b0 + k
        for f in INT:
            assert got[f][k] == rec[f], (f, b, got[f][k], rec[f])
        for f in ERR:
            worst["err"] = max(worst["err"], _rel(got[f][k], rec[f]))
        for f in NEES:
            worst["nees"] = max(worst["nees"], _rel(got[f][k], rec[f]))
        worst["err"] = max(worst["err"], _rel(got["feat_err"][k], fe))
        worst["nees"] = max(worst["nees"], _rel(got["feat_nees"][k], fn))
    assert worst["err"] < 1e-9 and worst["nees"] < 1e-6, worst


def test_closed_loop_matches_mirror_every_frame(pkg):
    frames = 50
    world = _world(4, frames)
    worst = dict(err=0.0, nees=0.0, map=0.0, tot=0.0)
    seen = dict(cart=0, n_map=0)
    per_frame = []

    def on_frame(bank, t):
        bank.evaluate(t)
        got = bank.download_eval()
        mirror, ty, nf = _mirror(bank, world, t)
        _compare(got, mirror, worst)
        p, C = bank.map_cartesian()
        for b, m in enumerate(mirror):
            worst["map"] = max(worst["map"], _rel(p[b], m[3][0]), _rel(C[b], m[3][1]))
        assert worst["map"] < 1e-9, worst
        per_frame.append({f: got[f].copy() for f in FLOAT + INT})
        seen["cart"] += int(sum((ty[b, :nf[b]] == 2).sum() for b in range(len(nf))))
        seen["n_map"] += int(got["n_map"].sum())

    bank = _closed_loop(pkg, world, frames, on_frame)
    tot = bank.download_eval(totals=True)
    for f in FLOAT:
        s = np.zeros(bank.B)
        for r in per_frame:
            s = s + r[f]
        worst["tot"] = max(worst["tot"], _rel(tot[f], s))
    for f in ["n_map", "n_skip"]:
        assert np.array_equal(tot[f], sum(r[f] for r in per_frame)), f
    assert (tot["frames"] == frames).all()
    assert np.array_equal(tot["status"], np.bitwise_or.reduce([r["status"] for r in per_frame]))
    assert worst["tot"] < 1e-12, worst
    assert seen["cart"] > 0 and seen["n_map"] > 0, seen
    anees = tot["nees_pose"] / tot["frames"]
    print("closed loop eval: worst rel err %.2e (errors, C_f, p), %.2e (NEES), %.2e (map export), %.2e (totals); "
          "camera ANEES (6 dof) per filter %s; map ANEES %s"
          % (worst["err"], worst["nees"], worst["map"], worst["tot"], np.round(anees, 2),
             np.round(tot["map_nees"] / np.maximum(tot["n_map"], 1), 2)))
    bank.close()


def test_evaluation_is_read_only(pkg):
    frames = 25
    world = _world(4, frames)

    def score(bank, t):
        bank.evaluate(t)
        bank.map_cartesian()

    out = []
    for hook in (None, score):
        bank = _closed_loop(pkg, world, frames, hook)
        x, P, ns = bank.download_state()
        xp, _, _ = bank.download_state(which=1, want_P=False)
        d = bank.download_features()
        out.append(dict(x=x, P=P, ns=ns, xp=xp, flags=d["flags"], counters=d["counters"],
                        tags=bank.download_feature_tags(), types=bank.download_feature_types()[0],
                        stats=np.stack([v for v in bank.download_stats().values()])))
        bank.close()
    for k in out[0]:
        assert np.array_equal(out[0][k].view(np.uint8), out[1][k].view(np.uint8)), k


def test_evaluation_is_deterministic(pkg):
    world = _world(4, 12)
    bank = _closed_loop(pkg, world, 12)
    recs = []
    for _ in range(2):
        bank.evaluate(12)
        recs.append(bank.download_eval())
    for k in recs[0]:
        assert np.array_equal(recs[0][k].view(np.uint8), recs[1][k].view(np.uint8)), k
    tot = bank.download_eval(totals=True)
    assert (tot["frames"] == 2).all()
    bank.close()


def test_map_export_without_world(pkg):
    import ekf_slam_b200.synth as synth
    B, N = 3, 12
    seq = synth.SynthSequence(B=B, N=N, T=2, seed=5)
    x0, P0, types = seq.initial_state()
    nfeat = np.array([N, 7, 3], dtype=np.int32)
    types[1, 7:] = 0
    types[2, 3:] = 0
    bank = pkg.FilterBank(B, N)
    bank.upload_feature_types(types, nfeat)
    bank.upload_state(x0, P0)
    bank.inversedepth_2_cartesian(force_index=2)           # a Cartesian block in every map
    p, C = bank.map_cartesian()
    x, P, _ = bank.download_state()
    ty, nf = bank.download_feature_types()
    assert all((ty[b] == 2).sum() == 1 for b in range(B))
    worst = 0.0
    for b in range(B):
        pm, Cm = E.map_cartesian(x[b], P[b], ty[b], nf[b], N)
        worst = max(worst, _rel(p[b], pm), _rel(C[b], Cm))
        assert np.isnan(p[b, nf[b]:]).all() and np.isnan(C[b, nf[b]:]).all()
    assert worst < 1e-9, worst
    # a partial range returns the same slots
    p1, C1 = bank.map_cartesian(b0=1, nb=1)
    assert np.array_equal(p1[0], p[1], equal_nan=True) and np.array_equal(C1[0], C[1], equal_nan=True)
    with pytest.raises(pkg.EkfSlamError) as e:
        bank.evaluate(0)
    assert e.value.code == -4                               # ERR_STATE: no world
    with pytest.raises(pkg.EkfSlamError) as e:
        bank.download_eval()
    assert e.value.code == -4                               # nothing evaluated yet
    bank.close()


def test_errors_and_reset(pkg):
    import ctypes as C
    from ekf_slam_b200 import _lib as L
    world = _world(2, 6)
    bank = pkg.FilterBank(2, 16)
    bytes0 = bank.device_bytes
    bank.reset_filters()
    bank.world_upload(world)
    assert bank.device_bytes == bytes0                      # nothing allocated before the first evaluation
    for t in (-1, 7):
        with pytest.raises(pkg.EkfSlamError) as e:
            bank.evaluate(t)
        assert e.value.code == -1                           # ERR_INVALID: t outside [0, T]
    bank.evaluate(0)
    bank.evaluate(6)
    tot = bank.download_eval(totals=True)
    assert (tot["frames"] == 2).all()
    rec = (L.Eval * 1)()
    fe = np.empty((1, 16, 3))
    code = bank.lib.ekfslam_download_eval(bank._h, 0, 1, 1, C.cast(rec, C.c_void_p), fe.ctypes.data_as(C.c_void_p), None)
    assert code == -1                                       # per-feature outputs exist for the last frame only
    bank.reset_eval()
    tot = bank.download_eval(totals=True)
    for k in FLOAT + INT:
        assert (tot[k] == 0).all(), k
    rec = bank.download_eval()
    assert (rec["frames"] == 1).all()                       # the last frame's record survives the reset
    bank.close()


def test_full_size_sample_matches_mirror(pkg):
    """B=4096, N=100 (the bench shape) on SynthSequence + truth_world(), 3 frames; 64 seeded filters against the
    mirror, downloading only their state."""
    import ekf_slam_b200.synth as synth
    B, N, frames = 4096, 100, 3
    seq = synth.SynthSequence(B=B, N=N, T=frames, seed=2024)
    bank = pkg.FilterBank(B, N)
    bank.reset_filters()
    for k in range(N):
        bank.add_features_inverse_depth(np.ascontiguousarray(seq.zc[0, :, k]))
    bank.upload_feature_meta(tag=np.tile(np.arange(N, dtype=np.int32), (B, 1)))
    world = seq.truth_world()
    bank.world_upload(world)
    sample = np.sort(np.random.RandomState(11).choice(B, 64, replace=False))
    worst = dict(err=0.0, nees=0.0)
    for t in range(1, frames + 1):
        zc, has = seq.frame(t)
        bank.upload_candidates(zc, has)
        bank.upload_uniforms(seq.uniforms(t))
        bank.step(reset=True, match_mode=1)
        bank.evaluate(t)
        for b in sample:
            got = bank.download_eval(b0=int(b), nb=1)
            mirror, _, _ = _mirror(bank, world, t, b0=int(b), nb=1)
            _compare(got, mirror, worst, b0=int(b))
    tot = bank.download_eval(totals=True)
    assert (tot["frames"] == frames).all() and (tot["n_map"] > 0).all()
    print("full size (B=%d, N=%d, %d frames, 64 sampled filters): worst rel err %.2e (errors), %.2e (NEES); "
          "mean camera NEES (6 dof) %.2f, mean map NEES per feature %.2f"
          % (B, N, frames, worst["err"], worst["nees"], tot["nees_pose"].mean() / frames,
             tot["map_nees"].sum() / tot["n_map"].sum()))
    bank.close()
