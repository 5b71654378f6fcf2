"""The Octave/MATLAB MEX gateway (mex/ekfslam_mex.c).  The image has neither mkoctfile nor mex.h, so the gateway
is compiled against mex/stub/mex.h and LINKED with mex/stub/mexrt.c - a minimal mxArray runtime (double
matrices, char rows, struct arrays, mexErrMsgIdAndTxt as a non-local exit) - and libekfslam.so.  The tests
drive mexFunction through that runtime exactly as Octave would call ekfslam_mex(cmd, ...):
  CPU : build + link, struct marshalling round trip, every argument-error path, the no-device error
  GPU : the reference-held golden frame and a full filter step through the gateway == the ctypes path
        (ekf_slam_b200.api) bit for bit; map_management / delete_a_feature / add_features_inverse_depth likewise."""
import copy
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def mexrt():
    if shutil.which("gcc") is None:
        pytest.skip("no C compiler")
    r = subprocess.run(["bash", os.path.join(ROOT, "mex", "build_test.sh")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    from tests import mexrt as m
    return m


def test_mex_gateway_compiles_against_stub():
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    r = subprocess.run([cc, "-fsyntax-only", "-Wall", "-Werror=implicit-function-declaration",
                        "-I" + os.path.join(ROOT, "mex", "stub"), "-I" + os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "mex", "ekfslam_mex.c")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_mex_gateway_only_calls_declared_abi():
    hdr = open(os.path.join(ROOT, "include", "ekfslam.h")).read()
    declared = set(re.findall(r"\b(ekfslam_[a-z0-9_]+)\s*\(", re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)))
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "mex", "ekfslam_mex.c")).read(), flags=re.S)
    used = set(re.findall(r"\b(ekfslam_[a-z0-9_]+)\s*\(", src)) - {"ekfslam_mex"}
    assert used and used <= declared, used - declared


def test_every_reference_function_has_a_shim():
    shims = {f[:-2] for f in os.listdir(os.path.join(ROOT, "mex", "shims")) if f.endswith(".m")}
    assert shims == {"ekf_prediction", "search_IC_matches", "ransac_hypotheses", "ekf_update_li_inliers",
                     "rescue_hi_inliers", "ekf_update_hi_inliers", "map_management", "inversedepth_2_cartesian",
                     "delete_a_feature", "add_features_inverse_depth"}
    src = open(os.path.join(ROOT, "mex", "ekfslam_mex.c")).read()
    for s in shims:
        assert '"%s"' % s in src
        body = open(os.path.join(ROOT, "mex", "shims", s + ".m")).read()
        assert "ekfslam_mex( '%s'" % s in body or "ekfslam_mex('%s'" % s in body


def test_octave_probe_is_reported(monkeypatch):
    """north_star asks for an Octave cross-run; where there is no Octave the benchmark says so instead of a number."""
    import bench
    monkeypatch.setattr(shutil, "which", lambda name: None)
    assert bench.octave_probe() == {"octave": None, "note": "OCTAVE ABSENT - reference CPU path not measured"}


def test_runtime_struct_round_trip(mexrt):
    fi = [{"type": "inversedepth", "h": np.array([[1.5, 2.5]]), "z": None, "R": np.eye(2)},
          {"type": "cartesian", "h": None, "z": np.array([[3.0], [4.0]]), "R": np.eye(2)}]
    back = mexrt.from_mx(mexrt.to_mx(fi))
    assert [e["type"] for e in back] == ["inversedepth", "cartesian"]
    assert back[0]["z"] is None and back[1]["h"] is None
    assert np.array_equal(back[0]["h"], fi[0]["h"]) and np.array_equal(back[1]["z"], fi[1]["z"])


def _s(v):
    """A 1x1 struct comes back as a one-element list (struct arrays are lists of dicts)."""
    return v[0] if isinstance(v, list) else v


def _filter(x, P):
    return {"type": "constant_velocity", "x_k_k": np.asarray(x).reshape(-1, 1), "p_k_k": np.asarray(P), "std_a": 0.007,
            "std_alpha": 0.007, "std_z": 1.0, "x_k_km1": None, "p_k_km1": None}


def _feature(ty="inversedepth"):
    return {"type": ty, "times_predicted": 0.0, "times_measured": 0.0, "individually_compatible": 0.0,
            "low_innovation_inlier": 0.0, "high_innovation_inlier": 0.0, "z": None, "h": None, "H": None, "S": None,
            "R": np.eye(2), "state_size": 6.0, "measurement_size": 2.0, "feature_when_initialized": -1.0}


def test_gateway_argument_errors(mexrt):
    f = _filter(np.zeros(13 + 6), np.eye(13 + 6))
    fi = [_feature()]
    cam = {"k1": 0.06333, "k2": 0.0139, "Cx": 160.2, "Cy": 128.9, "f": 2.1735, "dx": 0.0112, "dy": 0.0112, "nRows": 240.0,
           "nCols": 320.0}
    cases = [(("bogus_command", f, fi), "unknown command"),
             (("ekf_prediction",), "usage"),
             (("ekf_prediction", 1.0, fi), "usage"),
             (("search_IC_matches", f, fi), "needs cam"),
             (("ransac_hypotheses", f, fi, cam), "uniform stream"),
             (("rescue_hi_inliers", f, fi), "needs cam"),
             (("map_management", f, fi, cam), "needs cam, det"),
             (("map_management", f, fi, cam, np.zeros((2, 4)), 25.0, 2.0), "3 x K"),
             (("delete_a_feature", f["x_k_k"], f["p_k_k"], 1.0), "usage"),
             (("delete_a_feature", f["x_k_k"], f["p_k_k"], 3.0, fi), "out of range"),
             (("add_features_inverse_depth", np.zeros((2, 1)), np.zeros((14, 1)), np.eye(14), cam, 1.0, 1.0, 1.0), "not 13 +"),
             (("add_features_inverse_depth", np.zeros((2, 1))), "usage")]
    for args, needle in cases:
        with pytest.raises(mexrt.MexError) as e:
            mexrt.call(*args)
        assert e.value.ident == "ekfslam:arg" and needle in str(e.value), (args[0], str(e.value))
    # a features_info element without `type`
    with pytest.raises(mexrt.MexError) as e:
        mexrt.call("ekf_prediction", f, [{"h": None}])
    assert "type missing" in str(e.value)


def test_gateway_reports_missing_device_as_library_error(mexrt):
    """Runs in a child process with every device hidden, so that it also checks this where a GPU is present."""
    code = ("import numpy as np\n"
            "from tests import mexrt\n"
            "from tests.test_mex_gateway import _filter, _feature\n"
            "try:\n"
            "    mexrt.call('ekf_prediction', _filter(np.zeros(13 + 6), np.eye(13 + 6)), [_feature()], nargout=2)\n"
            "except mexrt.MexError as e:\n"
            "    print(e.ident, e)\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stderr
    ident, _, msg = r.stdout.strip().partition(" ")
    assert ident == "ekfslam:lib" and "no CUDA device" in msg, r.stdout     # no CPU fallback behind the gateway


# --------------------------------------------------------------------------------------------------------
# GPU: the gateway against the ctypes path
# --------------------------------------------------------------------------------------------------------
def _cam_dict():
    import ekf_slam_b200.api as api
    c = api.initialize_cam()
    return {k: float(getattr(c, k)) for k in ("k1", "k2", "Cx", "Cy", "f", "dx", "dy", "nRows", "nCols")}


def _api_features(fi_mx):
    import ekf_slam_b200.api as api
    out = []
    for e in fi_mx:
        a = api.new_feature(e["type"])
        for k in ("h", "z", "H", "S"):
            v = e.get(k)
            setattr(a, k, None if v is None else (np.asarray(v).reshape(-1) if k in ("h", "z") else np.asarray(v)))
        for k in ("individually_compatible", "low_innovation_inlier", "high_innovation_inlier", "times_predicted",
                  "times_measured"):
            v = e.get(k)
            setattr(a, k, int(np.asarray(v).reshape(-1)[0]) if v is not None else 0)
        fd = e.get("feature_when_initialized")
        a.feature_when_initialized = int(np.asarray(fd).reshape(-1)[0]) if fd is not None else -1
        out.append(a)
    return out


def _api_filter(f_mx):
    import ekf_slam_b200.api as api
    a = api.ekf_filter(f_mx["x_k_k"].reshape(-1), f_mx["p_k_k"], 0.007, 0.007, 1.0)
    if f_mx.get("x_k_km1") is not None:
        a.x_k_km1, a.p_k_km1 = f_mx["x_k_km1"].reshape(-1), f_mx["p_k_km1"]
    return a


@pytest.mark.gpu
def test_gateway_golden_frame_and_full_step_equal_ctypes_path(mexrt):
    import ekf_slam_b200.api as api
    from tests import helpers as T
    g = np.load(os.path.join(G, "features_information.npz"))
    cam = _cam_dict()
    # the reference-held frame: build the map through the gateway, predict, h/H/S
    x, P = api.initialize_x_and_p()
    X, Pm = x.reshape(-1, 1), P
    for k in range(g["uv_when_initialized"].shape[0]):
        X, Pm, newf = mexrt.call("add_features_inverse_depth", g["uv_when_initialized"][k].reshape(2, 1), X, Pm, cam,
                                 1.0, 1.0, 1.0, nargout=3)
        assert np.abs(newf.reshape(-1) - g["yi"][k]).max() < 1e-14
    f = _filter(X, Pm)
    fi = [_feature() for _ in range(13)]
    f, fi = mexrt.call("ekf_prediction", f, fi, nargout=2)
    f = _s(f)
    fi = mexrt.call("search_IC_matches", f, fi, cam)
    for k in range(13):
        assert np.abs(fi[k]["h"].reshape(-1) - g["h"][k]).max() < 1e-11
        assert T.rel_err(fi[k]["H"], g["H"][k]) < 1e-12 and T.rel_err(fi[k]["S"], g["S"][k]) < 1e-12
    # a full step on a synthetic frame, stage by stage, gateway vs api (same library underneath: bit-equal)
    import ekf_slam_b200.synth as synth
    N = 14
    seq = synth.SynthSequence(B=1, N=N, T=2, seed=77, n_u=64)
    x0, P0, _ = seq.initial_state()
    fm, fim = _filter(x0[0], P0[0]), [_feature() for _ in range(N)]
    fa, fia = api.ekf_filter(x0[0], P0[0], 0.007, 0.007, 1.0), [api.new_feature() for _ in range(N)]
    camo = api.initialize_cam()
    for t in (1, 2):
        cand = np.vstack([seq.zc[t, 0].T, seq.has[t, 0][None].astype(np.float64)])
        u = seq.uniforms(t)[0]
        for e in fim:                                                       # update_features_info.m (host side in both)
            e.update(individually_compatible=0.0, low_innovation_inlier=0.0, high_innovation_inlier=0.0, h=None, z=None, H=None, S=None)
        fia = api.update_features_info(fia)
        fm, fim = mexrt.call("ekf_prediction", fm, fim, nargout=2)
        fm = _s(fm)
        fa, fia = api.ekf_prediction(fa, fia)
        fim = mexrt.call("search_IC_matches", fm, fim, cam, cand)
        fia = api.search_IC_matches(fa, fia, camo, (seq.zc[t, 0], seq.has[t, 0]))
        fim = mexrt.call("ransac_hypotheses", fm, fim, cam, u.reshape(-1, 1))
        fia = api.ransac_hypotheses(fa, fia, camo, u=u)
        fm = _s(mexrt.call("ekf_update_li_inliers", fm, fim))
        fa = api.ekf_update_li_inliers(fa, fia)
        fim = mexrt.call("rescue_hi_inliers", fm, fim, cam)
        fia = api.rescue_hi_inliers(fa, fia, camo)
        fm = _s(mexrt.call("ekf_update_hi_inliers", fm, fim))
        fa = api.ekf_update_hi_inliers(fa, fia)
        assert np.array_equal(fm["x_k_k"].reshape(-1), fa.x_k_k) and np.array_equal(fm["p_k_k"], fa.p_k_k), t
        for e, a in zip(fim, fia):
            for k in ("individually_compatible", "low_innovation_inlier", "high_innovation_inlier"):
                assert int(e[k][0, 0]) == getattr(a, k)
        assert sum(int(e["low_innovation_inlier"][0, 0]) for e in fim) >= 4


@pytest.mark.gpu
def test_gateway_map_management_equals_ctypes_path(mexrt):
    import ekf_slam_b200.api as api
    fx = np.load(os.path.join(G, "ref_map_t80.npz"))
    cam, camo = _cam_dict(), api.initialize_cam()
    x, P = api.initialize_x_and_p()
    fm, fim = _filter(x, P), None                       # features_info = [] (mono_slam.m:35)
    fa, fia = api.ekf_filter(x, P, 0.007, 0.007, 1.0), []
    b, minf = 0, float(fx["min_features"])
    for t in range(12):
        nd = int(fx["det_n"][b, t])
        det = np.vstack([fx["det_uv"][b, t, :nd].T, fx["det_tag"][b, t, :nd][None].astype(np.float64)])
        fm, fim = mexrt.call("map_management", fm, fim, cam, det, minf, float(t + 1), nargout=2)
        fm = _s(fm)
        fa, fia = api.map_management(fa, fia, camo, (fx["det_uv"][b, t, :nd], fx["det_tag"][b, t, :nd]), int(minf), t + 1)
        k = len(fim)
        assert k == len(fia) == fx["nfeat"][b, t]
        assert np.array_equal(fm["x_k_k"].reshape(-1), fa.x_k_k) and np.array_equal(fm["p_k_k"], fa.p_k_k), t
        assert [e["type"] for e in fim] == [a.type for a in fia]
        assert [int(e["feature_when_initialized"][0, 0]) for e in fim] == [a.feature_when_initialized for a in fia] \
            == list(fx["tags"][b, t, :k])
        assert [int(e["times_predicted"][0, 0]) for e in fim] == [a.times_predicted for a in fia]
        for e, a in zip(fim, fia):
            if e["yi"] is not None and a.yi is not None:
                assert np.array_equal(e["yi"].reshape(-1), a.yi)
        # continue the sequence on the ctypes path and mirror its result into the gateway's structs
        fa, fia = api.filter_step(fa, fia, camo, (fx["zc"][b, t, :k], fx["has"][b, t, :k]), u=fx["U"][b, t])
        fm["x_k_k"], fm["p_k_k"] = fa.x_k_k.reshape(-1, 1), fa.p_k_k
        for e, a in zip(fim, fia):
            e.update(h=None if a.h is None else a.h.reshape(1, 2), z=None if a.z is None else a.z.reshape(2, 1),
                     individually_compatible=float(a.individually_compatible),
                     low_innovation_inlier=float(a.low_innovation_inlier),
                     high_innovation_inlier=float(a.high_innovation_inlier))
    # single-purpose commands
    X, Pn = mexrt.call("delete_a_feature", fm["x_k_k"], fm["p_k_k"], 3.0, fim, nargout=2)
    Xa, Pa = api.delete_a_feature(fa.x_k_k, fa.p_k_k, 2, fia)
    assert np.array_equal(X.reshape(-1), Xa) and np.array_equal(Pn, Pa)
    f2, fi2 = mexrt.call("inversedepth_2_cartesian", fm, fim, nargout=2)
    f2 = _s(f2)
    fa2, fia2 = api.inversedepth_2_cartesian(copy.deepcopy(fa), copy.deepcopy(fia))
    assert [e["type"] for e in fi2] == [a.type for a in fia2]
    assert np.array_equal(f2["x_k_k"].reshape(-1), fa2.x_k_k)
