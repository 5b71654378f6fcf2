"""FilterBank — B independent EKF-SLAM filters resident on one B200.

Thin, typed wrapper over the C ABI (include/ekfslam.h).  All arrays crossing this boundary
are host numpy arrays (C-contiguous); device memory belongs to the context.  The batched
layout is structure-of-arrays: ``x [B, n_max]``, ``P [B, n_max, n_max]``, per-feature fields
``[B, N_max, ...]`` (see the header for the exact shapes).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _c(a, dtype, shape=None):
    a = np.ascontiguousarray(a, dtype=dtype)
    if shape is not None and tuple(a.shape) != tuple(shape):
        raise ValueError("expected shape %s, got %s" % (tuple(shape), tuple(a.shape)))
    return a


class FilterBank:
    def __init__(self, B, N_max, n_max=None, device=0, camera=None, params=None):
        self.lib = L.load()
        n_max = int(n_max if n_max is not None else 13 + 6 * N_max)
        h = C.c_void_p()
        L.check(self.lib.ekfslam_create(C.byref(h), int(device), int(B), int(N_max), n_max))
        self._h = h
        self.B, self.N, self.n_max, self.device = int(B), int(N_max), n_max, int(device)
        self._lm_L = 0    # landmarks per filter of the last upload_landmarks
        ld = C.c_int()
        L.check(self.lib.ekfslam_dims(self._h, None, None, None, C.byref(ld)))
        self.ld = ld.value
        self.camera = L.Camera()
        self.lib.ekfslam_default_camera(C.byref(self.camera))
        self.params = L.Params()
        self.lib.ekfslam_default_params(C.byref(self.params))
        if camera is not None:
            self.set_camera(camera)
        if params is not None:
            self.set_params(**params)

    # -- lifetime -------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self.lib.ekfslam_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- configuration --------------------------------------------------------------------
    def set_camera(self, cam):
        """cam: any object with the fields of mc/initialize_cam.m (k1,k2,Cx,Cy,f,dx,dy,nRows,nCols)."""
        for name, _ in L.Camera._fields_:
            setattr(self.camera, name, getattr(cam, name))
        L.check(self.lib.ekfslam_set_camera(self._h, C.byref(self.camera)))

    def set_params(self, **kw):
        for k, v in kw.items():
            if not hasattr(self.params, k):
                raise KeyError(k)
            setattr(self.params, k, v)
        L.check(self.lib.ekfslam_set_params(self._h, C.byref(self.params)))

    def set_stream(self, cuda_stream):
        L.check(self.lib.ekfslam_set_stream(self._h, C.c_void_p(cuda_stream) if cuda_stream else None))

    def synchronize(self):
        L.check(self.lib.ekfslam_synchronize(self._h))

    @property
    def device_bytes(self):
        return int(self.lib.ekfslam_device_bytes(self._h))

    @property
    def launch_count(self):
        return int(self.lib.ekfslam_launch_count(self._h))

    def device_ptr(self, name):
        return self.lib.ekfslam_device_ptr(self._h, name.encode())

    # -- measurement hooks ------------------------------------------------------------------
    def enable_timing(self, on=True):
        L.check(self.lib.ekfslam_enable_timing(self._h, 1 if on else 0))

    def kernel_times(self):
        """{kernel name: (accumulated ms, launches)} since timing was (re-)enabled."""
        out = {}
        for slot in range(self.lib.ekfslam_kernel_count()):
            name = C.create_string_buffer(64)
            ms = C.c_double()
            cnt = C.c_int64()
            L.check(self.lib.ekfslam_kernel_time(self._h, slot, name, 64, C.byref(ms), C.byref(cnt)))
            out[name.value.decode()] = (ms.value, cnt.value)
        return out

    def bind_frame(self, d_zc, d_fl, d_u, n_u):
        """Device pointers (ints) of caller-owned frame buffers; see ekfslam_bind_frame."""
        L.check(self.lib.ekfslam_bind_frame(self._h, C.c_void_p(d_zc), C.c_void_p(d_fl), C.c_void_p(d_u), int(n_u)))

    def unbind_frame(self):
        L.check(self.lib.ekfslam_unbind_frame(self._h))

    # -- filter struct <-> device ---------------------------------------------------------
    def upload_state(self, x=None, P=None, nstate=None, which=0, b0=0):
        nb = None
        for a in (x, P, nstate):
            if a is not None:
                nb = len(a)
        if nb is None:
            return
        xx = None if x is None else _c(x, np.float64, (nb, self.n_max))
        PP = None if P is None else _c(P, np.float64, (nb, self.n_max, self.n_max))
        ns = None if nstate is None else _c(nstate, np.int32, (nb,))
        L.check(self.lib.ekfslam_upload_state(self._h, b0, nb, which, _ptr(xx), _ptr(PP), _ptr(ns)))

    def download_state(self, which=0, b0=0, nb=None, want_P=True):
        nb = self.B - b0 if nb is None else nb
        x = np.empty((nb, self.n_max))
        P = np.empty((nb, self.n_max, self.n_max)) if want_P else None
        ns = np.empty(nb, dtype=np.int32)
        L.check(self.lib.ekfslam_download_state(self._h, b0, nb, which, _ptr(x), _ptr(P), _ptr(ns)))
        return x, P, ns

    # -- features_info <-> device ---------------------------------------------------------
    def upload_feature_types(self, types, nfeat=None, b0=0):
        types = _c(types, np.uint8)
        nb = types.shape[0]
        if types.shape != (nb, self.N):
            raise ValueError("types must be [nb, N_max]")
        if nfeat is None:
            nfeat = (types != 0).sum(axis=1)
        nfeat = _c(nfeat, np.int32, (nb,))
        L.check(self.lib.ekfslam_upload_feature_types(self._h, b0, nb, _ptr(types), _ptr(nfeat)))

    def upload_matches(self, z, flags, b0=0):
        z = _c(z, np.float64)
        nb = z.shape[0]
        z = _c(z, np.float64, (nb, self.N, 2))
        flags = _c(flags, np.uint8, (nb, self.N))
        L.check(self.lib.ekfslam_upload_matches(self._h, b0, nb, _ptr(z), _ptr(flags)))

    def upload_candidates(self, zc, has, b0=0):
        zc = _c(zc, np.float64)
        nb = zc.shape[0]
        zc = _c(zc, np.float64, (nb, self.N, 2))
        has = _c(has, np.uint8, (nb, self.N))
        L.check(self.lib.ekfslam_upload_candidates(self._h, b0, nb, _ptr(zc), _ptr(has)))

    def upload_uniforms(self, u, b0=0):
        u = _c(u, np.float64)
        if u.ndim != 2:
            raise ValueError("u must be [nb, n_u]")
        L.check(self.lib.ekfslam_upload_uniforms(self._h, b0, u.shape[0], _ptr(u), u.shape[1]))
        self._n_u = u.shape[1]

    def upload_features(self, h=None, Hc=None, S=None, z=None, flags=None, b0=0):
        nb = None
        for a in (h, Hc, S, z, flags):
            if a is not None:
                nb = len(a)
        if nb is None:
            return
        h = None if h is None else _c(h, np.float64, (nb, self.N, 2))
        Hc = None if Hc is None else _c(Hc, np.float64, (nb, self.N, 2, 13))
        S = None if S is None else _c(S, np.float64, (nb, self.N, 2, 2))
        z = None if z is None else _c(z, np.float64, (nb, self.N, 2))
        flags = None if flags is None else _c(flags, np.uint8, (nb, self.N))
        L.check(self.lib.ekfslam_upload_features(self._h, b0, nb, _ptr(h), _ptr(Hc), _ptr(S), _ptr(z), _ptr(flags)))

    def download_features(self, b0=0, nb=None):
        nb = self.B - b0 if nb is None else nb
        out = dict(h=np.empty((nb, self.N, 2)), Hc=np.empty((nb, self.N, 2, 13)), S=np.empty((nb, self.N, 2, 2)),
                   z=np.empty((nb, self.N, 2)), flags=np.empty((nb, self.N), dtype=np.uint8),
                   offs=np.empty((nb, self.N), dtype=np.int32), counters=np.empty((nb, self.N, 2), dtype=np.int32))
        L.check(self.lib.ekfslam_download_features(self._h, b0, nb, _ptr(out["h"]), _ptr(out["Hc"]), _ptr(out["S"]),
                                                   _ptr(out["z"]), _ptr(out["flags"]), _ptr(out["offs"]),
                                                   _ptr(out["counters"])))
        return out

    def download_flags(self, b0=0, nb=None):
        nb = self.B - b0 if nb is None else nb
        flags = np.empty((nb, self.N), dtype=np.uint8)
        L.check(self.lib.ekfslam_download_features(self._h, b0, nb, None, None, None, None, _ptr(flags), None, None))
        return flags

    def download_stats(self, b0=0, nb=None):
        nb = self.B - b0 if nb is None else nb
        st = np.empty((nb, len(L.STATS_FIELDS)), dtype=np.int32)
        L.check(self.lib.ekfslam_download_stats(self._h, b0, nb, _ptr(st)))
        return {k: st[:, i].copy() for i, k in enumerate(L.STATS_FIELDS)}

    # -- map management ("next" rows of SURVEY §8f) ------------------------------------------
    def reset_filters(self, xv=None, Pxv=None, b0=0, nb=None):
        """mc/initialize_x_and_p.m for filters [b0, b0+nb): camera-only state, empty map."""
        nb = self.B - b0 if nb is None else nb
        if xv is None:
            xv = np.array([0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 1e-15, 1e-15, 1e-15], dtype=np.float64)
        if Pxv is None:
            eps = float(np.finfo(np.float64).eps)
            Pxv = np.diag([eps] * 7 + [0.025 ** 2] * 6)
        xv = _c(xv, np.float64, (13,))
        Pxv = _c(Pxv, np.float64, (13, 13))
        L.check(self.lib.ekfslam_reset_filters(self._h, b0, nb, _ptr(xv), _ptr(Pxv)))

    def add_features_inverse_depth(self, uvd, add=None, std_pxl=1.0, initial_rho=1.0, std_rho=1.0, b0=0):
        """mc/add_features_inverse_depth.m: one new inverse-depth feature per filter from uvd [nb,2]."""
        uvd = _c(uvd, np.float64)
        nb = uvd.shape[0]
        uvd = _c(uvd, np.float64, (nb, 2))
        add = None if add is None else _c(add, np.uint8, (nb,))
        L.check(self.lib.ekfslam_add_features(self._h, b0, nb, _ptr(uvd), _ptr(add), float(std_pxl),
                                              float(initial_rho), float(std_rho)))

    def inversedepth_2_cartesian(self, threshold=0.1, force_index=-1):
        """mc/inversedepth_2_cartesian.m for every filter; returns the converted feature index per filter (-1 = none)."""
        conv = np.empty(self.B, dtype=np.int32)
        L.check(self.lib.ekfslam_inversedepth_2_cartesian(self._h, float(threshold), int(force_index), _ptr(conv)))
        return conv

    def delete_features(self, delete, b0=0):
        """mc/delete_a_feature.m for every feature with delete[b, i] != 0."""
        delete = _c(delete, np.uint8)
        nb = delete.shape[0]
        delete = _c(delete, np.uint8, (nb, self.N))
        L.check(self.lib.ekfslam_delete_features(self._h, b0, nb, _ptr(delete)))

    def download_feature_types(self, b0=0, nb=None):
        """(types [nb, N_max] u8, nfeat [nb] i32) — the map layout after conversions / deletions."""
        nb = self.B - b0 if nb is None else nb
        t = np.empty((nb, self.N), dtype=np.uint8)
        nf = np.empty(nb, dtype=np.int32)
        L.check(self.lib.ekfslam_download_feature_types(self._h, b0, nb, _ptr(t), _ptr(nf)))
        return t, nf

    def map_management(self, min_number_of_features_in_image=25):
        """mc/map_management.m:1-35 for every filter on the device (delete -> measured -> update_features_info ->
        at most one inverse-depth -> Cartesian conversion -> top up from the detection list).  Follow it with
        ``step(reset=False)``."""
        L.check(self.lib.ekfslam_map_management(self._h, int(min_number_of_features_in_image)))

    def upload_detections(self, uv, n, tag=None, b0=0):
        """Detection list for map_management: uv [nb,K,2] corner pixels, n [nb] valid entries, tag [nb,K]."""
        uv = _c(uv, np.float64)
        nb, K = uv.shape[0], uv.shape[1]
        uv = _c(uv, np.float64, (nb, K, 2))
        n = _c(n, np.int32, (nb,))
        tag = None if tag is None else _c(tag, np.int32, (nb, K))
        L.check(self.lib.ekfslam_upload_detections(self._h, b0, nb, K, _ptr(uv), _ptr(tag), _ptr(n)))

    def download_detections(self, K, b0=0, nb=None):
        nb = self.B - b0 if nb is None else nb
        uv, tag, n = np.empty((nb, K, 2)), np.empty((nb, K), dtype=np.int32), np.empty(nb, dtype=np.int32)
        L.check(self.lib.ekfslam_download_detections(self._h, b0, nb, K, _ptr(uv), _ptr(tag), _ptr(n)))
        return uv, tag, n

    def upload_feature_meta(self, counters=None, tag=None, b0=0):
        """times_predicted / times_measured [nb,N,2] and the feature identities tag [nb,N]."""
        nb = len(counters) if counters is not None else len(tag)
        counters = None if counters is None else _c(counters, np.int32, (nb, self.N, 2))
        tag = None if tag is None else _c(tag, np.int32, (nb, self.N))
        L.check(self.lib.ekfslam_upload_feature_meta(self._h, b0, nb, _ptr(counters), _ptr(tag)))

    def download_feature_tags(self, b0=0, nb=None):
        nb = self.B - b0 if nb is None else nb
        tag = np.empty((nb, self.N), dtype=np.int32)
        L.check(self.lib.ekfslam_download_feature_tags(self._h, b0, nb, _ptr(tag)))
        return tag

    def download_candidates(self, b0=0, nb=None):
        """The staged candidates of the current frame: zc [nb,N,2], has [nb,N] (0/1)."""
        nb = self.B - b0 if nb is None else nb
        zc, fl = np.empty((nb, self.N, 2)), np.empty((nb, self.N), dtype=np.uint8)
        L.check(self.lib.ekfslam_download_candidates(self._h, b0, nb, _ptr(zc), _ptr(fl)))
        return zc, ((fl & L.F_CAND) != 0).astype(np.uint8)

    # -- synthetic world on the device (stand-in for the image front-end) ---------------------
    def world_upload(self, world, b0=0):
        """world: synth.SynthWorld (filters [b0, b0+B) of it live in this bank)."""
        pts = _c(world.points[b0:b0 + self.B], np.float64, (self.B, world.M, 3))
        poses = np.concatenate([world.pose_r[b0:b0 + self.B], world.pose_q[b0:b0 + self.B]], axis=2)   # [B,T+1,7]
        poses = _c(np.transpose(poses, (1, 0, 2)), np.float64, (world.T + 1, self.B, 7))
        wp = L.WorldParams(seed=world.seed, b_offset=world.b_offset + b0, flaky_mod=world.flaky_mod,
                           noise_px=world.noise_px, gross_px=world.gross_px, p_outlier=world.p_outlier,
                           p_flaky=world.p_flaky, band_px=float(world.BAND))
        L.check(self.lib.ekfslam_world_upload(self._h, world.M, world.T, _ptr(pts), _ptr(poses), C.byref(wp)))

    def world_candidates(self, t):
        L.check(self.lib.ekfslam_world_candidates(self._h, int(t)))

    def world_uniforms(self, t, n_u):
        L.check(self.lib.ekfslam_world_uniforms(self._h, int(t), int(n_u)))
        self._n_u = int(n_u)

    def download_uniforms(self, b0=0, nb=None):
        nb = self.B - b0 if nb is None else nb
        u = np.empty((nb, self._n_u))
        L.check(self.lib.ekfslam_download_uniforms(self._h, b0, nb, _ptr(u), self._n_u))
        return u

    def world_detect(self, t, K):
        L.check(self.lib.ekfslam_world_detect(self._h, int(t), int(K)))

    # -- scoring against the resident ground truth ------------------------------------------------
    def evaluate(self, t):
        """Scores every filter's (x_k_k, P) against frame t of the uploaded world (see ekfslam_evaluate): the frame's
        record replaces the last one and is added into the running totals.  Stream-ordered, no host copies."""
        L.check(self.lib.ekfslam_evaluate(self._h, int(t)))

    def download_eval(self, totals=False, b0=0, nb=None, features=True):
        """{field: [nb] array} of the last frame's records (totals=False) or of the running totals (totals=True);
        float64 for the error / NEES sums, int32 for n_map, n_skip, frames, status.  With totals=False and
        features=True also feat_err [nb, N, 3] and feat_nees [nb, N] (NaN where a slot is empty, has no truth or is
        not evaluable)."""
        nb = self.B - b0 if nb is None else nb
        rec = (L.Eval * nb)()
        fe = fn = None
        if features and not totals:
            fe, fn = np.empty((nb, self.N, 3)), np.empty((nb, self.N))
        L.check(self.lib.ekfslam_download_eval(self._h, b0, nb, 1 if totals else 0, C.cast(rec, C.c_void_p),
                                               _ptr(fe), _ptr(fn)))
        out = {k: np.array([getattr(r, k) for r in rec], dtype=np.float64 if i < 6 else np.int32)
               for i, k in enumerate(L.EVAL_FIELDS)}
        if fe is not None:
            out["feat_err"], out["feat_nees"] = fe, fn
        return out

    def reset_eval(self):
        """Zeroes the running totals."""
        L.check(self.lib.ekfslam_reset_eval(self._h))

    def map_cartesian(self, b0=0, nb=None):
        """The maps in Cartesian coordinates: p [nb, N, 3] and C [nb, N, 3, 3] (NaN for empty and not evaluable
        slots).  Needs no world."""
        nb = self.B - b0 if nb is None else nb
        p, packed = np.empty((nb, self.N, 3)), np.empty((nb, self.N, 6))
        L.check(self.lib.ekfslam_map_cartesian(self._h, b0, nb, _ptr(p), _ptr(packed)))
        C3 = np.empty((nb, self.N, 3, 3))
        for k, (i, j) in enumerate(((0, 0), (1, 0), (1, 1), (2, 0), (2, 1), (2, 2))):
            C3[..., i, j] = packed[..., k]
            C3[..., j, i] = packed[..., k]
        return p, C3

    # -- camera-state measurement update (extension) ---------------------------------------------
    def update_camera(self, H, z, R, on=None, gate=0.0, which=0, b0=0):
        """Linear update of the camera state x[0:13] with m rows z = H x[0:13] + v, v ~ N(0, R), per filter (see
        ekfslam_update_camera).  H [m,13] and R [m,m] are shared by every filter, [nb,m,13] and [nb,m,m] are taken per
        filter; z [nb,m]; on [nb] (None = all).  which=0 updates (x_k_k, P), which=1 (x_k_km1, P); gate <= 0: no
        chi-square gate.  Stream-ordered; the per-filter NIS and status come from download_camera_update()."""
        z = _c(z, np.float64)
        if z.ndim != 2:
            raise ValueError("z must be [nb, m]")
        nb, m = z.shape
        H = np.asarray(H, dtype=np.float64)
        R = np.asarray(R, dtype=np.float64)
        if H.shape == (m, 13):
            H = np.broadcast_to(H, (nb, m, 13))
        if R.shape == (m, m):
            R = np.broadcast_to(R, (nb, m, m))
        H = _c(H, np.float64, (nb, m, 13))
        R = _c(R, np.float64, (nb, m, m))
        on = None if on is None else _c(on, np.uint8, (nb,))
        L.check(self.lib.ekfslam_update_camera(self._h, int(b0), nb, m, _ptr(H), _ptr(z), _ptr(R), _ptr(on),
                                               float(gate), int(which)))

    def download_camera_update(self, b0=0, nb=None):
        """{"nis": float64 [nb], "status": int32 [nb]} of the last update_camera (status: CAM_APPLIED, CAM_OFF,
        CAM_GATED, CAM_NOT_SPD; NIS is NaN for CAM_OFF and CAM_NOT_SPD)."""
        nb = self.B - b0 if nb is None else nb
        nis, st = np.empty(nb), np.empty(nb, dtype=np.int32)
        L.check(self.lib.ekfslam_download_camera_update(self._h, b0, nb, _ptr(nis), _ptr(st)))
        return {"nis": nis, "status": st}

    # -- known-landmark update (extension) ------------------------------------------------------
    def upload_landmarks(self, pts, cov=None, tag=None, nlm=None, b0=0):
        """Landmarks of filters [b0, b0+nb) (see ekfslam_upload_landmarks): pts [nb,L,3] world positions, cov [nb,L,6]
        packed (xx, yx, yy, zx, zy, zz) or [nb,L,3,3] (None: exactly known), tag [nb,L] world points for
        world_landmark_obs (None: -1), nlm [nb] landmarks in use (None: L).  L <= min(LM_MAX, N_max) becomes the
        bank's landmark count."""
        pts = _c(pts, np.float64)
        if pts.ndim != 3 or pts.shape[2] != 3:
            raise ValueError("pts must be [nb, L, 3]")
        nb, Lm = pts.shape[:2]
        if cov is not None:
            cov = np.asarray(cov, dtype=np.float64)
            if cov.shape == (nb, Lm, 3, 3):
                cov = cov[..., [0, 1, 1, 2, 2, 2], [0, 0, 1, 0, 1, 2]]
            cov = _c(cov, np.float64, (nb, Lm, 6))
        tag = None if tag is None else _c(tag, np.int32, (nb, Lm))
        nlm = None if nlm is None else _c(nlm, np.int32, (nb,))
        L.check(self.lib.ekfslam_upload_landmarks(self._h, int(b0), nb, Lm, _ptr(pts), _ptr(cov), _ptr(tag), _ptr(nlm)))
        self._lm_L = Lm

    def upload_landmark_obs(self, uv, has=None, b0=0):
        """This frame's observations: uv [nb,L,2] distorted pixels, has [nb,L] (None: all observed)."""
        uv = _c(uv, np.float64)
        if uv.ndim != 3 or uv.shape[2] != 2:
            raise ValueError("uv must be [nb, L, 2]")
        nb = uv.shape[0]
        if self._lm_L and uv.shape[1] != self._lm_L:
            raise ValueError("uv must have L = %d landmarks" % self._lm_L)
        has = None if has is None else _c(has, np.uint8, uv.shape[:2])
        L.check(self.lib.ekfslam_upload_landmark_obs(self._h, int(b0), nb, _ptr(uv), _ptr(has)))

    def world_landmark_obs(self, t):
        """Synthetic observations of frame t of the uploaded world for the tagged landmarks (stream-ordered)."""
        L.check(self.lib.ekfslam_world_landmark_obs(self._h, int(t)))

    def download_landmark_obs(self, b0=0, nb=None):
        """The staged observations: uv [nb,L,2], has [nb,L] u8."""
        nb = self.B - b0 if nb is None else nb
        uv, has = np.empty((nb, self._lm_L or 1, 2)), np.empty((nb, self._lm_L or 1), dtype=np.uint8)
        L.check(self.lib.ekfslam_download_landmark_obs(self._h, b0, nb, _ptr(uv), _ptr(has)))
        return uv, has

    def update_landmarks(self, std_px, gate=0.0, which=0):
        """Known-landmark update of every filter (see ekfslam_update_landmarks): which=0 updates (x_k_k, P), which=1
        (x_k_km1, P); gate <= 0: no chi-square gate.  Stream-ordered; results from download_landmark_update()."""
        L.check(self.lib.ekfslam_update_landmarks(self._h, float(std_px), float(gate), int(which)))

    def download_landmark_update(self, b0=0, nb=None):
        """{"nis", "k", "status"} [nb] per filter (LMU_*; NIS NaN unless applied) and {"lm_status" [nb,L] (LM_*),
        "lm_h" [nb,L,2], "lm_nis" [nb,L]} per landmark of the last update_landmarks."""
        nb = self.B - b0 if nb is None else nb
        Lm = self._lm_L or 1    # before any upload the call fails with ERR_STATE
        out = {"nis": np.empty(nb), "k": np.empty(nb, dtype=np.int32), "status": np.empty(nb, dtype=np.int32),
               "lm_status": np.empty((nb, Lm), dtype=np.int32), "lm_h": np.empty((nb, Lm, 2)),
               "lm_nis": np.empty((nb, Lm))}
        L.check(self.lib.ekfslam_download_landmark_update(self._h, b0, nb, *(_ptr(out[k]) for k in (
            "nis", "k", "status", "lm_status", "lm_h", "lm_nis"))))
        return out

    # -- stages (names follow the reference functions they replace) --------------------------
    def begin_frame(self):
        L.check(self.lib.ekfslam_begin_frame(self._h))

    def ekf_prediction(self):
        L.check(self.lib.ekfslam_predict(self._h))

    def measure(self, which=1):
        L.check(self.lib.ekfslam_measure(self._h, which))

    def features(self, which=1, parts=3):
        L.check(self.lib.ekfslam_features(self._h, which, parts))

    def hp(self, need=L.F_HAS_H, forbid=0):
        L.check(self.lib.ekfslam_hp(self._h, need, forbid))

    def innovation(self):
        L.check(self.lib.ekfslam_innovation(self._h))

    def gate(self):
        L.check(self.lib.ekfslam_gate(self._h))

    def apply_matches(self):
        L.check(self.lib.ekfslam_apply_matches(self._h))

    def ransac_hypotheses(self):
        L.check(self.lib.ekfslam_ransac(self._h))

    def ekf_update_li_inliers(self):
        L.check(self.lib.ekfslam_update_li(self._h))

    def rescue_hi_inliers(self):
        L.check(self.lib.ekfslam_rescue(self._h))

    def ekf_update_hi_inliers(self):
        L.check(self.lib.ekfslam_update_hi(self._h))

    def update_masked(self, mask, which_prior):
        L.check(self.lib.ekfslam_update_masked(self._h, mask, which_prior))

    def update_iterated(self, mask, which_prior=1, n_iter=3):
        """Iterated EKF update (extension; see ekfslam_update_iterated)."""
        L.check(self.lib.ekfslam_update_iterated(self._h, mask, which_prior, n_iter))

    def step(self, reset=True, match_mode=1, graph=False):
        """One filter step on resident data (mc/mono_slam.m:56-74).  graph=True replays it from a captured CUDA
        graph (latency path; see ekfslam_step_graph)."""
        fn = self.lib.ekfslam_step_graph if graph else self.lib.ekfslam_step
        L.check(fn(self._h, 1 if reset else 0, match_mode))

    def stage_frame(self, d_zc, d_fl, d_u, n_u):
        """Device pointers (ints) of a resident frame, copied into the context's own frame buffers."""
        L.check(self.lib.ekfslam_stage_frame(self._h, C.c_void_p(d_zc), C.c_void_p(d_fl), C.c_void_p(d_u), int(n_u)))
        self._n_u = int(n_u)

    def step_host(self, zc, fl, u, match_mode=1, x_out=None, flags_out=None, stats_out=None):
        """The per-frame call with HOST buffers (pinned buffers make the copies asynchronous).
        zc [B,N,2] f64, fl [B,N] u8, u [B,n_u] f64; outputs are written in place if given."""
        for a, dt in ((zc, np.float64), (fl, np.uint8), (u, np.float64)):
            if a.dtype != dt or not a.flags["C_CONTIGUOUS"]:
                raise ValueError("step_host takes C-contiguous arrays of the exact dtype (no hidden copies)")
        if zc.shape != (self.B, self.N, 2) or fl.shape != (self.B, self.N) or u.ndim != 2 or u.shape[0] != self.B:
            raise ValueError("step_host: bad shapes")
        # the library writes B*n_max doubles, B*N bytes and B stats records straight into these
        for name, a, dt, shape in (("x_out", x_out, np.float64, (self.B, self.n_max)),
                                   ("flags_out", flags_out, np.uint8, (self.B, self.N)),
                                   ("stats_out", stats_out, np.int32, (self.B, len(L.STATS_FIELDS)))):
            if a is None:
                continue
            if not isinstance(a, np.ndarray) or a.dtype != dt or not a.flags["C_CONTIGUOUS"] or \
                    not a.flags["WRITEABLE"] or tuple(a.shape) != shape:
                raise ValueError("step_host: %s must be a writable C-contiguous %s array of shape %s"
                                 % (name, np.dtype(dt).name, shape))
        L.check(self.lib.ekfslam_step_host(self._h, match_mode, _ptr(zc), _ptr(fl), _ptr(u), u.shape[1],
                                           _ptr(x_out), _ptr(flags_out), _ptr(stats_out)))
