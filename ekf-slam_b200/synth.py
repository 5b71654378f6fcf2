"""Synthetic point-field sequences (the reference ships no image sequence — its
``../sequences/ic/rawoutput`` of mc/mono_slam.m:21 is absent — and its matcher needs MATLAB's
Computer Vision Toolbox, mc/matching.m:29-46).

A sequence is: N world points per filter inside the frustum of the first camera, a smooth
camera trajectory, and per frame and feature a candidate pixel
``z = distort(project(truth)) + N(0, noise_px^2)``, replaced with probability ``p_outlier`` by
a gross outlier ``z_true + U(-8, 8)^2``.  The candidates go through the matcher's gating rule
on the device (mc/matching.m:16,38).  Filter b of a batch is seeded with ``seed + b`` so any
sub-range of a batch can be regenerated on its own (multi-GPU sharding).

Everything here is host-side numpy: workload generation, not the filter.  The map of frame 0
is built with the closed form of the reference's sequential augmentation
(mc/add_features_inverse_depth.m:18-22 -> mc/hinv.m:8-26,
mc/add_a_feature_covariance_inverse_depth.m:8-64): with A = [I13; J_1; ...; J_N],
P0 = A Pxv A' + blkdiag(0, D_1..D_N), J_i = dy_dxv, D_i = dy_dhd Padd dy_dhd'.
"""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np

EPS = float(np.finfo(np.float64).eps)


def default_camera():
    """mc/initialize_cam.m:3-25."""
    d = 0.0112
    return SimpleNamespace(k1=6.333e-2, k2=1.390e-2, nRows=240, nCols=320, Cx=1.7945 / d, Cy=1.4433 / d,
                           f=2.1735, dx=d, dy=d, model="two_distortion_parameters",
                           K=np.array([[2.1735 / d, 0, 1.7945 / d], [0, 2.1735 / d, 1.4433 / d], [0, 0, 1.0]]))


# ---------------------------------------------------------------------------- camera model
def quat_to_rot(q):
    """[..., 4] scalar-first quaternion -> [..., 3, 3]."""
    r, x, y, z = q[..., 0], q[..., 1], q[..., 2], q[..., 3]
    R = np.empty(q.shape[:-1] + (3, 3))
    R[..., 0, 0] = r * r + x * x - y * y - z * z
    R[..., 0, 1] = 2 * (x * y - r * z)
    R[..., 0, 2] = 2 * (z * x + r * y)
    R[..., 1, 0] = 2 * (x * y + r * z)
    R[..., 1, 1] = r * r - x * x + y * y - z * z
    R[..., 1, 2] = 2 * (y * z - r * x)
    R[..., 2, 0] = 2 * (z * x - r * y)
    R[..., 2, 1] = 2 * (y * z + r * x)
    R[..., 2, 2] = r * r - x * x - y * y + z * z
    return R


def quat_mul(q, p):
    a, v = q[..., :1], q[..., 1:]
    x, u = p[..., :1], p[..., 1:]
    return np.concatenate([a * x - np.sum(v * u, -1, keepdims=True), a * u + x * v + np.cross(v, u)], -1)


def distort(uv, cam):
    xu = (uv[..., 0] - cam.Cx) * cam.dx
    yu = (uv[..., 1] - cam.Cy) * cam.dy
    ru = np.sqrt(xu * xu + yu * yu)
    rd = ru / (1 + cam.k1 * ru ** 2 + cam.k2 * ru ** 4)
    for _ in range(10):
        f = rd + cam.k1 * rd ** 3 + cam.k2 * rd ** 5 - ru
        fp = 1 + 3 * cam.k1 * rd ** 2 + 5 * cam.k2 * rd ** 4
        rd = rd - f / fp
    D = 1 + cam.k1 * rd ** 2 + cam.k2 * rd ** 4
    return np.stack([xu / D / cam.dx + cam.Cx, yu / D / cam.dy + cam.Cy], -1)


def undistort(uvd, cam):
    xd = (uvd[..., 0] - cam.Cx) * cam.dx
    yd = (uvd[..., 1] - cam.Cy) * cam.dy
    rd2 = xd * xd + yd * yd
    D = 1 + cam.k1 * rd2 + cam.k2 * rd2 * rd2
    return np.stack([xd * D / cam.dx + cam.Cx, yd * D / cam.dy + cam.Cy], -1)


def project(points_w, r, q, cam):
    """points_w [...,N,3], r [...,3], q [...,4] -> distorted pixels [...,N,2] and depth [...,N]."""
    R = quat_to_rot(q)
    d = points_w - r[..., None, :]
    hc = np.einsum("...ji,...nj->...ni", R, d)  # R' d
    fku, fkv = cam.f / cam.dx, cam.f / cam.dy
    uvu = np.stack([cam.Cx + hc[..., 0] / hc[..., 2] * fku, cam.Cy + hc[..., 1] / hc[..., 2] * fkv], -1)
    return distort(uvu, cam), hc[..., 2]


def _undistort_jac(uvd, cam):
    """d(undistorted pixel)/d(distorted pixel), [...,2,2] (mc/jacob_undistor_fm.m:20-34)."""
    du, dv = uvd[..., 0] - cam.Cx, uvd[..., 1] - cam.Cy
    xd, yd = du * cam.dx, dv * cam.dy
    rd2 = xd * xd + yd * yd
    g = 1 + cam.k1 * rd2 + cam.k2 * rd2 * rd2
    e = cam.k1 + 2 * cam.k2 * rd2
    J = np.empty(uvd.shape[:-1] + (2, 2))
    J[..., 0, 0] = g + du * e * (2 * du * cam.dx * cam.dx)
    J[..., 1, 1] = g + dv * e * (2 * dv * cam.dy * cam.dy)
    J[..., 0, 1] = du * e * (2 * dv * cam.dy * cam.dy)
    J[..., 1, 0] = dv * e * (2 * du * cam.dx * cam.dx)
    return J


def _dRq_times_a_by_dq(q, a):
    """[...,3,4]: d(R(q) a)/dq for q [...,4], a [...,3] (mc/dRq_times_a_by_dq.m)."""
    q0, qx, qy, qz = (q[..., i] for i in range(4))
    a0, a1, a2 = (a[..., i] for i in range(3))
    out = np.empty(a.shape[:-1] + (3, 4))
    out[..., 0, 0] = 2 * q0 * a0 - 2 * qz * a1 + 2 * qy * a2
    out[..., 1, 0] = 2 * qz * a0 + 2 * q0 * a1 - 2 * qx * a2
    out[..., 2, 0] = -2 * qy * a0 + 2 * qx * a1 + 2 * q0 * a2
    out[..., 0, 1] = 2 * qx * a0 + 2 * qy * a1 + 2 * qz * a2
    out[..., 1, 1] = 2 * qy * a0 - 2 * qx * a1 - 2 * q0 * a2
    out[..., 2, 1] = 2 * qz * a0 + 2 * q0 * a1 - 2 * qx * a2
    out[..., 0, 2] = -2 * qy * a0 + 2 * qx * a1 + 2 * q0 * a2
    out[..., 1, 2] = 2 * qx * a0 + 2 * qy * a1 + 2 * qz * a2
    out[..., 2, 2] = -2 * q0 * a0 + 2 * qz * a1 - 2 * qy * a2
    out[..., 0, 3] = -2 * qz * a0 - 2 * q0 * a1 + 2 * qx * a2
    out[..., 1, 3] = 2 * q0 * a0 - 2 * qz * a1 + 2 * qy * a2
    out[..., 2, 3] = 2 * qx * a0 + 2 * qy * a1 + 2 * qz * a2
    return out


def initial_map(xv, Pxv, uvd, cam, std_pxl=1.0, initial_rho=1.0, std_rho=1.0):
    """Batched frame-0 map: xv [B,13], Pxv [B,13,13], uvd [B,N,2] -> x [B,n], P [B,n,n] with
    all N features inverse-depth (closed form of the reference's sequential augmentation)."""
    B, N = uvd.shape[:2]
    n = 13 + 6 * N
    fku, fkv = cam.f / cam.dx, cam.f / cam.dy
    q = xv[:, None, 3:7]
    R = quat_to_rot(xv[:, 3:7])                                    # [B,3,3]
    uvu = undistort(uvd, cam)
    hc = np.stack([-(cam.Cx - uvu[..., 0]) / fku, -(cam.Cy - uvu[..., 1]) / fkv, np.ones((B, N))], -1)
    nw = np.einsum("bij,bnj->bni", R, hc)                          # mc/hinv.m:21
    nx, ny, nz = nw[..., 0], nw[..., 1], nw[..., 2]
    x = np.zeros((B, n))
    x[:, :13] = xv
    feat = x[:, 13:].reshape(B, N, 6)
    feat[..., 0:3] = xv[:, None, 0:3]
    feat[..., 3] = np.arctan2(nx, nz)
    feat[..., 4] = np.arctan2(-ny, np.sqrt(nx * nx + nz * nz))
    feat[..., 5] = initial_rho
    # Jacobians (mc/add_a_feature_covariance_inverse_depth.m:28-49)
    xz2 = nx * nx + nz * nz
    n2 = xz2 + ny * ny
    dth = np.stack([nz / xz2, np.zeros_like(nx), -nx / xz2], -1)                  # [B,N,3]
    dph = np.stack([nx * ny / (n2 * np.sqrt(xz2)), -np.sqrt(xz2) / n2, nz * ny / (n2 * np.sqrt(xz2))], -1)
    dgw_dq = _dRq_times_a_by_dq(np.broadcast_to(q, (B, N, 4)), hc)               # [B,N,3,4]
    J = np.zeros((B, N, 6, 13))                                                  # dy_dxv
    J[..., 0, 0] = J[..., 1, 1] = J[..., 2, 2] = 1.0
    J[..., 3, 3:7] = np.einsum("bni,bnij->bnj", dth, dgw_dq)
    J[..., 4, 3:7] = np.einsum("bni,bnij->bnj", dph, dgw_dq)
    dyp_dgw = np.zeros((B, N, 5, 3))
    dyp_dgw[..., 3, :] = dth
    dyp_dgw[..., 4, :] = dph
    dgc_dhu = np.array([[1 / fku, 0.0], [0.0, 1 / fkv], [0.0, 0.0]])
    dhu_dhd = _undistort_jac(uvd, cam)
    dyp_dhd = np.einsum("bnij,bjk,kl,bnlm->bnim", dyp_dgw, R, dgc_dhu, dhu_dhd)  # [B,N,5,2]
    dy_dhd = np.zeros((B, N, 6, 3))
    dy_dhd[..., 0:5, 0:2] = dyp_dhd
    dy_dhd[..., 5, 2] = 1.0
    Padd = np.diag([std_pxl ** 2, std_pxl ** 2, std_rho ** 2])
    D = np.einsum("bnij,jk,bnlk->bnil", dy_dhd, Padd, dy_dhd)                     # [B,N,6,6]
    A = np.zeros((B, n, 13))
    A[:, :13, :] = np.eye(13)
    A[:, 13:, :] = J.reshape(B, 6 * N, 13)
    P = np.matmul(np.matmul(A, Pxv), np.transpose(A, (0, 2, 1)))
    P = 0.5 * (P + np.transpose(P, (0, 2, 1)))
    for i in range(N):
        s = 13 + 6 * i
        P[:, s:s + 6, s:s + 6] += D[:, i]
    return x, P


def convert_to_cartesian(x, P, types, which):
    """mc/inversedepth_2_cartesian.m:35-45 applied at once to the inverse-depth features listed in
    ``which`` of ONE filter (x [n], P [n,n], types [N] uint8).  Returns new (x, P, types)."""
    types = np.array(types, dtype=np.uint8)
    offs = []
    pos = 13
    for t in types:
        offs.append(pos)
        pos += 6 if t == 1 else 3
    n_old = pos
    rows = []
    newx = [x[:13]]
    Jall_blocks = []
    for i, t in enumerate(types):
        o = offs[i]
        if t == 1 and i in set(which):
            th, ph, rho = x[o + 3], x[o + 4], x[o + 5]
            mi = np.array([np.cos(ph) * np.sin(th), -np.sin(ph), np.cos(ph) * np.cos(th)])
            newx.append(x[o:o + 3] + mi / rho)
            J = np.zeros((3, 6))
            J[:, :3] = np.eye(3)
            J[:, 3] = (1 / rho) * np.array([np.cos(ph) * np.cos(th), 0.0, -np.cos(ph) * np.sin(th)])
            J[:, 4] = (1 / rho) * np.array([-np.sin(ph) * np.sin(th), -np.cos(ph), -np.sin(ph) * np.cos(th)])
            J[:, 5] = -mi / rho ** 2
            Jall_blocks.append((o, J))
            types[i] = 2
        else:
            w = 6 if t == 1 else 3
            newx.append(x[o:o + w])
            Jall_blocks.append((o, np.eye(w)))
    n_new = 13 + sum(b[1].shape[0] for b in Jall_blocks)
    Jall = np.zeros((n_new, n_old))
    Jall[:13, :13] = np.eye(13)
    r = 13
    for o, J in Jall_blocks:
        Jall[r:r + J.shape[0], o:o + J.shape[1]] = J
        r += J.shape[0]
    return np.concatenate(newx), Jall @ P @ Jall.T, types


# ---------------------------------------------------------------------------- sequences
class SynthSequence:
    """T frames of candidate measurements for B filters x N features (all generated up front).

    Filter b draws everything from ``RandomState(seed + b_offset + b)`` in a fixed order, so a
    shard [b0, b0+nb) of a larger batch is reproduced by ``b_offset=b0`` (multi-GPU partitioning).
    """

    def __init__(self, B, N, T, seed=0, b_offset=0, p_outlier=0.2, noise_px=0.5, cam=None,
                 depth_range=(2.0, 10.0), margin_px=45.0, n_u=64):
        self.B, self.N, self.T, self.n_u = B, N, T, n_u
        self.seed, self.b_offset, self.p_outlier, self.noise_px = int(seed), int(b_offset), float(p_outlier), float(noise_px)
        self.cam = cam or default_camera()
        cam = self.cam
        T1 = T + 1
        self.seeds = np.arange(B) + seed + b_offset
        uv = np.empty((B, N, 2))
        depth = np.empty((B, N))
        v = np.empty((B, 3))
        w = np.empty((B, 3))
        dv = np.empty((B, T1, 3))
        dw = np.empty((B, T1, 3))
        noise = np.empty((B, T1, N, 2))
        out = np.empty((B, T1, N), dtype=bool)
        gross = np.empty((B, T1, N, 2))
        self.U = np.empty((B, T1, n_u))
        for b in range(B):
            rng = np.random.RandomState(int(self.seeds[b]) % (2 ** 32))
            uv[b, :, 0] = rng.uniform(margin_px, cam.nCols - margin_px, N)
            uv[b, :, 1] = rng.uniform(margin_px, cam.nRows - margin_px, N)
            depth[b] = rng.uniform(depth_range[0], depth_range[1], N)
            vv = rng.uniform(-1, 1, 3)
            v[b] = vv / np.linalg.norm(vv) * rng.uniform(0.01, 0.03)
            ww = rng.uniform(-1, 1, 3)
            w[b] = ww / np.linalg.norm(ww) * rng.uniform(0.005, 0.02)
            dv[b] = rng.normal(0, 0.002, (T1, 3))
            dw[b] = rng.normal(0, 0.002, (T1, 3))
            noise[b] = rng.normal(0, noise_px, (T1, N, 2))
            out[b] = rng.uniform(size=(T1, N)) < p_outlier
            gross[b] = rng.uniform(-8, 8, (T1, N, 2))
            self.U[b] = rng.rand(T1, n_u)
        fku, fkv = cam.f / cam.dx, cam.f / cam.dy
        # world points: a distorted pixel inside the image margin, back-projected at a depth
        uvu = undistort(uv, cam)
        ray = np.stack([(uvu[..., 0] - cam.Cx) / fku, (uvu[..., 1] - cam.Cy) / fkv, np.ones((B, N))], -1)
        self.points = ray * depth[..., None]
        # smooth trajectory: slowly varying velocity / angular velocity (never exactly zero)
        self.pose_r = np.empty((B, T1, 3))
        self.pose_q = np.empty((B, T1, 4))
        r = np.zeros((B, 3))
        q = np.tile(np.array([1.0, 0, 0, 0]), (B, 1))
        for t in range(T1):
            self.pose_r[:, t] = r
            self.pose_q[:, t] = q
            # weak springs towards the initial pose keep the points in view over long sequences
            v = v + dv[:, t] - 0.02 * r
            w = np.clip(w + dw[:, t] - 0.04 * (2.0 * q[:, 1:4]), -0.02, 0.02)
            r = r + v
            th = np.linalg.norm(w, axis=1, keepdims=True)
            dq = np.concatenate([np.cos(th / 2), np.sin(th / 2) * w / th], axis=1)
            q = quat_mul(q, dq)
            q = q / np.linalg.norm(q, axis=1, keepdims=True)
        zt, dep = project(self.points[:, None], self.pose_r, self.pose_q, cam)      # [B,T1,N,2]
        out[:, 0] = False  # the initialisation frame is clean
        z = np.where(out[..., None], zt + gross, zt + noise)
        vis = (dep > 0) & (zt[..., 0] > 0) & (zt[..., 0] < cam.nCols) & (zt[..., 1] > 0) & (zt[..., 1] < cam.nRows)
        self.zc = np.ascontiguousarray(np.transpose(z, (1, 0, 2, 3)))               # [T1,B,N,2]
        self.has = np.ascontiguousarray(np.transpose(vis, (1, 0, 2))).astype(np.uint8)
        self.is_outlier = np.ascontiguousarray(np.transpose(out, (1, 0, 2)))

    @property
    def n(self):
        return 13 + 6 * self.N

    def initial_state(self, b0=0, nb=None, std_pxl=1.0):
        """x0 [nb,n], P0 [nb,n,n], types [nb,N] — features initialised from the frame-0 pixels."""
        nb = self.B - b0 if nb is None else nb
        xv = np.tile(np.array([0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 1e-15, 1e-15, 1e-15], dtype=np.float64), (nb, 1))
        Pxv = np.zeros((nb, 13, 13))
        for i in range(7):
            Pxv[:, i, i] = EPS
        for i in range(7, 13):
            Pxv[:, i, i] = 0.025 ** 2
        x, P = initial_map(xv, Pxv, self.zc[0, b0:b0 + nb], self.cam, std_pxl=std_pxl)
        return x, P, np.ones((nb, self.N), dtype=np.uint8)

    def truth_world(self):
        """The sequence's own ground truth as a world for ``FilterBank.world_upload``: M = N points (world point k is
        feature k, so ``upload_feature_meta(tag=arange(N))`` lets ``FilterBank.evaluate`` score the filters) and the
        T+1 true poses.  Candidates the device world draws from it follow this sequence's noise model (pixel noise,
        U(-8, 8) gross outliers with probability p_outlier), not its draws."""
        return SimpleNamespace(points=self.points, pose_r=self.pose_r, pose_q=self.pose_q, M=self.N, T=self.T,
                               seed=self.seed, b_offset=self.b_offset, flaky_mod=1, noise_px=self.noise_px,
                               gross_px=8.0, p_outlier=self.p_outlier, p_flaky=self.p_outlier, BAND=SynthWorld.BAND)

    def frame(self, t):
        """Candidates of frame t (1..T): zc [B,N,2], has [B,N] u8."""
        return self.zc[t], self.has[t]

    def uniforms(self, t, n_u=None):
        """RANSAC uniform stream of frame t: u [B, n_u] (the first n_u of the stored stream)."""
        n_u = self.n_u if n_u is None else n_u
        if n_u > self.n_u:
            raise ValueError("sequence was generated with n_u=%d" % self.n_u)
        return np.ascontiguousarray(self.U[:, t, :n_u])


# ---------------------------------------------------------------------------- closed-loop world
# A persistent synthetic WORLD (as opposed to SynthSequence's pre-drawn candidate arrays): M world
# points per filter, a camera trajectory, and counter-based noise, so that candidate pixels for the
# features currently in the map (whatever map management did to it) and corner detections for new
# features can be produced per frame — on the device by k_synth_candidates / k_synth_detect
# (csrc/k_map.cu), and here in numpy as their mirror.  A feature's identity is its world-point id,
# carried in the per-feature `tag` (the stand-in for features_info(i).feature_when_initialized,
# mc/add_feature_to_info_vector.m:10, which the reference's matcher uses to recognise a feature).
_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)
_GOLD = np.uint64(0x9E3779B97F4A7C15)


def _mix64(x):
    x = np.asarray(x, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = x ^ (x >> np.uint64(30))
        x = x * np.uint64(0xBF58476D1CE4E5B9)
        x = x ^ (x >> np.uint64(27))
        x = x * np.uint64(0x94D049BB133111EB)
        x = x ^ (x >> np.uint64(31))
    return x


def world_uniform(seed, b, t, w, c):
    """Counter-based uniform in [0,1): key (seed, filter b, frame t, world point w, channel c).
    Same integer arithmetic as `world_u01` in csrc/k_map.cu."""
    with np.errstate(over="ignore"):
        k = _mix64(np.uint64(seed) + _GOLD * (np.asarray(b, dtype=np.uint64) + np.uint64(1)))
        k = _mix64(k + np.asarray(t, dtype=np.uint64))
        k = _mix64(k + np.asarray(w, dtype=np.uint64))
        k = _mix64(k + np.asarray(c, dtype=np.uint64))
    return (k >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


class SynthWorld:
    """M world points per filter, T+1 camera poses, counter-based measurement noise.

    points [B,M,3], pose_r [B,T+1,3], pose_q [B,T+1,4].  World point w of filter b is *flaky* when
    w % flaky_mod == flaky_mod - 1: its candidate is a gross outlier with probability p_flaky (such
    features get deleted by the rule of `delete_features`).
    """
    BAND = 22   # excluded image band for new features (mc/initialize_a_feature.m:8: half patch 20 + 1)

    def __init__(self, B, M, T, seed=0, b_offset=0, p_outlier=0.2, noise_px=0.5, gross_px=8.0, p_flaky=0.8,
                 flaky_mod=7, cam=None, depth_range=(2.0, 10.0), spread_px=80.0, speed=(0.01, 0.03), spring=0.02):
        self.B, self.M, self.T = B, M, T
        self.seed, self.b_offset = int(seed), int(b_offset)
        self.p_outlier, self.noise_px, self.gross_px = float(p_outlier), float(noise_px), float(gross_px)
        self.p_flaky, self.flaky_mod = float(p_flaky), int(flaky_mod)
        self.cam = cam or default_camera()
        cam = self.cam
        T1 = T + 1
        uv = np.empty((B, M, 2))
        depth = np.empty((B, M))
        self.pose_r = np.empty((B, T1, 3))
        self.pose_q = np.empty((B, T1, 4))
        # undistorted-pixel extent of the image (the wide-angle lens pulls a much larger field into view)
        ext = undistort(np.array([[0.0, 0.0], [float(cam.nCols), float(cam.nRows)]]), cam)
        for b in range(B):
            rng = np.random.RandomState((self.seed + self.b_offset + b) % (2 ** 32))
            # points spread over a field wider than the image so that features enter and leave the view
            uv[b, :, 0] = rng.uniform(ext[0, 0] - spread_px, ext[1, 0] + spread_px, M)
            uv[b, :, 1] = rng.uniform(ext[0, 1] - spread_px, ext[1, 1] + spread_px, M)
            depth[b] = rng.uniform(depth_range[0], depth_range[1], M)
            vv = rng.uniform(-1, 1, 3)
            v = vv / np.linalg.norm(vv) * rng.uniform(speed[0], speed[1])
            ww = rng.uniform(-1, 1, 3)
            w = ww / np.linalg.norm(ww) * rng.uniform(0.003, 0.01)
            dv = rng.normal(0, 0.002, (T1, 3))
            dw = rng.normal(0, 0.001, (T1, 3))
            r = np.zeros(3)
            q = np.array([1.0, 0, 0, 0])
            for t in range(T1):
                self.pose_r[b, t] = r
                self.pose_q[b, t] = q
                v = v + dv[t] - spring * r
                w = np.clip(w + dw[t] - 0.04 * (2.0 * q[1:4]), -0.02, 0.02)
                r = r + v
                th = np.linalg.norm(w)
                dq = np.concatenate([[np.cos(th / 2)], np.sin(th / 2) * w / th])
                q = quat_mul(q, dq)
                q = q / np.linalg.norm(q)
        fku, fkv = cam.f / cam.dx, cam.f / cam.dy
        ray = np.stack([(uv[..., 0] - cam.Cx) / fku, (uv[..., 1] - cam.Cy) / fkv, np.ones((B, M))], -1)
        self.points = ray * depth[..., None]

    # -- what a camera at frame t sees ----------------------------------------------------------
    def truth_pixels(self, t):
        """zt [B,M,2] distorted pixels of all world points at the true pose of frame t, vis [B,M]."""
        zt, dep = project(self.points, self.pose_r[:, t], self.pose_q[:, t], self.cam)
        cam = self.cam
        with np.errstate(invalid="ignore"):
            vis = (dep > 0) & (zt[..., 0] > 0) & (zt[..., 0] < cam.nCols) & (zt[..., 1] > 0) & (zt[..., 1] < cam.nRows)
        return zt, vis

    def _noise(self, b, t, w):
        u = [world_uniform(self.seed, b + self.b_offset, t, w, c) for c in range(6)]
        rad = np.sqrt(-2.0 * np.log(1.0 - u[1]))
        n0, n1 = rad * np.cos(2.0 * np.pi * u[2]), rad * np.sin(2.0 * np.pi * u[2])
        return u, n0, n1

    def candidates(self, t, tags, nfeat):
        """Candidate pixels at frame t for the features of the current maps.
        tags [B,N] world ids, nfeat [B].  Returns zc [B,N,2], has [B,N] u8 (numpy mirror of
        k_synth_candidates)."""
        B, N = tags.shape
        zt, vis = self.truth_pixels(t)
        zc = np.zeros((B, N, 2))
        has = np.zeros((B, N), dtype=np.uint8)
        for b in range(B):
            k = int(nfeat[b])
            if k == 0:
                continue
            w = tags[b, :k].astype(np.int64)
            u, n0, n1 = self._noise(b, t, w)
            p_out = np.where(w % self.flaky_mod == self.flaky_mod - 1, self.p_flaky, self.p_outlier)
            out = u[0] < p_out
            zg = zt[b, w] + np.stack([(2 * u[3] - 1), (2 * u[4] - 1)], -1) * self.gross_px
            zn = zt[b, w] + np.stack([n0, n1], -1) * self.noise_px
            zc[b, :k] = np.where(out[:, None], zg, zn)
            has[b, :k] = vis[b, w]
            zc[b, :k][~vis[b, w]] = 0.0
        return zc, has

    def uniforms(self, t, n_u):
        """RANSAC uniform stream of frame t, [B, n_u] — bit-identical to k_synth_uniforms (integer hash, exact scaling)."""
        b = (np.arange(self.B) + self.b_offset)[:, None]
        return world_uniform(self.seed, b, t, np.arange(n_u)[None, :], 7)

    def detections(self, t, tags, nfeat, K):
        """Corner detections for new features in the image of frame t: the first K world points (by id)
        that are visible inside the excluded band and not yet in the map, at integer pixels (FAST corners
        are integer locations).  Returns uv [B,K,2], tag [B,K] (-1 = unused), n [B] (mirror of
        k_synth_detect)."""
        B = tags.shape[0]
        zt, vis = self.truth_pixels(t)
        cam = self.cam
        uv = np.zeros((B, K, 2))
        tg = np.full((B, K), -1, dtype=np.int32)
        n = np.zeros(B, dtype=np.int32)
        for b in range(B):
            have = set(int(x) for x in tags[b, :int(nfeat[b])])
            for w in range(self.M):
                if n[b] >= K:
                    break
                if not vis[b, w] or w in have:
                    continue
                u, n0, n1 = self._noise(b, t, w)
                px = np.floor(zt[b, w] + np.array([n0, n1]) * self.noise_px + 0.5)
                if px[0] < self.BAND or px[0] > cam.nCols - self.BAND or px[1] < self.BAND or px[1] > cam.nRows - self.BAND:
                    continue
                uv[b, n[b]] = px
                tg[b, n[b]] = w
                n[b] += 1
        return uv, tg, n
