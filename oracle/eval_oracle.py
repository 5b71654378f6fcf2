"""numpy restatement of the scoring against the ground truth (csrc/k_eval.cu, ekfslam_evaluate / ekfslam_map_cartesian).

Test infrastructure: it works on one filter's downloaded state (x, P, feature types, tags) plus the world, with the
definitions of include/ekfslam.h and the kernel's loop and summation orders (Cholesky column by column, sums over the
evaluable features in feature order).  P is read through its lower triangle, which the device treats as authoritative.
"""
from __future__ import annotations

import math

import numpy as np

from oracle.ekf_oracle import dq3_by_dq1

FIELDS = ["pos_sq_err", "rot_sq_err", "nees_pos", "nees_pose", "map_sq_err", "map_nees",
          "n_map", "n_skip", "frames", "status"]
CAM_NOT_SPD, NO_TRUTH, NOT_EVALUABLE = 1, 2, 4


def sym_lower(P):
    """The symmetric matrix whose lower triangle is that of P."""
    L = np.tril(P)
    return L + np.tril(L, -1).T


def chol_nees(C, e):
    """e' inv(C) e through C = L L', in the kernel's order; None when a pivot C_jj - sum_k L_jk^2 is not > 0."""
    n = len(e)
    L = np.zeros((n, n))
    for j in range(n):
        d = C[j, j]
        for k in range(j):
            d -= L[j, k] * L[j, k]
        if not d > 0.0:
            return None
        L[j, j] = math.sqrt(d)
        for i in range(j + 1, n):
            s = C[i, j]
            for k in range(j):
                s -= L[i, k] * L[j, k]
            L[i, j] = s / L[j, j]
    y = np.zeros(n)
    acc = 0.0
    for i in range(n):
        s = e[i]
        for k in range(i):
            s -= L[i, k] * y[k]
        y[i] = s / L[i, i]
        acc += y[i] * y[i]
    return acc


def qconj(q):
    return np.array([q[0], -q[1], -q[2], -q[3]])


def camera(x, P, r_t, q_t):
    """Camera errors against the true pose (r_t, q_t): dict with e_r, e_theta, angle, J (6x7), C_pose, nees_pos,
    nees_pose (NaN where the Cholesky fails) and spd."""
    x = np.asarray(x, dtype=np.float64)
    e_r = x[0:3] - r_t
    QL = dq3_by_dq1(qconj(q_t))          # left-multiplication matrix of conj(q_t)
    d = QL @ x[3:7]                      # conj(q_t) * q_hat, not renormalised
    s = -1.0 if d[0] < 0.0 else 1.0
    e_th = 2.0 * s * d[1:4]
    angle = 2.0 * math.atan2(math.sqrt(d[1] * d[1] + d[2] * d[2] + d[3] * d[3]), abs(d[0]))
    J = np.zeros((6, 7))
    J[0:3, 0:3] = np.eye(3)
    J[3:6, 3:7] = 2.0 * s * QL[1:4, :]
    P7 = sym_lower(np.asarray(P)[0:7, 0:7])
    C_pose = J @ P7 @ J.T
    e = np.concatenate([e_r, e_th])
    nees_pos = chol_nees(P7[0:3, 0:3], e_r)
    nees_pose = chol_nees(C_pose, e)
    return dict(e_r=e_r, e_theta=e_th, angle=angle, J=J, C_pose=C_pose,
                nees_pos=math.nan if nees_pos is None else nees_pos,
                nees_pose=math.nan if nees_pose is None else nees_pose,
                spd=nees_pos is not None and nees_pose is not None)


def feature_cartesian(y, ftype):
    """(p, J_f) of one feature block: inverse depth [x y z theta phi rho] (mc/inversedepth_2_cartesian.m:37-45) or
    Cartesian [X Y Z] (J_f = I).  None when rho <= 0."""
    y = np.asarray(y, dtype=np.float64)
    if ftype == 2:
        return y[0:3].copy(), np.eye(3)
    th, ph, rho = y[3], y[4], y[5]
    if not rho > 0.0:
        return None
    st, ct, sp, cp = math.sin(th), math.cos(th), math.sin(ph), math.cos(ph)
    m = np.array([cp * st, -sp, cp * ct])
    ir = 1.0 / rho
    J = np.zeros((3, 6))
    J[:, 0:3] = np.eye(3)
    J[:, 3] = ir * np.array([cp * ct, 0.0, -cp * st])
    J[:, 4] = ir * np.array([-sp * st, -cp, -sp * ct])
    J[:, 5] = -m / (rho * rho)
    return y[0:3] + ir * m, J


def offsets(types, nfeat):
    offs, pos = [], 13
    for i in range(int(nfeat)):
        offs.append(pos)
        pos += 6 if types[i] == 1 else 3
    return offs


def _feature(x, P, types, i, off):
    w = 6 if types[i] == 1 else 3
    r = feature_cartesian(x[off:off + w], types[i])
    if r is None:
        return None
    p, J = r
    C = J @ sym_lower(np.asarray(P)[off:off + w, off:off + w]) @ J.T
    return p, C


def map_cartesian(x, P, types, nfeat, N):
    """p [N,3], C [N,3,3] of every slot; NaN for empty and not evaluable slots."""
    p_out = np.full((N, 3), np.nan)
    C_out = np.full((N, 3, 3), np.nan)
    for i, off in enumerate(offsets(types, nfeat)):
        r = _feature(x, P, types, i, off)
        if r is None or chol_nees(r[1], np.zeros(3)) is None:
            continue
        p_out[i], C_out[i] = r
    return p_out, C_out


def evaluate(x, P, types, nfeat, tags, points, r_t, q_t, N=None):
    """The record of one filter at one frame plus feat_err [N,3] and feat_nees [N] (NaN where a slot is empty, has
    no truth or is not evaluable).  points [M,3] = the filter's world points."""
    N = len(types) if N is None else N
    M = len(points)
    cam = camera(x, P, r_t, q_t)
    rec = dict(pos_sq_err=float(cam["e_r"] @ cam["e_r"]), rot_sq_err=cam["angle"] ** 2,
               nees_pos=cam["nees_pos"], nees_pose=cam["nees_pose"], map_sq_err=0.0, map_nees=0.0,
               n_map=0, n_skip=0, frames=1, status=0 if cam["spd"] else CAM_NOT_SPD)
    feat_err = np.full((N, 3), np.nan)
    feat_nees = np.full(N, np.nan)
    for i, off in enumerate(offsets(types, nfeat)):
        tg = int(tags[i])
        if tg < 0 or tg >= M:
            rec["n_skip"] += 1
            rec["status"] |= NO_TRUTH
            continue
        r = _feature(x, P, types, i, off)
        nees = None
        if r is not None:
            e = r[0] - points[tg]
            nees = chol_nees(r[1], e)
        if nees is None:
            rec["n_skip"] += 1
            rec["status"] |= NOT_EVALUABLE
            continue
        feat_err[i], feat_nees[i] = e, nees
        rec["n_map"] += 1
        rec["map_sq_err"] += float(e[0] * e[0] + e[1] * e[1] + e[2] * e[2])
        rec["map_nees"] += nees
    return rec, feat_err, feat_nees
