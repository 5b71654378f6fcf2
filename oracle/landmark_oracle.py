"""CPU mirror (numpy fp64) of the known-landmark update, ekfslam_update_landmarks.

TEST INFRASTRUCTURE ONLY, like ekf_oracle.  The definition is that of include/ekfslam.h (DESIGN.md §3.5): a landmark is
a Cartesian point outside the state; its prediction is ``ekf_oracle.hi_cartesian`` (mc/hi_cartesian.m:7-49), its
Jacobian the (r, q) and point columns of ``ekf_oracle.calculate_Hi_cartesian`` (mc/calculate_Hi_cartesian.m, linearised
at the predicted pixel as in the reference), R_j = std^2 I + J_p C_j J_p', the individual chi-square gate of
mc/rescue_hi_inliers.m, and the stacked update ``ekf_oracle.update`` (mc/update.m:3-32) with H = [A | 0] and the
block-diagonal R.
"""
import math

import numpy as np

from oracle import ekf_oracle as O

LM_USED, LM_NOT_OBSERVED, LM_NOT_VISIBLE, LM_GATED, LM_NOT_SPD, LM_ABSENT = 0, 1, 2, 3, 4, 5
LMU_APPLIED, LMU_NONE, LMU_NOT_SPD = 0, 1, 2


def unpack_cov(c6):
    """(xx, yx, yy, zx, zy, zz) -> 3x3."""
    xx, yx, yy, zx, zy, zz = c6
    return np.array([[xx, yx, zx], [yx, yy, zy], [zx, zy, zz]])


def predict(xv, p, cam):
    """h (2,) of landmark p seen from camera state xv[0:7], or None when not visible (mc/hi_cartesian.m)."""
    return O.hi_cartesian(np.asarray(p, dtype=np.float64), xv[0:3], O.q2r(xv[3:7]), cam)


def jacobians(xv, p, cam, h):
    """A (2x7: d/dr, d/dq) and J_p (2x3: d/dp) of mc/calculate_Hi_cartesian.m, linearised at pixel h."""
    f = O.Feature(type="cartesian", h=np.asarray(h, dtype=np.float64))
    Hi = O.calculate_Hi_cartesian(xv[0:13], np.asarray(p, dtype=np.float64), cam, 0, [f])   # [2, 16], point at 13
    return Hi[:, 0:7], Hi[:, 13:16]


def _chol2_nis(S, nu):
    """Individual NIS through the 2x2 Cholesky factor; None when S is not SPD (a pivot not > 0)."""
    if not S[0, 0] > 0.0:
        return None
    l00 = math.sqrt(S[0, 0])
    l10 = S[1, 0] / l00
    d = S[1, 1] - l10 * l10
    if not d > 0.0:
        return None
    y0 = nu[0] / l00
    y1 = (nu[1] - l10 * y0) / math.sqrt(d)
    return y0 * y0 + y1 * y1


def landmark_update(x, P, cam, pts, uv, has, nlm, std_px, gate=0.0, cov=None):
    """One filter's update.  x [n], P [n,n]; pts [L,3], uv [L,2], has [L], cov [L,6] or None.
    Returns dict(x, P, nis, k, status, lm_status [L], lm_h [L,2], lm_nis [L]); x and P are copies of the inputs
    unless the status is LMU_APPLIED."""
    x = np.asarray(x, dtype=np.float64)
    P = np.asarray(P, dtype=np.float64)
    Lm = len(pts)
    lm_status = np.full(Lm, LM_ABSENT, dtype=np.int32)
    lm_h = np.full((Lm, 2), np.nan)
    lm_nis = np.full(Lm, np.nan)
    rows, R_blocks, z, h = [], [], [], []
    for j in range(min(int(nlm), Lm)):
        if not has[j]:
            lm_status[j] = LM_NOT_OBSERVED
            continue
        hj = predict(x, pts[j], cam)
        if hj is None:
            lm_status[j] = LM_NOT_VISIBLE
            continue
        lm_h[j] = hj
        A, Jp = jacobians(x, pts[j], cam, hj)
        Rj = std_px ** 2 * np.eye(2)
        if cov is not None:
            Rj = Rj + Jp @ unpack_cov(cov[j]) @ Jp.T
        Sj = A @ P[0:7, 0:7] @ A.T + Rj
        nu = np.asarray(uv[j], dtype=np.float64) - hj
        nis_j = _chol2_nis(Sj, nu)
        if nis_j is None:
            lm_status[j] = LM_NOT_SPD
            continue
        lm_nis[j] = nis_j
        if gate > 0 and not nis_j < gate:
            lm_status[j] = LM_GATED
            continue
        lm_status[j] = LM_USED
        rows.append(A)
        R_blocks.append(Rj)
        z.append(np.asarray(uv[j], dtype=np.float64))
        h.append(hj)
    out = dict(x=x.copy(), P=P.copy(), nis=np.nan, k=2 * len(rows), status=LMU_NONE, lm_status=lm_status, lm_h=lm_h,
               lm_nis=lm_nis)
    if not rows:
        return out
    k = 2 * len(rows)
    H = np.zeros((k, len(x)))
    H[:, 0:7] = np.vstack(rows)
    R = np.zeros((k, k))
    for i, Rj in enumerate(R_blocks):
        R[2 * i:2 * i + 2, 2 * i:2 * i + 2] = Rj
    z, h = np.concatenate(z), np.concatenate(h)
    S = H @ P @ H.T + R
    try:
        np.linalg.cholesky(S)
    except np.linalg.LinAlgError:
        out["status"] = LMU_NOT_SPD
        return out
    nis = float((z - h) @ np.linalg.solve(S, z - h))
    if not np.isfinite(nis):
        out["status"] = LMU_NOT_SPD
        return out
    xo, Po, _ = O.update(x, P, H, R, z, h)
    out.update(x=xo, P=Po, nis=nis, status=LMU_APPLIED)
    return out
