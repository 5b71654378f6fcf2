// Camera / quaternion device math of the filter step (fp64).  Each function names the
// reference file it replaces ("mc/" = matlab_code/); the arithmetic is re-derived in
// closed form (no 3x3 inv() calls, shared sub-expressions computed once).
#pragma once
#include "common.cuh"

#define EKF_DEV __device__ __forceinline__

// mc/q2r.m:8-10 — rotation matrix of q = [r x y z] (not assumed unit), row-major R[9]
EKF_DEV void q2r_dev(const double* q, double* R) {
    const double r = q[0], x = q[1], y = q[2], z = q[3];
    R[0] = r * r + x * x - y * y - z * z; R[1] = 2.0 * (x * y - r * z);         R[2] = 2.0 * (z * x + r * y);
    R[3] = 2.0 * (x * y + r * z);         R[4] = r * r - x * x + y * y - z * z; R[5] = 2.0 * (y * z - r * x);
    R[6] = 2.0 * (z * x - r * y);         R[7] = 2.0 * (y * z + r * x);         R[8] = r * r - x * x - y * y + z * z;
}

// mc/normJac.m + mc/update.m:18,24 — J[16] (row-major 4x4) = normJac(q+) of the un-normalised quaternion q+ = x[3..6],
// then q+ <- q+/|q+|.  Thread-0 code of the update epilogues.
EKF_DEV void normjac_normalize(double* x, double* J) {
    const double r = x[3], qx = x[4], qy = x[5], qz = x[6];
    const double nn = r * r + qx * qx + qy * qy + qz * qz;
    const double sc = 1.0 / (nn * sqrt(nn));  // (.)^(-3/2)
    J[0] = sc * (qx * qx + qy * qy + qz * qz); J[1] = sc * (-r * qx); J[2] = sc * (-r * qy); J[3] = sc * (-r * qz);
    J[4] = sc * (-qx * r); J[5] = sc * (r * r + qy * qy + qz * qz); J[6] = sc * (-qx * qy); J[7] = sc * (-qx * qz);
    J[8] = sc * (-qy * r); J[9] = sc * (-qy * qx); J[10] = sc * (r * r + qx * qx + qz * qz); J[11] = sc * (-qy * qz);
    J[12] = sc * (-qz * r); J[13] = sc * (-qz * qx); J[14] = sc * (-qz * qy); J[15] = sc * (r * r + qx * qx + qy * qy);
    const double nrm = sqrt(nn);
    x[3] = r / nrm; x[4] = qx / nrm; x[5] = qy / nrm; x[6] = qz / nrm;
}

// mc/distort_fm.m:22-38 — undistorted pixel -> distorted pixel (10 Newton steps on
// rd + k1 rd^3 + k2 rd^5 = ru).  The loop leaves early once rd reaches a fixed point:
// from there every further step of the reference reproduces the same rd bit for bit.
EKF_DEV void distort_dev(const DevCam& c, double uu, double vu, double& ud, double& vd) {
    const double xu = (uu - c.Cx) * c.dx;
    const double yu = (vu - c.Cy) * c.dy;
    const double ru = sqrt(xu * xu + yu * yu);
    const double ru2 = ru * ru;
    double rd = ru / (1.0 + c.k1 * ru2 + c.k2 * (ru2 * ru2));
#pragma unroll 1
    for (int k = 0; k < 10; ++k) {
        const double rd2 = rd * rd;
        const double rd4 = rd2 * rd2;
        const double f = rd + c.k1 * (rd2 * rd) + c.k2 * (rd4 * rd) - ru;
        const double fp = 1.0 + 3.0 * c.k1 * rd2 + 5.0 * c.k2 * rd4;
        const double rn = rd - f / fp;
        if (rn == rd) break;
        rd = rn;
    }
    const double rd2 = rd * rd;
    const double D = 1.0 + c.k1 * rd2 + c.k2 * (rd2 * rd2);
    ud = (xu / D) / c.dx + c.Cx;
    vd = (yu / D) / c.dy + c.Cy;
}

// mc/jacob_undistor_fm.m:20-34, returned already inverted (mc/calculate_Hi_inverse_depth.m:125-126)
EKF_DEV void dhd_dhu_dev(const DevCam& c, double ud, double vd, double* A /*2x2 row-major*/) {
    const double du = ud - c.Cx, dv = vd - c.Cy;
    const double xd = du * c.dx, yd = dv * c.dy;
    const double rd2 = xd * xd + yd * yd;
    const double rd4 = rd2 * rd2;
    const double g = 1.0 + c.k1 * rd2 + c.k2 * rd4;
    const double e = c.k1 + 2.0 * c.k2 * rd2;
    const double uu_ud = g + du * e * (2.0 * du * c.dx * c.dx);
    const double vu_vd = g + dv * e * (2.0 * dv * c.dy * c.dy);
    const double uu_vd = du * e * (2.0 * dv * c.dy * c.dy);
    const double vu_ud = dv * e * (2.0 * du * c.dx * c.dx);
    const double idet = 1.0 / (uu_ud * vu_vd - uu_vd * vu_ud);
    A[0] = vu_vd * idet;  A[1] = -uu_vd * idet;
    A[2] = -vu_ud * idet; A[3] = uu_ud * idet;
}

// mc/hi_inverse_depth.m:37-43 — field-of-view gate (+-60 deg in both image axes)
EKF_DEV bool fov_reject_dev(double hx, double hy, double hz) {
    const double k = 180.0 / 3.14159265358979323846;
    const double ax = atan2(hx, hz) * k;
    const double ay = atan2(hy, hz) * k;
    return (ax < -60.0) || (ax > 60.0) || (ay < -60.0) || (ay > 60.0);
}

// Predicted measurement of one feature.
//   inverse depth: mc/hi_inverse_depth.m:7-57 (m.m:12-14, hu.m:12-13, distort_fm.m)
//   Cartesian:     mc/hi_cartesian.m:7-49
// y = the feature's state block, xv = camera state.  d (out) = the un-rotated ray
// (y-r)*rho + m  (or y - r), reused by the Jacobian.  Returns visibility.
EKF_DEV bool predict_h_dev(const DevCam& c, const double* xv, const double* R, const double* y, int type,
                           double& hu_out, double& hv_out) {
    double d0, d1, d2;
    if (type == EKFSLAM_FEAT_INVERSEDEPTH) {
        const double theta = y[3], phi = y[4], rho = y[5];
        const double cphi = cos(phi);
        d0 = (y[0] - xv[0]) * rho + cphi * sin(theta);
        d1 = (y[1] - xv[1]) * rho - sin(phi);
        d2 = (y[2] - xv[2]) * rho + cphi * cos(theta);
    } else {
        d0 = y[0] - xv[0]; d1 = y[1] - xv[1]; d2 = y[2] - xv[2];
    }
    // hrl = R' d  (for Cartesian features the reference uses inv(R); identical for unit q
    // up to the positive factor 1/|q|^4, which cancels in the gates and in the projection)
    const double hx = R[0] * d0 + R[3] * d1 + R[6] * d2;
    const double hy = R[1] * d0 + R[4] * d1 + R[7] * d2;
    const double hz = R[2] * d0 + R[5] * d1 + R[8] * d2;
    if (fov_reject_dev(hx, hy, hz)) return false;
    const double uu = c.Cx + (hx / hz) * c.f * (1.0 / c.dx);
    const double vu = c.Cy + (hy / hz) * c.f * (1.0 / c.dy);
    double ud, vd;
    distort_dev(c, uu, vu, ud, vd);
    if ((ud > 0.0) && (ud < c.nCols) && (vd > 0.0) && (vd < c.nRows)) {
        hu_out = ud; hv_out = vd;
        return true;
    }
    return false;
}

// Compact measurement Jacobian of one feature, linearised at pixel (zu,zv) = the stored h.
//   mc/calculate_Hi_inverse_depth.m:20-23,43-156 / mc/calculate_Hi_cartesian.m:20-23,37-113
//   (dRq_times_a_by_dq.m, qconj.m, dqbar_by_dq.m, jacob_undistor_fm.m)
// Hc[0..12] = row u, Hc[13..25] = row v; columns 0-2 d/dr, 3-6 d/dq, 7-12 d/d(feature block).
EKF_DEV void jacobian_dev(const DevCam& c, const double* xv, const double* R, const double* y, int type,
                          double zu, double zv, double* Hc) {
    const double q0 = xv[3], qx = xv[4], qy = xv[5], qz = xv[6];
    const double s = q0 * q0 + qx * qx + qy * qy + qz * qz;
    const double is2 = 1.0 / (s * s);  // inv(q2r(q)) = R' / |q|^4
    double Ri[9];                      // Rrw = inv(R), row-major
    Ri[0] = R[0] * is2; Ri[1] = R[3] * is2; Ri[2] = R[6] * is2;
    Ri[3] = R[1] * is2; Ri[4] = R[4] * is2; Ri[5] = R[7] * is2;
    Ri[6] = R[2] * is2; Ri[7] = R[5] * is2; Ri[8] = R[8] * is2;

    double d0, d1, d2, rho = 1.0, st = 0, ct = 0, sp = 0, cp = 0;
    if (type == EKFSLAM_FEAT_INVERSEDEPTH) {
        rho = y[5];
        sincos(y[3], &st, &ct);
        sincos(y[4], &sp, &cp);
        d0 = (y[0] - xv[0]) * rho + cp * st;
        d1 = (y[1] - xv[1]) * rho - sp;
        d2 = (y[2] - xv[2]) * rho + cp * ct;
    } else {
        d0 = y[0] - xv[0]; d1 = y[1] - xv[1]; d2 = y[2] - xv[2];
    }
    const double hcx = Ri[0] * d0 + Ri[1] * d1 + Ri[2] * d2;
    const double hcy = Ri[3] * d0 + Ri[4] * d1 + Ri[5] * d2;
    const double hcz = Ri[6] * d0 + Ri[7] * d1 + Ri[8] * d2;
    const double fku = c.f * (1.0 / c.dx), fkv = c.f * (1.0 / c.dy);
    // dhu_dhrl (2x3)
    const double a00 = fku / hcz, a02 = -hcx * fku / (hcz * hcz);
    const double a11 = fkv / hcz, a12 = -hcy * fkv / (hcz * hcz);
    double A[4];
    dhd_dhu_dev(c, zu, zv, A);
    // dh_dhrl = A * dhu_dhrl  (2x3)
    double D[6];
    D[0] = A[0] * a00; D[1] = A[1] * a11; D[2] = A[0] * a02 + A[1] * a12;
    D[3] = A[2] * a00; D[4] = A[3] * a11; D[5] = A[2] * a02 + A[3] * a12;
    // E = dh_dhrl * Rrw (2x3): shared by d/dr and d/dy
    double E[6];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int k = 0; k < 3; ++k)
            E[r * 3 + k] = D[r * 3 + 0] * Ri[0 + k] + D[r * 3 + 1] * Ri[3 + k] + D[r * 3 + 2] * Ri[6 + k];
    // d/dq: dRq_times_a_by_dq(qconj(q), d) * diag(1,-1,-1,-1); qconj(q) = [q0,-qx,-qy,-qz]
    {
        const double b0 = q0, bx = -qx, by = -qy, bz = -qz;
        double T[12];  // 3x4 row-major
        // column 0: dR_by_dq0 * d
        T[0] = 2 * b0 * d0 - 2 * bz * d1 + 2 * by * d2;
        T[4] = 2 * bz * d0 + 2 * b0 * d1 - 2 * bx * d2;
        T[8] = -2 * by * d0 + 2 * bx * d1 + 2 * b0 * d2;
        // column 1: dR_by_dqx * d
        T[1] = 2 * bx * d0 + 2 * by * d1 + 2 * bz * d2;
        T[5] = 2 * by * d0 - 2 * bx * d1 - 2 * b0 * d2;
        T[9] = 2 * bz * d0 + 2 * b0 * d1 - 2 * bx * d2;
        // column 2: dR_by_dqy * d
        T[2] = -2 * by * d0 + 2 * bx * d1 + 2 * b0 * d2;
        T[6] = 2 * bx * d0 + 2 * by * d1 + 2 * bz * d2;
        T[10] = -2 * b0 * d0 + 2 * bz * d1 - 2 * by * d2;
        // column 3: dR_by_dqz * d
        T[3] = -2 * bz * d0 - 2 * b0 * d1 + 2 * bx * d2;
        T[7] = 2 * b0 * d0 - 2 * bz * d1 + 2 * by * d2;
        T[11] = 2 * bx * d0 + 2 * by * d1 + 2 * bz * d2;
#pragma unroll
        for (int r = 0; r < 2; ++r) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const double v = D[r * 3 + 0] * T[k] + D[r * 3 + 1] * T[4 + k] + D[r * 3 + 2] * T[8 + k];
                Hc[r * EKF_HC + 3 + k] = (k == 0) ? v : -v;
            }
        }
    }
    if (type == EKFSLAM_FEAT_INVERSEDEPTH) {
        const double w0 = y[0] - xv[0], w1 = y[1] - xv[1], w2 = y[2] - xv[2];
        // dm/dtheta = [cp*ct, 0, -cp*st], dm/dphi = [-sp*st, -cp, -sp*ct]
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const double e0 = E[r * 3 + 0], e1 = E[r * 3 + 1], e2 = E[r * 3 + 2];
            Hc[r * EKF_HC + 0] = -(e0 * rho); Hc[r * EKF_HC + 1] = -(e1 * rho); Hc[r * EKF_HC + 2] = -(e2 * rho);
            Hc[r * EKF_HC + 7] = rho * e0;    Hc[r * EKF_HC + 8] = rho * e1;    Hc[r * EKF_HC + 9] = rho * e2;
            Hc[r * EKF_HC + 10] = e0 * (cp * ct) + e2 * (-cp * st);
            Hc[r * EKF_HC + 11] = e0 * (-sp * st) + e1 * (-cp) + e2 * (-sp * ct);
            Hc[r * EKF_HC + 12] = e0 * w0 + e1 * w1 + e2 * w2;
        }
    } else {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const double e0 = E[r * 3 + 0], e1 = E[r * 3 + 1], e2 = E[r * 3 + 2];
            Hc[r * EKF_HC + 0] = -e0; Hc[r * EKF_HC + 1] = -e1; Hc[r * EKF_HC + 2] = -e2;
            Hc[r * EKF_HC + 7] = e0;  Hc[r * EKF_HC + 8] = e1;  Hc[r * EKF_HC + 9] = e2;
            Hc[r * EKF_HC + 10] = 0.0; Hc[r * EKF_HC + 11] = 0.0; Hc[r * EKF_HC + 12] = 0.0;
        }
    }
}

// Re-projection used inside the RANSAC support count: mc/compute_hypothesis_support_fast.m:17-43
// (inverse depth) / :57-82 (Cartesian).  No visibility gates, rotcw = q2r(q)' (not inv), and the
// pixel is formed as f*ku*h_norm + u0 — the reference's order for this call site.
EKF_DEV double support_residual_dev(const DevCam& c, const double* cam7, const double* R, const double* y, int type,
                                    double zu, double zv) {
    double d0, d1, d2;
    if (type == EKFSLAM_FEAT_INVERSEDEPTH) {
        const double cphi = cos(y[4]);
        d0 = (y[0] - cam7[0]) * y[5] + cphi * sin(y[3]);
        d1 = (y[1] - cam7[1]) * y[5] - sin(y[4]);
        d2 = (y[2] - cam7[2]) * y[5] + cphi * cos(y[3]);
    } else {
        d0 = y[0] - cam7[0]; d1 = y[1] - cam7[1]; d2 = y[2] - cam7[2];
    }
    const double hx = R[0] * d0 + R[3] * d1 + R[6] * d2;
    const double hy = R[1] * d0 + R[4] * d1 + R[7] * d2;
    const double hz = R[2] * d0 + R[5] * d1 + R[8] * d2;
    const double uu = c.fku * (hx / hz) + c.Cx;
    const double vu = c.fkv * (hy / hz) + c.Cy;
    double ud, vd;
    distort_dev(c, uu, vu, ud, vd);
    const double nu0 = zu - ud, nu1 = zv - vd;
    return sqrt(nu0 * nu0 + nu1 * nu1);
}
