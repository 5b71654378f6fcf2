// Known-landmark update (ekfslam_update_landmarks): pixel observations of points with known world coordinates, the
// landmarks outside the state.  The definition is that of include/ekfslam.h: per landmark the Cartesian prediction and
// Jacobian of the feature model (predict_h_dev / jacobian_dev, mc/hi_cartesian.m, mc/calculate_Hi_cartesian.m), its
// own R_j = std^2 I + J_p C_j J_p' and chi-square gate; the used landmarks stacked as H = [A | 0] and mc/update.m:3-32
// computed the way the feature updates compute it.  This kernel forms W, x+, q normalisation and normJac; the
// covariance downdate is the feature updates' own (launch_downdate, k_downdate.cu), which reads ktot[b] = k rows of W
// and jn[b].
#include <math.h>
#include <math_constants.h>

#include "model.cuh"

#define LM_THREADS 128
#define LM_ROWS (2 * EKFSLAM_LM_MAX)

// One block per filter.
//   1. the 7x7 (r, q) block of P and x[0:7] in shared memory; warp 0, a lane per landmark slot: prediction, Jacobian,
//      R_j, S_j, nu_j, the 2x2 Cholesky factor, the individual NIS and the gate; a ballot gives the stacked rows
//      (landmark order) and k.
//   2. warp 0, a lane per stacked row: S = A Pc A' + blkdiag(R_j), its Cholesky factor L, inv(L), M = inv(L) A (k x 7),
//      y = inv(L) nu and NIS = |y|^2, and the status.
//   3. a thread per state column c < ld: W[:, c] = M P[0:7, c] from the coalesced rows 0..6 (P is exactly symmetric in
//      memory; with k up to 32, folding inv(L) into the 7 columns of A keeps a thread's registers at 7 column values
//      instead of k entries of H P), padding columns [n, ld) written as zero, x[c] += sum_a W[a][c] y[a].
//   4. normJac(q+) from the un-normalised quaternion, q+ <- q+/|q+|, rows a < k of W get columns 3..6 <- . Jt'
//      (w_fold_jt), jn[b] = Jt, ktot[b] = k.
// A filter whose status is not applied ends with ktot[b] = 0 (the downdate skips it) and its state is not written.
__global__ void __launch_bounds__(LM_THREADS) k_lm_update(DevView v, DevCam cam, DevLm lm, double std_px, double gate,
                                                          int which) {
    const int b = blockIdx.x, tid = threadIdx.x, ld = v.ld;
    const int n = v.nstate[b];
    double* __restrict__ x = (which ? v.xp : v.x) + (size_t)b * ld;
    const double* __restrict__ P = v.P + (size_t)b * v.nmax * ld;
    double* __restrict__ W = v.W + (size_t)b * v.wstride;
    __shared__ double Pc[7][8];
    __shared__ double As[LM_ROWS][8];             // stacked A rows (r, q columns)
    __shared__ double Ts[LM_ROWS][8];             // A Pc, then M = inv(L) A
    __shared__ double Ls[LM_ROWS][LM_ROWS + 1];   // S, then L (lower)
    __shared__ double Li[LM_ROWS][LM_ROWS + 1];   // inv(L) (lower)
    __shared__ double Rb[LM_ROWS][2];             // row a of its landmark's 2x2 R_j
    __shared__ double nu[LM_ROWS], ys[LM_ROWS], xs[7], Jt[16];
    __shared__ int s_k, s_status;
    for (int e = tid; e < 49; e += blockDim.x) {
        const int r = e / 7, cc = e - r * 7;
        Pc[r][cc] = (cc <= r) ? P[(size_t)r * ld + cc] : P[(size_t)cc * ld + r];   // the lower triangle is authoritative
    }
    if (tid < 7) xs[tid] = x[tid];
    __syncthreads();
    if (tid < 32) {
        const int lane = tid, j = lane;
        const size_t e = (size_t)b * EKFSLAM_LM_MAX + j;
        bool used = false;
        int st = EKFSLAM_LM_ABSENT;
        double hu = CUDART_NAN, hv = CUDART_NAN, nis_j = CUDART_NAN;
        double A[2][7], R00 = 0.0, R10 = 0.0, R11 = 0.0, nu0 = 0.0, nu1 = 0.0;
        if (j < EKFSLAM_LM_MAX && j < lm.nlm[b]) {
            st = EKFSLAM_LM_NOT_OBSERVED;
            if (lm.has[e]) {
                st = EKFSLAM_LM_NOT_VISIBLE;
                double Rq[9], p[3];
                q2r_dev(xs + 3, Rq);
                p[0] = lm.p[3 * e]; p[1] = lm.p[3 * e + 1]; p[2] = lm.p[3 * e + 2];
                double pu, pv;
                if (predict_h_dev(cam, xs, Rq, p, EKFSLAM_FEAT_CARTESIAN, pu, pv)) {
                    hu = pu; hv = pv;
                    double Hc[2 * EKF_HC];
                    jacobian_dev(cam, xs, Rq, p, EKFSLAM_FEAT_CARTESIAN, hu, hv, Hc);
#pragma unroll
                    for (int r = 0; r < 2; ++r)
#pragma unroll
                        for (int c = 0; c < 7; ++c) A[r][c] = Hc[r * EKF_HC + c];
                    // R_j = std^2 I + J_p C J_p'  (J_p = columns 7..9)
                    const double* Cp = lm.C + 6 * e;
                    const double C3[3][3] = {{Cp[0], Cp[1], Cp[3]}, {Cp[1], Cp[2], Cp[4]}, {Cp[3], Cp[4], Cp[5]}};
                    double JC[2][3];
#pragma unroll
                    for (int r = 0; r < 2; ++r)
#pragma unroll
                        for (int c = 0; c < 3; ++c)
                            JC[r][c] = Hc[r * EKF_HC + 7] * C3[0][c] + Hc[r * EKF_HC + 8] * C3[1][c] + Hc[r * EKF_HC + 9] * C3[2][c];
                    const double s2 = std_px * std_px;
                    R00 = s2 + (JC[0][0] * Hc[7] + JC[0][1] * Hc[8] + JC[0][2] * Hc[9]);
                    R10 = JC[1][0] * Hc[7] + JC[1][1] * Hc[8] + JC[1][2] * Hc[9];
                    R11 = s2 + (JC[1][0] * Hc[EKF_HC + 7] + JC[1][1] * Hc[EKF_HC + 8] + JC[1][2] * Hc[EKF_HC + 9]);
                    // S_j = A Pc A' + R_j
                    double T[2][7];
#pragma unroll
                    for (int r = 0; r < 2; ++r)
#pragma unroll
                        for (int c = 0; c < 7; ++c) {
                            double s = 0.0;
#pragma unroll
                            for (int k = 0; k < 7; ++k) s += A[r][k] * Pc[k][c];
                            T[r][c] = s;
                        }
                    double S00 = 0.0, S10 = 0.0, S11 = 0.0;
#pragma unroll
                    for (int k = 0; k < 7; ++k) {
                        S00 += T[0][k] * A[0][k];
                        S10 += T[1][k] * A[0][k];
                        S11 += T[1][k] * A[1][k];
                    }
                    S00 += R00; S10 += R10; S11 += R11;
                    nu0 = lm.uv[2 * e] - hu;
                    nu1 = lm.uv[2 * e + 1] - hv;
                    st = EKFSLAM_LM_NOT_SPD;
                    if (S00 > 0.0) {
                        const double l00 = sqrt(S00), l10 = S10 / l00, d = S11 - l10 * l10;
                        if (d > 0.0) {
                            const double y0 = nu0 / l00, y1 = (nu1 - l10 * y0) / sqrt(d);
                            nis_j = y0 * y0 + y1 * y1;
                            used = !(gate > 0.0) || nis_j < gate;
                            st = used ? EKFSLAM_LM_USED : EKFSLAM_LM_GATED;
                        }
                    }
                }
            }
        }
        const unsigned mask = __ballot_sync(0xffffffffu, used);
        if (j < EKFSLAM_LM_MAX) {
            lm.lm_status[e] = st;
            lm.lm_h[2 * e] = hu;
            lm.lm_h[2 * e + 1] = hv;
            lm.lm_nis[e] = nis_j;
        }
        if (used) {
            const int a = 2 * __popc(mask & ((1u << j) - 1u));
#pragma unroll
            for (int c = 0; c < 7; ++c) { As[a][c] = A[0][c]; As[a + 1][c] = A[1][c]; }
            Rb[a][0] = R00; Rb[a][1] = R10;
            Rb[a + 1][0] = R10; Rb[a + 1][1] = R11;
            nu[a] = nu0; nu[a + 1] = nu1;
        }
        const int k = 2 * __popc(mask);
        __syncwarp();
        for (int e2 = lane; e2 < k * 7; e2 += 32) {   // T = A Pc
            const int a = e2 / 7, r = e2 - a * 7;
            double s = 0.0;
#pragma unroll
            for (int q = 0; q < 7; ++q) s += As[a][q] * Pc[q][r];
            Ts[a][r] = s;
        }
        __syncwarp();
        for (int e2 = lane; e2 < k * k; e2 += 32) {   // S = T A' + blkdiag(R_j) (lower triangle)
            const int a = e2 / k, t = e2 - a * k;
            if (t > a) continue;
            double s = 0.0;
#pragma unroll
            for (int q = 0; q < 7; ++q) s += Ts[a][q] * As[t][q];
            Ls[a][t] = ((a >> 1) == (t >> 1)) ? s + Rb[a][t & 1] : s;
        }
        __syncwarp();
        // Cholesky, left-looking by columns: lane i >= j forms S(i,j) - sum_q<j L(i,q) L(j,q)
        bool ok = true;
        for (int c = 0; c < k; ++c) {
            double s = 0.0;
            if (lane >= c && lane < k) {
                s = Ls[lane][c];
                for (int q = 0; q < c; ++q) s -= Ls[lane][q] * Ls[c][q];
            }
            const double d = __shfl_sync(0xffffffffu, s, c);
            ok = ok && (d > 0.0);
            const double lcc = sqrt(d);
            if (lane == c) Ls[c][c] = lcc;
            else if (lane > c && lane < k) Ls[lane][c] = s / lcc;
            __syncwarp();
        }
        if (lane < k) {                                  // column `lane` of inv(L) by forward substitution
            const int t = lane;
            Li[t][t] = 1.0 / Ls[t][t];
            for (int a = t + 1; a < k; ++a) {
                double s = 0.0;
                for (int q = t; q < a; ++q) s += Ls[a][q] * Li[q][t];
                Li[a][t] = -s / Ls[a][a];
            }
        }
        __syncwarp();
        if (lane < k) {                                  // y = inv(L) nu, M = inv(L) A (row `lane`)
            double s = 0.0, mr[7] = {0, 0, 0, 0, 0, 0, 0};
            for (int t = 0; t <= lane; ++t) {
                const double l = Li[lane][t];
                s += l * nu[t];
#pragma unroll
                for (int c = 0; c < 7; ++c) mr[c] += l * As[t][c];
            }
            ys[lane] = s;
#pragma unroll
            for (int c = 0; c < 7; ++c) Ts[lane][c] = mr[c];
        }
        __syncwarp();
        if (lane == 0) {
            double nis = 0.0;
            for (int a = 0; a < k; ++a) nis += ys[a] * ys[a];
            int s = EKFSLAM_LMU_APPLIED;
            if (k == 0) s = EKFSLAM_LMU_NONE;
            else if (!ok || !isfinite(nis)) s = EKFSLAM_LMU_NOT_SPD;
            lm.status[b] = s;
            lm.k[b] = k;
            lm.nis[b] = (s == EKFSLAM_LMU_APPLIED) ? nis : CUDART_NAN;
            if (s != EKFSLAM_LMU_APPLIED) v.ktot[b] = 0;
            s_status = s;
            s_k = k;
        }
    }
    __syncthreads();
    if (s_status != EKFSLAM_LMU_APPLIED) return;
    const int k = s_k;
    for (int c = tid; c < ld; c += blockDim.x) {
        const bool incol = c < n;
        double pc[7];
#pragma unroll
        for (int r = 0; r < 7; ++r) pc[r] = incol ? P[(size_t)r * ld + c] : 0.0;
        double* __restrict__ wcol = W + w_at(v.wrows, 0, c);
        double xa = 0.0;
        for (int a = 0; a < k; ++a) {
            double s = 0.0;
#pragma unroll
            for (int r = 0; r < 7; ++r) s += Ts[a][r] * pc[r];
            wcol[(size_t)a * EKF_WPAD] = incol ? s : 0.0;   // the padding columns [n, ld) are kept zero
            xa += s * ys[a];
        }
        if (incol) x[c] += xa;
    }
    __syncthreads();
    if (tid == 0) normjac_normalize(x, Jt);
    __syncthreads();
    if (tid < k) w_fold_jt(W + w_at(v.wrows, tid, 3), Jt);
    if (tid < 16) v.jn[(size_t)b * 16 + tid] = Jt[tid];
    if (tid == 0) v.ktot[b] = k;
}

void launch_lm_update(ekfslam_ctx* c, double std_px, double gate, int which) {
    {
        KScope ks(c, KT_LM_UPDATE);
        k_lm_update<<<c->v.B, LM_THREADS, 0, c->stream>>>(c->v, c->cam, c->lm, std_px, gate, which);
    }
    launch_downdate(c, KT_DOWNDATE_LM);
}
