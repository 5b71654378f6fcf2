// Camera-state measurement update (ekfslam_update_camera): m <= 13 rows z = H x[0:13] + v, v ~ N(0, R), per filter.
// The definition is that of include/ekfslam.h: mc/update.m:3-32 with the full Jacobian [H | 0], computed the way the
// feature updates compute it (S = L L', W = inv(L) H P, x+ = x + W' y with y = inv(L) nu, P+ = J P J' - (W J')'(W J')).
// This kernel forms W, x+, q normalisation and normJac; the covariance downdate is the feature updates' own
// (launch_downdate, k_downdate.cu), which reads ktot[b] = m rows of W and jn[b].
#include <math.h>
#include <math_constants.h>

#include "model.cuh"

#define CU_THREADS 128

// One block per filter.
//   1. H, z, R and the 13x13 camera block of P in shared memory; warp 0 forms S = H Pcc H' + R, its Cholesky factor L,
//      inv(L), nu = z - H x, y = inv(L) nu and NIS = |y|^2, and decides the status.
//   2. a thread per state column c < ld: g = H P[0:13, c] from the coalesced rows 0..12 (P is exactly symmetric in
//      memory), W[:, c] = inv(L) g (padding columns [n, ld) written as zero), x[c] += sum_a W[a][c] y[a].
//   3. normJac(q+) from the un-normalised quaternion, q+ <- q+/|q+| (mc/update.m:18,24), rows a < m of W get columns
//      3..6 <- . Jt' (w_fold_jt, as in k_wfix), jn[b] = Jt, ktot[b] = m.
// A filter whose status is not 0 ends with ktot[b] = 0 (the downdate skips it) and is not written.
__global__ void __launch_bounds__(CU_THREADS) k_cam_update(DevView v, DevCamUpd cu, int which) {
    const int b = blockIdx.x;
    const int m = cu.m, ld = v.ld, tid = threadIdx.x;
    const bool sel = b >= cu.b0 && b < cu.b0 + cu.nb && cu.on[b] != 0;
    if (!sel) {
        if (tid == 0) { cu.status[b] = EKFSLAM_CAM_OFF; cu.nis[b] = CUDART_NAN; v.ktot[b] = 0; }
        return;
    }
    const int n = v.nstate[b];
    double* __restrict__ x = (which ? v.xp : v.x) + (size_t)b * ld;
    const double* __restrict__ P = v.P + (size_t)b * v.nmax * ld;
    double* __restrict__ W = v.W + (size_t)b * v.wstride;
    __shared__ double Pc[EKF_XV][EKF_XV + 1];
    __shared__ double Hs[EKF_XV][EKF_XV + 1];
    __shared__ double Ts[EKF_XV][EKF_XV + 1];   // H Pcc
    __shared__ double Ls[EKF_XV][EKF_XV + 1];   // S, then L (lower)
    __shared__ double Li[EKF_XV][EKF_XV + 1];   // inv(L) (lower, zeros above)
    __shared__ double nu[EKF_XV], ys[EKF_XV], xs[EKF_XV], Jt[16];
    __shared__ int s_status;
    const double* __restrict__ Hg = cu.H + (size_t)b * m * EKF_XV;
    const double* __restrict__ Rg = cu.R + (size_t)b * m * m;
    for (int e = tid; e < EKF_XV * EKF_XV; e += blockDim.x) {
        const int r = e / EKF_XV, cc = e - r * EKF_XV;
        Pc[r][cc] = (cc <= r) ? P[(size_t)r * ld + cc] : P[(size_t)cc * ld + r];   // the lower triangle is authoritative
        Hs[r][cc] = (r < m) ? Hg[e] : 0.0;
        Ls[r][cc] = (r < m && cc <= r) ? Rg[r * m + cc] : 0.0;
    }
    if (tid < EKF_XV) xs[tid] = x[tid];
    if (tid < m) nu[tid] = cu.z[(size_t)b * m + tid];
    __syncthreads();
    if (tid < 32) {
        const int lane = tid;
        for (int e = lane; e < m * EKF_XV; e += 32) {   // T = H Pcc
            const int a = e / EKF_XV, r = e - a * EKF_XV;
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < EKF_XV; ++k) s += Hs[a][k] * Pc[k][r];
            Ts[a][r] = s;
        }
        __syncwarp();
        for (int e = lane; e < m * m; e += 32) {        // S = T H' + R (lower triangle)
            const int a = e / m, t = e - a * m;
            if (t > a) continue;
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < EKF_XV; ++k) s += Ts[a][k] * Hs[t][k];
            Ls[a][t] = s + Ls[a][t];
        }
        if (lane < m) {                                  // nu = z - H x
            double h = 0.0;
#pragma unroll
            for (int k = 0; k < EKF_XV; ++k) h += Hs[lane][k] * xs[k];
            nu[lane] = nu[lane] - h;
        }
        __syncwarp();
        // Cholesky, left-looking by columns: lane i >= j forms S(i,j) - sum_k<j L(i,k) L(j,k)
        bool ok = true;
        for (int j = 0; j < m; ++j) {
            double s = 0.0;
            if (lane >= j && lane < m) {
                s = Ls[lane][j];
                for (int k = 0; k < j; ++k) s -= Ls[lane][k] * Ls[j][k];
            }
            const double d = __shfl_sync(0xffffffffu, s, j);
            ok = ok && (d > 0.0);
            const double ljj = sqrt(d);
            if (lane == j) Ls[j][j] = ljj;
            else if (lane > j && lane < m) Ls[lane][j] = s / ljj;
            __syncwarp();
        }
        if (lane < m) {                                  // column `lane` of inv(L) by forward substitution
            const int t = lane;
            for (int a = 0; a < EKF_XV; ++a) Li[a][t] = 0.0;
            Li[t][t] = 1.0 / Ls[t][t];
            for (int a = t + 1; a < m; ++a) {
                double s = 0.0;
                for (int k = t; k < a; ++k) s += Ls[a][k] * Li[k][t];
                Li[a][t] = -s / Ls[a][a];
            }
        }
        __syncwarp();
        if (lane < m) {                                  // y = inv(L) nu
            double s = 0.0;
            for (int t = 0; t <= lane; ++t) s += Li[lane][t] * nu[t];
            ys[lane] = s;
        }
        __syncwarp();
        if (lane == 0) {
            double nis = 0.0;
            for (int a = 0; a < m; ++a) nis += ys[a] * ys[a];
            int st = EKFSLAM_CAM_APPLIED;
            if (!ok || !isfinite(nis)) st = EKFSLAM_CAM_NOT_SPD;
            else if (cu.gate > 0.0 && nis > cu.gate) st = EKFSLAM_CAM_GATED;
            cu.status[b] = st;
            cu.nis[b] = (st == EKFSLAM_CAM_NOT_SPD) ? CUDART_NAN : nis;
            if (st != EKFSLAM_CAM_APPLIED) v.ktot[b] = 0;
            s_status = st;
        }
    }
    __syncthreads();
    if (s_status != EKFSLAM_CAM_APPLIED) return;
    double yr[EKF_XV];
#pragma unroll
    for (int a = 0; a < EKF_XV; ++a) yr[a] = (a < m) ? ys[a] : 0.0;
    for (int c = tid; c < ld; c += blockDim.x) {
        const bool incol = c < n;
        double pc[EKF_XV];
#pragma unroll
        for (int r = 0; r < EKF_XV; ++r) pc[r] = incol ? P[(size_t)r * ld + c] : 0.0;
        double g[EKF_XV];
#pragma unroll
        for (int a = 0; a < EKF_XV; ++a) {
            double s = 0.0;
            if (a < m) {
#pragma unroll
                for (int r = 0; r < EKF_XV; ++r) s += Hs[a][r] * pc[r];
            }
            g[a] = s;
        }
        double* __restrict__ wcol = W + w_at(v.wrows, 0, c);
        double xa = 0.0;
#pragma unroll
        for (int a = 0; a < EKF_XV; ++a) {
            if (a < m) {
                double s = 0.0;
#pragma unroll
                for (int t = 0; t <= a; ++t) s += Li[a][t] * g[t];
                wcol[(size_t)a * EKF_WPAD] = incol ? s : 0.0;   // the padding columns [n, ld) are kept zero
                xa += s * yr[a];
            }
        }
        if (incol) x[c] += xa;
    }
    __syncthreads();
    if (tid == 0) normjac_normalize(x, Jt);
    __syncthreads();
    if (tid < m) w_fold_jt(W + w_at(v.wrows, tid, 3), Jt);
    if (tid < 16) v.jn[(size_t)b * 16 + tid] = Jt[tid];
    if (tid == 0) v.ktot[b] = m;
}

void launch_cam_update(ekfslam_ctx* c, int which) {
    {
        KScope ks(c, KT_CAM_UPDATE);
        k_cam_update<<<c->v.B, CU_THREADS, 0, c->stream>>>(c->v, c->cu, which);
    }
    launch_downdate(c, KT_DOWNDATE_CAM);
}
