// Scoring every filter against the resident ground truth (ekfslam_evaluate) and the Cartesian map export
// (ekfslam_map_cartesian).  The definitions are those of include/ekfslam.h; oracle/eval_oracle.py restates them in numpy
// with the same loop and summation orders.  Read-only on the filter: the kernel writes only the DevEval buffers.
#include <math.h>
#include <math_constants.h>

#include "model.cuh"

#define EV_THREADS 128   // (EV_THREADS, 2): 144 registers, no spills; the 40-byte stack frame is the sincos slow path

// per-slot outcome, kept in shared memory for the fixed-order reduction
enum { EV_OK = 0, EV_NO_TRUTH = 1, EV_BAD = 2, EV_EMPTY = 3 };

// nees = e' inv(A) e through A = L L'.  A: packed lower triangle of an n x n matrix, A[i(i+1)/2 + j] = A(i, j), j <= i,
// overwritten by L.  Returns false (nees untouched) when a pivot A(j,j) - sum_k L(j,k)^2 is not > 0.  Every loop has a
// compile-time trip count (triangular bounds as guards) and there is no early exit, so A stays in registers.
#define EV_TRI(i, j) ((i) * ((i) + 1) / 2 + (j))
template <int n>
EKF_DEV bool chol_nees(double* A, const double* e, double& nees) {
    bool ok = true;
#pragma unroll
    for (int j = 0; j < n; ++j) {
        double d = A[EV_TRI(j, j)];
#pragma unroll
        for (int k = 0; k < n; ++k)
            if (k < j) d -= A[EV_TRI(j, k)] * A[EV_TRI(j, k)];
        ok = ok && (d > 0.0);
        const double ljj = sqrt(d);
        A[EV_TRI(j, j)] = ljj;
#pragma unroll
        for (int i = 0; i < n; ++i) {
            if (i > j) {
                double s = A[EV_TRI(i, j)];
#pragma unroll
                for (int k = 0; k < n; ++k)
                    if (k < j) s -= A[EV_TRI(i, k)] * A[EV_TRI(j, k)];
                A[EV_TRI(i, j)] = s / ljj;
            }
        }
    }
    double y[n];
    double acc = 0.0;
#pragma unroll
    for (int i = 0; i < n; ++i) {
        double s = e[i];
#pragma unroll
        for (int k = 0; k < n; ++k)
            if (k < i) s -= A[EV_TRI(i, k)] * y[k];
        y[i] = s / A[EV_TRI(i, i)];
        acc += y[i] * y[i];
    }
    if (ok) nees = acc;
    return ok;
}

// Cartesian position p and its covariance C (packed lower: xx, yx, yy, zx, zy, zz) of the feature block at state offset
// `off`.  The diagonal block of P is gathered like k_innov_gather does it: one short row segment of the authoritative
// lower triangle per block row, each element requested once.  Returns false when rho <= 0 (inverse depth).
EKF_DEV bool feature_cartesian(const double* __restrict__ x, const double* __restrict__ P, int ld, int off, int type,
                               double* p, double* C) {
    if (type == EKFSLAM_FEAT_CARTESIAN) {
        p[0] = x[off]; p[1] = x[off + 1]; p[2] = x[off + 2];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int cc = 0; cc <= r; ++cc) C[r * (r + 1) / 2 + cc] = P[(size_t)(off + r) * ld + off + cc];
        return true;
    }
    double L[21];   // L[r(r+1)/2 + c] = P(off + r, off + c), c <= r
#pragma unroll
    for (int r = 0; r < 6; ++r) {
        const double* __restrict__ prow = P + (size_t)(off + r) * ld + off;
#pragma unroll
        for (int cc = 0; cc <= r; ++cc) L[r * (r + 1) / 2 + cc] = prow[cc];
    }
    const double th = x[off + 3], ph = x[off + 4], rho = x[off + 5];
    if (!(rho > 0.0)) return false;
    double st, ct, sp, cp;
    sincos(th, &st, &ct);
    sincos(ph, &sp, &cp);
    // mc/inversedepth_2_cartesian.m:37-45, in the order of k_id2cart
    const double m[3] = {cp * st, -sp, cp * ct};
    const double dmt[3] = {cp * ct, 0.0, -cp * st};
    const double dmp[3] = {-sp * st, -cp, -sp * ct};
    const double ir = 1.0 / rho;
    double J[3][6];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        p[r] = x[off + r] + ir * m[r];
        J[r][0] = (r == 0) ? 1.0 : 0.0; J[r][1] = (r == 1) ? 1.0 : 0.0; J[r][2] = (r == 2) ? 1.0 : 0.0;
        J[r][3] = ir * dmt[r];
        J[r][4] = ir * dmp[r];
        J[r][5] = -m[r] / (rho * rho);
    }
    // T = J P_ff (3x6), C = T J' (lower triangle)
    double T[3][6];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int cc = 0; cc < 6; ++cc) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < 6; ++k) s += J[a][k] * ((k >= cc) ? L[k * (k + 1) / 2 + cc] : L[cc * (cc + 1) / 2 + k]);
            T[a][cc] = s;
        }
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int bb = 0; bb <= a; ++bb) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < 6; ++k) s += T[a][k] * J[bb][k];
            C[a * (a + 1) / 2 + bb] = s;
        }
    return true;
}

// The camera part (one thread): errors and NEES of the (r, q) estimate against the true pose (rt, qt).  Pc: the 7x7
// camera block of P, packed lower.  Returns the status bit 0 when a Cholesky pivot is not > 0.
EKF_DEV int camera_eval(const double* xv, const double* rt, const double* qt, const double* Pc, ekfslam_eval& rec) {
    const double er[3] = {xv[0] - rt[0], xv[1] - rt[1], xv[2] - rt[2]};
    // Q_L(conj(q_t)), rows 1..3 (left-multiplication matrix, dq3_by_dq1 of the oracle)
    const double a = qt[0], b = -qt[1], c = -qt[2], d = -qt[3];
    const double QL[4][4] = {{a, -b, -c, -d}, {b, a, -d, c}, {c, d, a, -b}, {d, -c, b, a}};
    double dl[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) dl[i] = QL[i][0] * xv[3] + QL[i][1] * xv[4] + QL[i][2] * xv[5] + QL[i][3] * xv[6];
    const double s = (dl[0] < 0.0) ? -1.0 : 1.0;
    double e[6] = {er[0], er[1], er[2], 2.0 * s * dl[1], 2.0 * s * dl[2], 2.0 * s * dl[3]};
    const double nv = sqrt(dl[1] * dl[1] + dl[2] * dl[2] + dl[3] * dl[3]);
    const double ang = 2.0 * atan2(nv, fabs(dl[0]));
    rec.pos_sq_err = er[0] * er[0] + er[1] * er[1] + er[2] * er[2];
    rec.rot_sq_err = ang * ang;
    int status = 0;
    // position: P_rr
    double A3[6] = {Pc[0], Pc[1], Pc[2], Pc[3], Pc[4], Pc[5]};
    double nees = 0.0;
    if (chol_nees<3>(A3, er, nees)) rec.nees_pos = nees;
    else { rec.nees_pos = CUDART_NAN; status = 1; }
    // pose: C_pose = J P J', J = blockdiag(I3, 2 s E Q_L) (6x7)
    double J[6][7];
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int k = 0; k < 7; ++k) J[r][k] = 0.0;
    J[0][0] = 1.0; J[1][1] = 1.0; J[2][2] = 1.0;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int k = 0; k < 4; ++k) J[3 + r][3 + k] = 2.0 * s * QL[1 + r][k];
    double T[6][7];
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int cc = 0; cc < 7; ++cc) {
            double acc = 0.0;
#pragma unroll
            for (int k = 0; k < 7; ++k) acc += J[r][k] * ((k >= cc) ? Pc[k * (k + 1) / 2 + cc] : Pc[cc * (cc + 1) / 2 + k]);
            T[r][cc] = acc;
        }
    double A6[21];
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int cc = 0; cc <= r; ++cc) {
            double acc = 0.0;
#pragma unroll
            for (int k = 0; k < 7; ++k) acc += T[r][k] * J[cc][k];
            A6[r * (r + 1) / 2 + cc] = acc;
        }
    if (chol_nees<6>(A6, e, nees)) rec.nees_pose = nees;
    else { rec.nees_pose = CUDART_NAN; status = 1; }
    return status;
}

// One block per filter, threads over feature slots.
//   mode 0: score filter b against frame t: per-feature e_f / nees_f, the record of the frame, added into the totals;
//   mode 1: map export (p, C_f of every slot; NaN where empty or not evaluable).  Needs no world.
__global__ void __launch_bounds__(EV_THREADS, 2) k_eval(DevView v, DevWorld w, DevEval ev, int t, int b0, int mode) {
    extern __shared__ double ev_sm[];   // mode 0: sq [N], nees [N], code [N] (bytes)
    __shared__ double s_pc[28];         // camera block of P, packed lower
    __shared__ ekfslam_eval s_rec;
    __shared__ int s_mstatus;           // status bits of the map part
    const int b = b0 + blockIdx.x;
    const int N = v.N, ld = v.ld;
    const int nf = v.nfeat[b];
    const double* __restrict__ x = v.x + (size_t)b * ld;
    const double* __restrict__ P = v.P + (size_t)b * v.nmax * ld;
    double* s_sq = ev_sm;
    double* s_nees = ev_sm + N;
    uint8_t* s_code = reinterpret_cast<uint8_t*>(ev_sm + 2 * N);
    const double nan = CUDART_NAN;
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        const size_t fi = (size_t)b * N + i;
        int code = EV_EMPTY;
        double p[3], C[6];
        if (i < nf) {
            code = EV_OK;
            if (mode == 0) {
                const int tg = v.tag[fi];
                if (tg < 0 || tg >= w.M) code = EV_NO_TRUTH;
            }
            if (code == EV_OK && !feature_cartesian(x, P, ld, v.foff[fi], v.ftype[fi], p, C)) code = EV_BAD;
        }
        if (mode == 1) {
            if (code == EV_OK) {
                double Lc[6] = {C[0], C[1], C[2], C[3], C[4], C[5]};
                const double z3[3] = {0.0, 0.0, 0.0};
                double dummy;
                if (!chol_nees<3>(Lc, z3, dummy)) code = EV_BAD;
            }
            const bool ok = code == EV_OK;
#pragma unroll
            for (int k = 0; k < 3; ++k) ev.mp[3 * fi + k] = ok ? p[k] : nan;
#pragma unroll
            for (int k = 0; k < 6; ++k) ev.mc[6 * fi + k] = ok ? C[k] : nan;
            continue;
        }
        double e[3] = {nan, nan, nan}, nees = nan, sq = 0.0;
        if (code == EV_OK) {
            const double* pt = w.points + ((size_t)b * w.M + v.tag[fi]) * 3;
            double ef[3] = {p[0] - pt[0], p[1] - pt[1], p[2] - pt[2]};
            if (chol_nees<3>(C, ef, nees)) {
                e[0] = ef[0]; e[1] = ef[1]; e[2] = ef[2];
                sq = ef[0] * ef[0] + ef[1] * ef[1] + ef[2] * ef[2];
            } else {
                code = EV_BAD;
                nees = nan;
            }
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) ev.ferr[3 * fi + k] = e[k];
        ev.fnees[fi] = nees;
        s_sq[i] = sq; s_nees[i] = nees; s_code[i] = (uint8_t)code;
    }
    if (mode == 1) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (warp == 0 && lane < 28) {   // the 28 elements of the camera block's lower triangle, one per lane
        int r = 0;
        while ((r + 1) * (r + 2) / 2 <= lane) ++r;
        s_pc[lane] = P[(size_t)r * ld + (lane - r * (r + 1) / 2)];
    }
    __syncthreads();
    if (threadIdx.x == 0) {   // the camera part
        const double* pose = w.poses + ((size_t)t * v.B + b) * 7;
        double xv[7], pc[28];
#pragma unroll
        for (int k = 0; k < 7; ++k) xv[k] = x[k];
#pragma unroll
        for (int k = 0; k < 28; ++k) pc[k] = s_pc[k];
        ekfslam_eval rc;
        const int st = camera_eval(xv, pose, pose + 3, pc, rc);
        s_rec.pos_sq_err = rc.pos_sq_err; s_rec.rot_sq_err = rc.rot_sq_err;
        s_rec.nees_pos = rc.nees_pos; s_rec.nees_pose = rc.nees_pose;
        s_rec.status = st;
    } else if (threadIdx.x == 32) {   // the map sums: one thread, feature order (fixed, bit-reproducible)
        double sq = 0.0, ne = 0.0;
        int n_map = 0, n_skip = 0, status = 0;
        for (int i = 0; i < nf; ++i) {
            const int code = s_code[i];
            if (code == EV_OK) { sq += s_sq[i]; ne += s_nees[i]; ++n_map; }
            else { ++n_skip; status |= (code == EV_NO_TRUTH) ? 2 : 4; }
        }
        s_rec.map_sq_err = sq; s_rec.map_nees = ne;
        s_rec.n_map = n_map; s_rec.n_skip = n_skip;
        s_mstatus = status;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        ekfslam_eval r = s_rec;
        r.status |= s_mstatus;
        r.frames = 1;
        ev.rec[b] = r;
        ekfslam_eval tt = ev.tot[b];   // one block per filter: a plain read-modify-write, no atomics
        tt.pos_sq_err += r.pos_sq_err; tt.rot_sq_err += r.rot_sq_err;
        tt.nees_pos += r.nees_pos; tt.nees_pose += r.nees_pose;
        tt.map_sq_err += r.map_sq_err; tt.map_nees += r.map_nees;
        tt.n_map += r.n_map; tt.n_skip += r.n_skip; tt.frames += 1; tt.status |= r.status;
        ev.tot[b] = tt;
    }
}

void launch_eval(ekfslam_ctx* c, int mode, int t, int b0, int nb) {
    const size_t smem = (mode == 0) ? (((size_t)c->v.N * 17 + 7) / 8) * 8 : 0;
    ENSURE_DYN_SMEM(k_eval, smem, c->device);
    KScope ks(c, KT_EVAL);
    k_eval<<<nb, EV_THREADS, smem, c->stream>>>(c->v, c->world, c->ev, t, b0, mode);
}
