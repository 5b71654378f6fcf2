// Large stacked innovation (large maps: N = 500 -> k up to 1000 rows) for FEW filters: S = L L', X = inv(L).
// The inv(S) of mc/update.m:9 on the fp64 tensor pipe.
//
// One CTA per filter (k_chol / k_chol_sm) is a serial bottleneck here and the 16-wide lock-step kernels it replaced
// spent ~200 launches per update on DFMA work (2.0 of 5.2 ms per step at N = 500, B = 8).  This path is a blocked
// right-looking factorisation with 64-wide panels whose panel, trailing-update and triangular-inverse products are
// 64x64x64 DMMA (mma.sync m8n8k4 f64) tiles:
//   per panel j (2 launches):
//     k_cb_diagpanel  every CTA factors the 64x64 diagonal block S_jj = L_jj L_jj' and inverts L_jj in shared memory
//                     (redundantly - identical arithmetic, no grid-wide dependency), CTA 0 stores L_jj and
//                     inv(L_jj); CTA i > 0 forms the panel block L_ij = S_ij inv(L_jj)' on the tensor pipe
//     k_cb_trail      S_ab -= L_aj L_bj' for the lower tiles behind the panel
//   inverse, divide and conquer over block pairs [A 0; C D] -> [inv(A) 0; -inv(D) C inv(A), inv(D)], doubling the
//   block size per level (2 launches per level, every output tile independent):
//     k_cb_inv<0>     T = C inv(A)     (T parked in the unused UPPER triangle of the S buffer)
//     k_cb_inv<1>     X_C = -inv(D) T
// followed by the existing y = X nu / inv(S) nu kernels (k_mk_y, k_mk_cv, k_mk_fin in k_update.cu).
// Rows / columns >= k of a filter behave as an identity extension (loads are masked, stores are clipped), so filters
// of one batch may stack different numbers of rows and k need not be a multiple of 64.
#include "tc_common.cuh"

#define CB 64            // block size
#define CBP 68           // shared-memory pitch of a 64x64 block (pitch % 16 == 4: conflict-free DMMA fragments)
#define CBD 65           // pitch of the diagonal-block work arrays (column accesses)

// 64x64 block (r0, c0) of a kmax x kmax row-major matrix -> shared [64][CBP]; element (i, j) outside [0,k)^2 reads as
// delta_ij (identity extension).  lower_only: entries above the global diagonal read as 0.
__device__ __forceinline__ void cb_load(double* __restrict__ dst, const double* __restrict__ src, int kmax, int k, int r0,
                                        int c0, bool lower_only) {
    // 256 threads x 8 double2 pieces, all loads issued before the first use (predicated, no divergent control flow:
    // a loop with a branch around the load serialises the eight round trips to L2)
    double2 val[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int e = threadIdx.x + 256 * r;
        const int i = e >> 5, j = (e & 31) * 2;
        const int gi = r0 + i, gj = c0 + j;
        const bool okx = gi < k && gj < k && (!lower_only || gj <= gi);
        const bool oky = gi < k && gj + 1 < k && (!lower_only || gj + 1 <= gi);
        const double* p = src + (size_t)gi * kmax + gj;
        val[r].x = okx ? p[0] : ((gi >= k || gj >= k) && gi == gj ? 1.0 : 0.0);
        val[r].y = oky ? p[1] : ((gi >= k || gj + 1 >= k) && gi == gj + 1 ? 1.0 : 0.0);
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int e = threadIdx.x + 256 * r;
        const int i = e >> 5, j = (e & 31) * 2;
        dst[i * CBP + j] = val[r].x;
        dst[i * CBP + j + 1] = val[r].y;
    }
}

// acc (+)= A * B  (transB: A * B') for one 64x64x64 step; 8 warps in a 2x4 grid, 32x16 per warp.
// As[i][t] row-major; Bs[t][j] K-major, or - transB - the source block as stored, Bs[j][t].
template <bool transB>
__device__ __forceinline__ void cb_mma(double (&acc)[4][2][2], const double* __restrict__ As, const double* __restrict__ Bs) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wr = warp >> 2, wc = warp & 3, g = lane >> 2, q = lane & 3;
#pragma unroll 4
    for (int k4 = 0; k4 < CB / 4; ++k4) {
        double a[4], b[2];
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) a[mi] = As[(wr * 32 + mi * 8 + g) * CBP + k4 * 4 + q];
#pragma unroll
        for (int ni = 0; ni < 2; ++ni)
            b[ni] = transB ? Bs[(wc * 16 + ni * 8 + g) * CBP + k4 * 4 + q] : Bs[(k4 * 4 + q) * CBP + wc * 16 + ni * 8 + g];
#pragma unroll
        for (int mi = 0; mi < 4; ++mi)
#pragma unroll
            for (int ni = 0; ni < 2; ++ni) dmma(acc[mi][ni], a[mi], b[ni]);
    }
}

__device__ __forceinline__ void cb_zero(double (&acc)[4][2][2]) {
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 2; ++ni) { acc[mi][ni][0] = 0.0; acc[mi][ni][1] = 0.0; }
}

// dst block (r0, c0) = alpha * acc (+ beta_one * old), clipped to [0,k)^2
__device__ __forceinline__ void cb_store(double* __restrict__ dst, int kmax, int k, int r0, int c0, const double (&acc)[4][2][2],
                                         double alpha, bool accumulate) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wr = warp >> 2, wc = warp & 3, g = lane >> 2, q = lane & 3;
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 2; ++ni) {
            const int gi = r0 + wr * 32 + mi * 8 + g, gj = c0 + wc * 16 + ni * 8 + 2 * q;
            if (gi >= k) continue;
            double* o = dst + (size_t)gi * kmax + gj;
            if (gj + 1 < k) {
                double2 val = make_double2(alpha * acc[mi][ni][0], alpha * acc[mi][ni][1]);
                if (accumulate) { const double2 old = *reinterpret_cast<const double2*>(o); val.x += old.x; val.y += old.y; }
                *reinterpret_cast<double2*>(o) = val;
            } else if (gj < k) {
                o[0] = alpha * acc[mi][ni][0] + (accumulate ? o[0] : 0.0);
            }
        }
}

// ---------------------------------------------------------------------------------------
// panel j0: diagonal block factor + inverse (every CTA), panel block product (CTAs 1..)
// grid = (1 + blocks below the panel, B), 256 threads, dynamic shared memory 3 blocks
// The 64x64 diagonal block is factored in shared memory in four 16-wide steps (warp 0 factors and inverts the 16x16
// diagonal sub-block in registers, all threads do the 16-wide panel and the rank-16 trailing update) and inverted by
// block forward substitution on the four 16x16 inverses - 18 block barriers in all.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_cb_diagpanel(DevView v, int j0) {
    extern __shared__ __align__(16) double sm[];
    const int b = blockIdx.y;
    const int k = 2 * v.ksel[b];
    if (j0 >= k) return;
    const int i0 = j0 + CB * blockIdx.x;            // blockIdx.x == 0: the diagonal block itself
    if (i0 >= k) return;
    const int kmax = v.kmax, tid = threadIdx.x;
    double* __restrict__ S = v.Sb + (size_t)b * kmax * kmax;
    double* __restrict__ X = v.Li + (size_t)b * kmax * kmax;
    double* D = sm;                      // [64][CBD]  S_jj -> L_jj (lower); pitch 65 inside a [64][CBP] region
    double* Xd = sm + CB * CBP;          // [64][CBP]  inv(L_jj), explicit zeros above the diagonal
    double* As = sm;                     // [64][CBP]  S_ij: prefetched into registers now, parked over D once D is dead
    __shared__ double Di[4][16 * 17];    // inverses of the four 16x16 diagonal sub-blocks
    __shared__ double Tt[3][16 * 17];    // block forward substitution temporaries
    __shared__ int s_bad;
    if (tid == 0) s_bad = 0;
    {
        double dv[16];                   // 16 entries of S_jj per thread, all loads in flight at once
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            const int e = tid + 256 * r;
            const int i = e >> 6, j = e & 63;
            const int gi = j0 + i, gj = j0 + j;
            const bool ok = j <= i && gi < k && gj < k;
            dv[r] = ok ? S[(size_t)gi * kmax + gj] : ((j == i && gi >= k) ? 1.0 : 0.0);
        }
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            const int e = tid + 256 * r;
            D[(e >> 6) * CBD + (e & 63)] = dv[r];
        }
    }
    for (int e = tid; e < CB * CBP; e += blockDim.x) Xd[e] = 0.0;
    double2 pre[8];                      // this thread's 16 entries of S_ij (same mapping as cb_load), in flight during the factorisation
    if (blockIdx.x > 0) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int e = tid + 256 * r;
            const int gi = i0 + (e >> 5), gj = j0 + (e & 31) * 2;
            pre[r].x = (gi < k && gj < k) ? S[(size_t)gi * kmax + gj] : 0.0;          // block (i, j), i > j: no diagonal entries
            pre[r].y = (gi < k && gj + 1 < k) ? S[(size_t)gi * kmax + gj + 1] : 0.0;
        }
    }
    __syncthreads();
    const int ti = tid >> 4, tj = tid & 15;
    for (int jb = 0; jb < 4; ++jb) {
        const int c0 = 16 * jb;
        if (tid < 32) {
            const bool bad = chol16_warp(D + c0 * CBD + c0, CBD, Di[jb]);
            if (bad && tid == 0) s_bad = 1;
        }
        __syncthreads();
        // 16-wide panel below: L[i][c0+cc] = sum_{t<=cc} D[i][c0+t] * Di[cc][t]   (old values read first, then written)
        double pn[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const int i = c0 + 16 + 16 * r + ti;
            double sacc = 0.0;
            if (i < CB) {
#pragma unroll
                for (int t = 0; t < 16; ++t) sacc += (t <= tj) ? D[i * CBD + c0 + t] * Di[jb][tj * 17 + t] : 0.0;
            }
            pn[r] = sacc;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const int i = c0 + 16 + 16 * r + ti;
            if (i < CB) D[i * CBD + c0 + tj] = pn[r];
        }
        __syncthreads();
        // rank-16 trailing update of the lower part behind the panel, by 16x16 sub-blocks (one element per thread)
        for (int bi = jb + 1; bi < 4; ++bi)
            for (int bj = jb + 1; bj <= bi; ++bj) {
                const int i = 16 * bi + ti, j = 16 * bj + tj;
                if (j <= i) {
                    double sacc = 0.0;
#pragma unroll
                    for (int t = 0; t < 16; ++t) sacc += D[i * CBD + c0 + t] * D[j * CBD + c0 + t];
                    D[i * CBD + j] -= sacc;
                }
            }
        __syncthreads();
    }
    // inv(L_jj) by block forward substitution: X_ii = Di_i;  X_{i,i-d} = -Di_i * sum_{t=i-d}^{i-1} L_it X_{t,i-d}
    for (int bi = 0; bi < 4; ++bi) Xd[(16 * bi + ti) * CBP + 16 * bi + tj] = Di[bi][ti * 17 + tj];
    __syncthreads();
    for (int d = 1; d < 4; ++d) {
        for (int bi = d; bi < 4; ++bi) {            // T = sum_t L[bi][t] X[t][bi-d]
            const int bj = bi - d;
            double sacc = 0.0;
            for (int t = bj; t < bi; ++t) {
#pragma unroll
                for (int u = 0; u < 16; ++u) sacc += D[(16 * bi + ti) * CBD + 16 * t + u] * Xd[(16 * t + u) * CBP + 16 * bj + tj];
            }
            Tt[bi - d][ti * 17 + tj] = sacc;
        }
        __syncthreads();
        for (int bi = d; bi < 4; ++bi) {
            const int bj = bi - d;
            double sacc = 0.0;
#pragma unroll
            for (int u = 0; u < 16; ++u) sacc += (u <= ti) ? Di[bi][ti * 17 + u] * Tt[bi - d][u * 17 + tj] : 0.0;
            Xd[(16 * bi + ti) * CBP + 16 * bj + tj] = -sacc;
        }
        __syncthreads();
    }
    if (blockIdx.x == 0) {
        if (tid == 0 && s_bad) atomicOr(&v.stats[b].status, 2);
        for (int e = tid; e < CB * CB; e += blockDim.x) {
            const int i = e >> 6, j = e & 63;
            const int gi = j0 + i, gj = j0 + j;
            if (gi < k && gj < k) {
                if (j <= i) S[(size_t)gi * kmax + gj] = D[i * CBD + j];
                X[(size_t)gi * kmax + gj] = Xd[i * CBP + j];      // zeros above the diagonal included (k_gemm reads them)
            }
        }
        return;
    }
    // L_ij = S_ij * inv(L_jj)'   (D is dead: every thread passed the last barrier of the inverse)
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int e = tid + 256 * r;
        As[(e >> 5) * CBP + (e & 31) * 2] = pre[r].x;
        As[(e >> 5) * CBP + (e & 31) * 2 + 1] = pre[r].y;
    }
    __syncthreads();
    double acc[4][2][2];
    cb_zero(acc);
    cb_mma<true>(acc, As, Xd);
    cb_store(S, kmax, k, i0, j0, acc, 1.0, false);
}

// ---------------------------------------------------------------------------------------
// trailing update behind panel j0: S_ab -= L_aj L_bj' for block rows a >= b > j.  grid = (lower tiles, B)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_cb_trail(DevView v, int j0) {
    extern __shared__ __align__(16) double sm[];
    const int b = blockIdx.y;
    const int k = 2 * v.ksel[b];
    const int i1 = j0 + CB;
    if (i1 >= k) return;
    const int e = blockIdx.x;
    int ta = (int)((sqrtf(8.0f * e + 1.0f) - 1.0f) * 0.5f);
    while ((ta + 1) * (ta + 2) / 2 <= e) ++ta;
    while (ta * (ta + 1) / 2 > e) --ta;
    const int tb = e - ta * (ta + 1) / 2;
    const int r0 = i1 + ta * CB, c0 = i1 + tb * CB;
    if (r0 >= k) return;
    const int kmax = v.kmax;
    double* __restrict__ S = v.Sb + (size_t)b * kmax * kmax;
    double* As = sm;
    double* Bs = sm + CB * CBP;
    cb_load(As, S, kmax, k, r0, j0, false);
    cb_load(Bs, S, kmax, k, c0, j0, false);
    __syncthreads();
    double acc[4][2][2];
    cb_zero(acc);
    cb_mma<true>(acc, As, Bs);
    cb_store(S, kmax, k, r0, c0, acc, -1.0, true);   // diagonal tiles also touch their upper half: never read
}

// ---------------------------------------------------------------------------------------
// triangular inverse, one level of the divide and conquer.  Blocks are 64 wide; at level s the diagonal blocks of
// 2s have known inverses for their two halves A = [2ps, 2ps+s), D = [2ps+s, 2ps+2s) and the coupling block C = L[D, A]
// becomes X[D, A] = -inv(D) C inv(A).  phase 0: T[ti][tj] = sum_{t in A, t >= tj} L[ti][t] X[t][tj], stored at block
// (tj, ti) of the S buffer (upper triangle, unused);  phase 1: X[ti][tj] = -sum_{t in D, t <= ti} X[ti][t] T[t][tj].
// grid = (nblk * s, B): blockIdx.x -> (ti, o), tj = pair base + o
// ---------------------------------------------------------------------------------------
template <int phase>
__global__ void __launch_bounds__(256) k_cb_inv(DevView v, int s) {
    extern __shared__ __align__(16) double sm[];
    const int b = blockIdx.y;
    const int k = 2 * v.ksel[b];
    const int ti = blockIdx.x / s, o = blockIdx.x % s;
    if (ti * CB >= k) return;
    if ((ti % (2 * s)) < s) return;                 // ti must lie in a D range
    const int base = (ti / (2 * s)) * (2 * s);      // first block of the pair
    const int tj = base + o;                        // in the A range
    const int kmax = v.kmax;
    double* __restrict__ S = v.Sb + (size_t)b * kmax * kmax;
    double* __restrict__ X = v.Li + (size_t)b * kmax * kmax;
    double* As = sm;
    double* Bs = sm + CB * CBP;
    double acc[4][2][2];
    cb_zero(acc);
    if (phase == 0) {
        for (int t = tj; t < base + s; ++t) {
            __syncthreads();
            cb_load(As, S, kmax, k, ti * CB, t * CB, false);        // L[ti][t]
            cb_load(Bs, X, kmax, k, t * CB, tj * CB, t == tj);      // X[t][tj] (diagonal block: lower part only)
            __syncthreads();
            cb_mma<false>(acc, As, Bs);
        }
        cb_store(S, kmax, kmax, tj * CB, ti * CB, acc, 1.0, false); // park T in the upper triangle, whole block
    } else {
        for (int t = base + s; t <= ti; ++t) {
            __syncthreads();
            cb_load(As, X, kmax, k, ti * CB, t * CB, t == ti);      // X[ti][t]
            cb_load(Bs, S, kmax, kmax, tj * CB, t * CB, false);     // T[t][tj] parked at (tj, t)
            __syncthreads();
            cb_mma<false>(acc, As, Bs);
        }
        cb_store(X, kmax, k, ti * CB, tj * CB, acc, -1.0, false);
    }
}

void launch_chol_blocked64(ekfslam_ctx* c, int kact) {
    DevView& v = c->v;
    cudaStream_t st = c->stream;
    const size_t sm_dp = sizeof(double) * (2 * CB * CBP);
    const size_t sm_2 = sizeof(double) * (2 * CB * CBP);
    ENSURE_DYN_SMEM(k_cb_diagpanel, sm_dp, c->device);
    ENSURE_DYN_SMEM(k_cb_trail, sm_2, c->device);
    ENSURE_DYN_SMEM(k_cb_inv<0>, sm_2, c->device);
    ENSURE_DYN_SMEM(k_cb_inv<1>, sm_2, c->device);
    const int nblk = (kact + CB - 1) / CB;
    for (int jb = 0; jb < nblk; ++jb) {
        const int below = nblk - 1 - jb;
        dim3 gp(1 + below, v.B);
        k_cb_diagpanel<<<gp, 256, sm_dp, st>>>(v, jb * CB);
        c->launches++;
        if (below > 0) {
            dim3 gt(below * (below + 1) / 2, v.B);
            k_cb_trail<<<gt, 256, sm_2, st>>>(v, jb * CB);
            c->launches++;
        }
    }
    for (int s = 1; s < nblk; s *= 2) {
        dim3 gi(nblk * s, v.B);
        k_cb_inv<0><<<gi, 256, sm_2, st>>>(v, s);
        k_cb_inv<1><<<gi, 256, sm_2, st>>>(v, s);
        c->launches += 2;
    }
}
