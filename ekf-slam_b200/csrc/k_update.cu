// EKF update of mc/update.m:3-32 for the features selected by a flag mask
// (mc/ekf_update_li_inliers.m:8-21, mc/ekf_update_hi_inliers.m:8-21), batched over filters.
//
// With G = H P (rows of the selected features, from k_hp) and S = G_sel H_sel' + I = L L':
//     K (z-h) = G_sel' inv(S) nu = W' y,      W = inv(L) G_sel,  y = inv(L) nu
//     K S K'  = G_sel' inv(S) G_sel = W' W
// so  x+ = x + W' y  and  P+ = P - W' W  (exactly symmetric, so the reference's
// 0.5 P + 0.5 P' (:14) is the identity here), followed by the quaternion normalisation
// Jacobian (:18-24) fused into the epilogue of the covariance downdate.
//
// Kernels: k_upd_S (select + stack S, nu) -> k_chol (blocked Cholesky, inv(L), y) ->
//          k_gemm (W = inv(L) G_sel, triangular GEMM on DMMA; also x+, q normalisation, normJac) ->
//          k_wfix (W <- W J', bookkeeping) -> k_downdate* (P <- J P J' - W'W, k_downdate.cu).
#include "model.cuh"
#include "tc_common.cuh"

#define NB 16

// index e of a lower triangle stored by rows -> (r, c), c <= r
__device__ __forceinline__ void tri_unrank(int e, int& r, int& c) {
    r = (int)((sqrt(8.0 * e + 1.0) - 1.0) * 0.5);
    while ((r + 1) * (r + 2) / 2 <= e) ++r;
    while (r * (r + 1) / 2 > e) --r;
    c = e - r * (r + 1) / 2;
}

// S = G_sel H_sel' + I, lower triangle at feature-pair granularity: pair e -> (fa >= fb) -> one 2x2 block.
// STAGED: the per-feature operands of the pair loop (feature index, state offset, block width, compact Jacobian) come from
// shared memory (k_upd_S stages them once per filter), so the only global loads left per pair are the 2 x 13 entries of G,
// all independent (ncu, round 2: the loop was a chain of dependent DRAM round trips - sel -> foff / ftype -> G - and the
// feature-block loop with its run-time width issued its loads one iteration at a time: 60 % of the kernel's samples).
#define UPS_NMAX 128   // features per filter the staged path holds (26.6 KB of Jacobians)
template <bool STAGED>
__device__ __forceinline__ void upd_S_pairs(const DevView& v, int b, int ns, int first, int stride, const int* s_sel,
                                            const int* s_off, const int* s_w, const double* s_H) {
    const int N = v.N, ld = v.ld, kmax = v.kmax;
    const int* __restrict__ sel = v.sel + (size_t)b * N;
    const double* __restrict__ G = v.G + (size_t)b * kmax * ld;
    double* __restrict__ S = v.Sb + (size_t)b * kmax * kmax;
    const int npair = ns * (ns + 1) / 2;
    for (int e = first; e < npair; e += stride) {
        int fa, fb;   // fa >= fb
        tri_unrank(e, fa, fb);
        int ia, off, w;
        const double* __restrict__ H;
        if (STAGED) {
            ia = s_sel[fa]; off = s_off[fb]; w = s_w[fb]; H = s_H + fb * EKF_HSTRIDE;
        } else {
            ia = sel[fa];
            const size_t tb = (size_t)b * N + sel[fb];
            H = v.Hc + tb * EKF_HSTRIDE;
            off = v.foff[tb];
            w = (v.ftype[tb] == EKFSLAM_FEAT_INVERSEDEPTH) ? 6 : 3;
        }
        const double* __restrict__ g0 = G + (size_t)(2 * ia) * ld;
        const double* __restrict__ g1 = g0 + ld;
        // all 26 entries of G first (independent loads), then the products in the order of the reference's sparse H
        double ga[EKF_HC], gb[EKF_HC];
#pragma unroll
        for (int c = 0; c < 7; ++c) { ga[c] = g0[c]; gb[c] = g1[c]; }
#pragma unroll
        for (int c = 0; c < 6; ++c) {
            const int cc = off + ((c < w) ? c : 0);
            ga[7 + c] = g0[cc]; gb[7 + c] = g1[cc];
        }
        double s00 = 0, s01 = 0, s10 = 0, s11 = 0;
#pragma unroll
        for (int c = 0; c < EKF_HC; ++c) {
            if (c < 7 + w) {
                const double h0 = H[c], h1 = H[EKF_HC + c];
                s00 += ga[c] * h0; s01 += ga[c] * h1; s10 += gb[c] * h0; s11 += gb[c] * h1;
            }
        }
        if (fa == fb) { s00 += 1.0; s11 += 1.0; }  // R = eye(length(z)), mc/ekf_update_li_inliers.m:18
        S[(size_t)(2 * fa) * kmax + 2 * fb] = s00;
        S[(size_t)(2 * fa) * kmax + 2 * fb + 1] = s01;      // (for fa == fb this upper entry is never read)
        S[(size_t)(2 * fa + 1) * kmax + 2 * fb] = s10;
        S[(size_t)(2 * fa + 1) * kmax + 2 * fb + 1] = s11;
    }
}

// ---------------------------------------------------------------------------------------
// select + S + nu.  One block per filter.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256, 4) k_upd_S(DevView v, int mask, int which_prior, int iter_nu, int do_pairs) {
    const int b = blockIdx.x;
    const int N = v.N, ld = v.ld, kmax = v.kmax;
    const int nf = v.nfeat[b];
    const int tid = threadIdx.x;
    __shared__ int s_k;
    int* __restrict__ sel = v.sel + (size_t)b * N;
    if (tid < 32) {
        // selected features in feature order: ballot + prefix popcount (a serial thread-0 loop over the features was
        // a third of this kernel's time)
        int cnt = 0;
        for (int i0 = 0; i0 < nf; i0 += 32) {
            const int i = i0 + tid;
            const bool on = (i < nf) && v.ftype[b * N + i] != EKFSLAM_FEAT_NONE && (v.flags[(size_t)b * N + i] & mask);
            const unsigned m = __ballot_sync(0xffffffffu, on);
            if (on) sel[cnt + __popc(m & ((1u << tid) - 1u))] = i;
            cnt += __popc(m);
        }
        if (tid == 0) {
            v.ksel[b] = cnt;
            s_k = cnt;
            if (mask & EKFSLAM_F_LI) v.stats[b].n_li = cnt;
            if (mask & EKFSLAM_F_HI) v.stats[b].n_hi = cnt;
            if (cnt > 0) atomicMax(v.kmaxdev, 2 * cnt);
        }
    }
    __syncthreads();
    const int ns = s_k;
    const int k = 2 * ns;
    // innovation nu = z - h; for an iterated update (x holds the current iterate x_j, xp the prior x^-)
    // nu_j = z - h(x_j) - H_j (x^- - x_j).  Computed before x is reset to the prior below.
    {
        double* __restrict__ yv0 = v.yv + (size_t)b * kmax;
        const double* __restrict__ xj = v.x + (size_t)b * ld;
        const double* __restrict__ x0 = v.xp + (size_t)b * ld;
        for (int a = tid; a < k; a += blockDim.x) {
            const size_t t = (size_t)b * N + sel[a >> 1];
            double nu = v.z[2 * t + (a & 1)] - v.h[2 * t + (a & 1)];
            if (iter_nu) {
                const double* __restrict__ H = v.Hc + t * EKF_HSTRIDE + (a & 1) * EKF_HC;
                const int off = v.foff[t];
                const int w = (v.ftype[t] == EKFSLAM_FEAT_INVERSEDEPTH) ? 6 : 3;
                double s = 0.0;
                for (int c = 0; c < 7; ++c) s += H[c] * (x0[c] - xj[c]);
                for (int c = 0; c < w; ++c) s += H[7 + c] * (x0[off + c] - xj[off + c]);
                nu -= s;
            }
            yv0[a] = nu;
        }
    }
    __syncthreads();
    if (which_prior == 1) {  // x_k_k starts from x_k_km1 (also the pass-through of mc/update.m:28)
        const int n = v.nstate[b];
        for (int j = tid; j < n; j += blockDim.x) v.x[(size_t)b * ld + j] = v.xp[(size_t)b * ld + j];
    }
    if (k == 0) return;
    if (!do_pairs) return;   // few filters: the pair loop runs as its own, wider launch (k_upd_pairs)
    if (N <= UPS_NMAX) {
        __shared__ int s_sel[UPS_NMAX], s_off[UPS_NMAX], s_w[UPS_NMAX];
        __shared__ double s_H[UPS_NMAX * EKF_HSTRIDE];
        for (int f = tid; f < ns; f += blockDim.x) {
            const int i = sel[f];
            const size_t t = (size_t)b * N + i;
            s_sel[f] = i;
            s_off[f] = v.foff[t];
            s_w[f] = (v.ftype[t] == EKFSLAM_FEAT_INVERSEDEPTH) ? 6 : 3;
        }
        for (int e = tid; e < ns * EKF_HSTRIDE; e += blockDim.x) {
            const int f = e / EKF_HSTRIDE;
            s_H[e] = v.Hc[((size_t)b * N + sel[f]) * EKF_HSTRIDE + (e - f * EKF_HSTRIDE)];
        }
        __syncthreads();
        upd_S_pairs<true>(v, b, ns, tid, blockDim.x, s_sel, s_off, s_w, s_H);
    } else {
        upd_S_pairs<false>(v, b, ns, tid, blockDim.x, nullptr, nullptr, nullptr, nullptr);
    }
}

// S = G_sel H_sel' + I for few filters with large maps: grid = (slices, B), the pairs of a filter spread over the slices
// (one block per filter leaves a 148-SM GPU with 8 busy blocks at cfg4).  Runs after k_upd_S(do_pairs = 0).
__global__ void __launch_bounds__(256) k_upd_pairs(DevView v) {
    const int b = blockIdx.y;
    const int ns = v.ksel[b];
    if (ns == 0) return;
    upd_S_pairs<false>(v, b, ns, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x, nullptr, nullptr, nullptr, nullptr);
}

// ---------------------------------------------------------------------------------------
// Blocked right-looking Cholesky S = L L' (lower, in place), X = inv(L), y <- X nu.
// One block per filter, panels of NB columns.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_chol(DevView v, int kskip) {
    extern __shared__ double sm[];
    const int b = blockIdx.x;
    const int k = 2 * v.ksel[b];
    if (k == 0 || k <= kskip) return;   // k <= kskip: handled by k_chol_sm
    const int kmax = v.kmax;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double* __restrict__ S = v.Sb + (size_t)b * kmax * kmax;
    double* __restrict__ X = v.Li + (size_t)b * kmax * kmax;
    double* D = sm;                       // [NB][NB+1] diagonal block factor
    double* Di = D + NB * (NB + 1);       // [NB][NB+1] its inverse
    double* Pn = Di + NB * (NB + 1);      // [kmax][NB+1] panel below the diagonal block / row panel
    __shared__ int s_bad;
    if (tid == 0) s_bad = 0;

    for (int j0 = 0; j0 < k; j0 += NB) {
        const int nb = min(NB, k - j0);
        for (int e = tid; e < NB * NB; e += blockDim.x) {
            const int r = e / NB, c = e - r * NB;
            // rows >= nb are padded with the identity so that the register factorisation below is benign
            D[r * (NB + 1) + c] = (r < nb && c <= r) ? S[(size_t)(j0 + r) * kmax + j0 + c] : ((r >= nb && r == c) ? 1.0 : 0.0);
            Di[r * (NB + 1) + c] = 0.0;
        }
        __syncthreads();
        if (warp == 0) {
            if (chol16_warp(D, NB + 1, Di) && lane == 0) s_bad = 1;
        }
        __syncthreads();
        for (int e = tid; e < nb * nb; e += blockDim.x) {
            const int r = e / nb, c = e - r * nb;
            if (c <= r) {
                S[(size_t)(j0 + r) * kmax + j0 + c] = D[r * (NB + 1) + c];
                X[(size_t)(j0 + r) * kmax + j0 + c] = Di[r * (NB + 1) + c];
            }
        }
        // panel: L[i][j0+c] = sum_{t<=c} S[i][j0+t] * Di[c][t]
        const int i1 = j0 + nb;
        for (int i = i1 + tid; i < k; i += blockDim.x) {
            double row[NB];
#pragma unroll
            for (int t = 0; t < NB; ++t) row[t] = (t < nb) ? S[(size_t)i * kmax + j0 + t] : 0.0;
#pragma unroll
            for (int c = 0; c < NB; ++c) {
                double s = 0.0;
#pragma unroll
                for (int t = 0; t <= c; ++t) s += row[t] * Di[c * (NB + 1) + t];
                if (c < nb) {
                    S[(size_t)i * kmax + j0 + c] = s;
                    Pn[(i - i1) * (NB + 1) + c] = s;
                }
            }
        }
        __syncthreads();
        // trailing update of the lower triangle: S[i][c] -= sum_t Pn[i][t] Pn[c][t]
        const int m = k - i1;
        if (m > 0) {
            const int mt = (m + 3) / 4;  // 4x4 micro tiles
            const int ntile = mt * (mt + 1) / 2;
            for (int e = tid; e < ntile; e += blockDim.x) {
                int ti, tj;
                tri_unrank(e, ti, tj);
                double acc[4][4];
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int c = 0; c < 4; ++c) acc[a][c] = 0.0;
                for (int t = 0; t < nb; ++t) {
                    double ra[4], rc[4];
#pragma unroll
                    for (int a = 0; a < 4; ++a) {
                        const int ia = ti * 4 + a, ic = tj * 4 + a;
                        ra[a] = (ia < m) ? Pn[ia * (NB + 1) + t] : 0.0;
                        rc[a] = (ic < m) ? Pn[ic * (NB + 1) + t] : 0.0;
                    }
#pragma unroll
                    for (int a = 0; a < 4; ++a)
#pragma unroll
                        for (int c = 0; c < 4; ++c) acc[a][c] += ra[a] * rc[c];
                }
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const int ia = ti * 4 + a, ic = tj * 4 + c;
                        if (ia < m && ic <= ia) S[(size_t)(i1 + ia) * kmax + i1 + ic] -= acc[a][c];
                    }
            }
        }
        __syncthreads();
    }

    // X = inv(L), block row by block row:  X[I][0:I0] = -Di_I * ( L[I][0:I0] * X[0:I0][0:I0] )
    for (int I0 = NB; I0 < k; I0 += NB) {
        const int nb = min(NB, k - I0);
        // stage the row panel L[I0..I0+nb)[0..I0) (transposed: Pn[t][r]) and Di of this block
        for (int e = tid; e < nb * I0; e += blockDim.x) {
            const int r = e / I0, t = e - r * I0;
            Pn[t * (NB + 1) + r] = S[(size_t)(I0 + r) * kmax + t];
        }
        for (int e = tid; e < NB * NB; e += blockDim.x) {
            const int r = e / NB, c = e - r * NB;
            Di[r * (NB + 1) + c] = (r < nb && c <= r) ? X[(size_t)(I0 + r) * kmax + I0 + c] : 0.0;
        }
        __syncthreads();
        for (int c = tid; c < I0; c += blockDim.x) {
            double y[NB];
#pragma unroll
            for (int r = 0; r < NB; ++r) y[r] = 0.0;
            // batches of 8 independent global loads keep the memory pipeline full (the FMAs only need them later)
            for (int t = c; t < I0; t += 8) {
                double xv[8];
#pragma unroll
                for (int u8 = 0; u8 < 8; ++u8) xv[u8] = (t + u8 < I0) ? X[(size_t)(t + u8) * kmax + c] : 0.0;
#pragma unroll
                for (int u8 = 0; u8 < 8; ++u8) {
                    const int tt = min(t + u8, I0 - 1);
#pragma unroll
                    for (int r = 0; r < NB; ++r) y[r] += Pn[tt * (NB + 1) + r] * xv[u8];
                }
            }
#pragma unroll
            for (int r = 0; r < NB; ++r) {
                double s = 0.0;
#pragma unroll
                for (int j = 0; j <= r; ++j) s += Di[r * (NB + 1) + j] * y[j];
                if (r < nb) X[(size_t)(I0 + r) * kmax + c] = -s;
            }
        }
        __syncthreads();
    }
    // explicit zeros above the diagonal of X: k_w streams X panels with cp.async and does not mask
    for (int e = tid; e < k * k; e += blockDim.x) {
        const int r = e / k, c = e - r * k;
        if (c > r) X[(size_t)r * kmax + c] = 0.0;
    }
    // y = X nu and cv = X' y = inv(S) nu (the state update is x+ = x + G_sel' cv, accumulated inside k_gemm).
    // One warp per row of X, lanes along the row (coalesced); fixed summation orders -> deterministic.
    double* nu = Pn;                 // [k]
    double* part = Pn + kmax;        // [nwarps][k] partial column sums of the second product
    const int nwarps = blockDim.x >> 5;
    double* __restrict__ yv = v.yv + (size_t)b * kmax;
    __syncthreads();
    for (int a = tid; a < k; a += blockDim.x) nu[a] = yv[a];
    __syncthreads();
    for (int a = warp; a < k; a += nwarps) {
        double s = 0.0;
        for (int t = lane; t <= a; t += 32) s += X[(size_t)a * kmax + t] * nu[t];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) yv[a] = s;
    }
    __syncthreads();
    for (int a = tid; a < k; a += blockDim.x) nu[a] = yv[a];
    for (int e = tid; e < nwarps * k; e += blockDim.x) part[e] = 0.0;
    __syncthreads();
    for (int a = warp; a < k; a += nwarps) {
        const double ya = nu[a];
        for (int t = lane; t <= a; t += 32) part[warp * k + t] += X[(size_t)a * kmax + t] * ya;
    }
    __syncthreads();
    double* __restrict__ cv = v.cv + (size_t)b * kmax;
    for (int t = tid; t < k; t += blockDim.x) {
        double s = 0.0;
        for (int w2 = 0; w2 < nwarps; ++w2) s += part[w2 * k + t];
        cv[t] = s;
    }
    if (tid == 0 && s_bad) atomicOr(&v.stats[b].status, 2);
}

// ---------------------------------------------------------------------------------------
// Shared-memory resident variant for k <= CHS_K (the common case at N = 100: k ~ 100): the lower triangle of S
// lives packed in shared memory for the whole factorisation and inv(L) is formed IN PLACE (block row I of X only
// needs block row I of L and the rows of X above it), so global memory is touched twice: S in, inv(L) out.
// k_chol above works on S in global memory (every panel / trailing update is an L2 round trip: long-scoreboard
// stalls were half of its issue stalls) and stays as the path for larger k.  Same blocked algorithm and pivots.
// ---------------------------------------------------------------------------------------
#define CHS_KL 200  // largest variant (a handful of filters per frame at N = 100): 144 < k <= 200, 512 threads, 190 KB -> 1 CTA/SM, own side stream
#define CHS_K 144   // large variant: KMIN < k <= 144, 256 threads, 2 CTAs/SM
#define CHS_KM 112  // middle variant (li update at N = 100: k ~ 100): 256 threads, <= 85 registers, 72 KB -> 3 CTAs/SM
#define CHS_KS 48   // small variant (hi update: k ~ 24): k <= 48, 128 threads, 21 KB of shared memory -> many CTAs/SM
// Packed lower triangle whose rows start on an even index (16-byte aligned): the trailing update reads and writes four
// neighbouring columns of a row as two 128-bit accesses.
__device__ __forceinline__ int tri(int r, int c) { return ((r * (r + 1)) >> 1) + ((r + 1) >> 1) + c; }
#define CHS_TRI(K) (((K) * ((K) + 1)) / 2 + ((K) + 1) / 2)
#define CHS_SMEM(K) (sizeof(double) * (CHS_TRI(K) + 3 * NB * (NB + 1) + (size_t)(K) * NB))

// What round 2's per-line ncu digest (tools/ncu_lines.py) and the A/B builds behind it showed about this kernel
// (B = 4096, k ~ 103: 0.82 -> 0.60 ms for the li update, 1.77 -> 1.41 ms for both Cholesky brackets of a step):
//   * it is a chain of LATENCY-bound phases (issue slots 35 % busy, fp64 pipe 14 %): what counts is the dependent chain
//     of each phase, not its instruction or shared-memory volume.  Vectorised / broadcast operands alone (transposed
//     panel PT[t][row] for the 4x4 micro tiles of the trailing update, 128-bit read-modify-writes of the packed
//     triangle) cut the shared wavefronts by half and the time by nothing;
//   * the biggest single loss was a DIVERGENT tail: rows of -Di*y selected per lane by `if ((r & 3) == q)` over a
//     compile-time r ran as 16 serial predicated blocks, each its own dependent chain (-0.16 ms once the four rows of a
//     lane became four interleaved chains over a zero-padded Di);
//   * the S load as per-element asynchronous copies (-0.09 ms: the plain loop paid a DRAM round trip per row);
//   * the inverse block rows need nothing from the CURRENT diagonal block, so they run in warps 1.. while warp 0 walks the
//     serial pivot chain (-0.05 ms; what is left at the barrier behind the pivot chain, a third of the kernel, is the chain
//     itself: shuffle -> MUFU.RSQ64H + 4 dependent fp64 operations -> multiply -> shuffle -> FMA per pivot);
//   * rolling loops to shrink the code (13 k -> 4 k instructions; no_instruction stalls were as frequent as dependency
//     stalls) LOST time for the pivot chain, the block inverse and the panel solve - an in-order warp stalls on every
//     rolled dependent chain - and won only for the two halves of chs_inv_compute.
// Block row I0/16 of X = inv(L), formed from L[I0..I0+16)[0..I0) (read in place from the packed triangle) and the rows of
// X above it:  X[I][0:I0] = -Di_I * ( L[I][0:I0] * X[0:I0][0:I0] ).  A warp takes the pair of 8-wide column blocks
// (pair, last - pair) - (I0 + 8) / 4 steps of 8 columns x 4 values of t whatever the pair is - and keeps its 2 x 4 results
// per lane in registers: the rows it overwrites are still being read by the other warps, so the store happens behind a
// barrier (chs_inv_store).
__device__ __forceinline__ void chs_inv_compute(const double* Ls, const double* Di, int I0, int nb, int pair, int lane, double (&res)[2][4]) {
    const int c8 = lane & 7, tq = lane >> 3;
    const int nblk = I0 >> 3;                       // I0 is a multiple of 16
    const double* lrow = Ls + tri(I0, 0);           // row I0 + r starts at lrow + r * I0 + tri(r, 0)   (I0 even)
#pragma unroll 1   // rolled: half the code of the hottest loop, 1.18 -> 1.14 ms
    for (int half = 0; half < 2; ++half) {
        const int cb = half ? nblk - 1 - pair : pair;
        const int c = cb * 8 + c8;
        double y[NB];
#pragma unroll
        for (int r = 0; r < NB; ++r) y[r] = 0.0;
#pragma unroll 2
        for (int t = cb * 8 + tq; t < I0; t += 4) {
            const double xv = (t >= c) ? Ls[tri(t, c)] : 0.0;
            const double* lt = lrow + t;
#pragma unroll
            for (int r = 0; r < NB; ++r) y[r] += ((r < nb) ? lt[r * I0 + tri(r, 0)] : 0.0) * xv;   // rows past k hold no data
        }
#pragma unroll
        for (int r = 0; r < NB; ++r) {
            y[r] += __shfl_xor_sync(0xffffffffu, y[r], 8);
            y[r] += __shfl_xor_sync(0xffffffffu, y[r], 16);
        }
        // rows tq, tq+4, tq+8, tq+12 of -Di*y: four independent chains over all 16 columns (Di is zero above its diagonal)
        double s4[4] = {0.0, 0.0, 0.0, 0.0};
        const double* dr = Di + tq * (NB + 1);
#pragma unroll
        for (int j = 0; j < NB; ++j) {
#pragma unroll
            for (int u = 0; u < 4; ++u) s4[u] += dr[u * 4 * (NB + 1) + j] * y[j];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (half) res[1][u] = -s4[u];
            else res[0][u] = -s4[u];
        }
    }
}
__device__ __forceinline__ void chs_inv_store(double* Ls, int I0, int nb, int pair, int lane, const double (&res)[2][4]) {
    const int c8 = lane & 7, tq = lane >> 3;
    const int nblk = I0 >> 3;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int c = (half ? nblk - 1 - pair : pair) * 8 + c8;
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (tq + 4 * u < nb) Ls[tri(I0 + tq + 4 * u, c)] = res[half][u];
    }
}

template <int KM, int CHS_T, int KMIN, int MINB = 1>
__global__ void __launch_bounds__(CHS_T, MINB) k_chol_sm(DevView v) {
    extern __shared__ __align__(16) double sm[];
    const int b = blockIdx.x;
    const int k = 2 * v.ksel[b];
    if (k == 0 || k > KM || k <= KMIN) return;
    const int kmax = v.kmax;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nwarps = CHS_T / 32;
    const double* __restrict__ S = v.Sb + (size_t)b * kmax * kmax;
    double* __restrict__ Xg = v.Li + (size_t)b * kmax * kmax;
    double* Ls = sm;                                   // packed lower triangle: L, then inv(L) in place
    double* D = Ls + CHS_TRI(KM);                      // [NB][NB+1] diagonal block factor
    double* DiA = D + NB * (NB + 1);                   // [2][NB][NB+1] its inverse: this panel's and the previous one's
    double* Pn = DiA + 2 * NB * (NB + 1);              // [NB][KM] transposed panel of the trailing update / vectors
    __shared__ int s_bad;
    if (tid == 0) s_bad = 0;
    // every element of the lower triangle is its own 8-byte asynchronous copy (LDGSTS.64): ~20 independent copies in
    // flight per thread instead of a dependent DRAM round trip per row (ncu: 11 % of the kernel's samples sat on the
    // plain load loop; k_chol 1.42 -> 1.33 ms)
    for (int r = warp; r < k; r += nwarps)
        for (int c = lane; c <= r; c += 32) cp_async8(Ls + tri(r, c), S + (size_t)r * kmax + c);
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();

    for (int j0 = 0; j0 < k; j0 += NB) {
        const int nb = min(NB, k - j0);
        double* Di = DiA + ((j0 >> 4) & 1) * NB * (NB + 1);
        const double* Dip = DiA + (((j0 >> 4) & 1) ^ 1) * NB * (NB + 1);
        double res[2][4];
        // While warp 0 walks the serial pivot chain of diagonal block j, the other warps form block row j-1 of inv(L): its
        // rows of L are final, its diagonal block inverse is Dip, the rows of X above it were stored one panel ago.
        // At most nwarps - 1 column-block pairs exist here (block row j-1 has j-1 pairs, j <= KM/16 - 1).
        const bool inv_prev = warp > 0 && j0 >= 2 * NB && (warp - 1) < ((j0 - NB) >> 4);
        for (int e = tid; e < NB * NB; e += CHS_T) {
            const int r = e / NB, c = e - r * NB;
            D[r * (NB + 1) + c] = (r < nb && c <= r) ? Ls[tri(j0 + r, j0 + c)] : ((r >= nb && r == c) ? 1.0 : 0.0);
            Di[r * (NB + 1) + c] = 0.0;
        }
        __syncthreads();
        if (warp == 0) {
            if (chol16_warp(D, NB + 1, Di) && lane == 0) s_bad = 1;
        }
        else if (inv_prev) chs_inv_compute(Ls, Dip, j0 - NB, NB, warp - 1, lane, res);
        __syncthreads();
        if (inv_prev) chs_inv_store(Ls, j0 - NB, NB, warp - 1, lane, res);
        // the diagonal block of X replaces the one of L (the panel solve and the inverse phase only use Di)
        for (int e = tid; e < nb * nb; e += CHS_T) {
            const int r = e / nb, c = e - r * nb;
            if (c <= r) Ls[tri(j0 + r, j0 + c)] = Di[r * (NB + 1) + c];
        }
        // panel: L[i][j0+c] = sum_{t<=c} S[i][j0+t] * Di[c][t]; a transposed copy PT[c][i - i1] feeds the trailing update
        const int i1 = j0 + nb;
        const int m = k - i1;                 // m > 0 implies nb == NB
        double* PT = Pn;                      // [NB][KM]
        for (int i = i1 + tid; i < k; i += CHS_T) {
            double2* lrow = reinterpret_cast<double2*>(Ls + tri(i, j0));   // j0 is a multiple of 16: 16-byte aligned
            double row[NB];
#pragma unroll
            for (int t = 0; t < NB; t += 2) { const double2 p = lrow[t >> 1]; row[t] = p.x; row[t + 1] = p.y; }
            double out[NB];
#pragma unroll
            for (int c = 0; c < NB; ++c) {
                double s = 0.0;
#pragma unroll
                for (int t = 0; t <= c; ++t) s += row[t] * Di[c * (NB + 1) + t];
                out[c] = s;
                PT[c * KM + (i - i1)] = s;
            }
#pragma unroll
            for (int c = 0; c < NB; c += 2) lrow[c >> 1] = make_double2(out[c], out[c + 1]);
        }
        if (m > 0 && tid < 4 && m + tid < ((m + 3) & ~3)) {   // rows of the last, partial micro tile
#pragma unroll
            for (int c = 0; c < NB; ++c) PT[c * KM + m + tid] = 0.0;
        }
        __syncthreads();
        // trailing update of the lower triangle: S[i][c] -= sum_t L[i][j0+t] L[c][j0+t]   (4x4 micro tiles)
        if (m > 0) {
            const int mt = (m + 3) / 4;
            const int ntile = mt * (mt + 1) / 2;
            for (int e = tid; e < ntile; e += CHS_T) {
                int ti = (int)((sqrtf(8.0f * e + 1.0f) - 1.0f) * 0.5f);
                while ((ti + 1) * (ti + 2) / 2 <= e) ++ti;
                while (ti * (ti + 1) / 2 > e) --ti;
                const int tj = e - ti * (ti + 1) / 2;
                double acc[4][4];
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int c = 0; c < 4; ++c) acc[a][c] = 0.0;
                const double2* pa = reinterpret_cast<const double2*>(PT + 4 * ti);
                const double2* pc = reinterpret_cast<const double2*>(PT + 4 * tj);
#pragma unroll 4
                for (int t = 0; t < NB; ++t) {
                    const double2 a01 = pa[t * (KM / 2)], a23 = pa[t * (KM / 2) + 1];
                    const double2 c01 = pc[t * (KM / 2)], c23 = pc[t * (KM / 2) + 1];
                    const double ra[4] = {a01.x, a01.y, a23.x, a23.y};
                    const double rc[4] = {c01.x, c01.y, c23.x, c23.y};
#pragma unroll
                    for (int a = 0; a < 4; ++a)
#pragma unroll
                        for (int c = 0; c < 4; ++c) acc[a][c] += ra[a] * rc[c];
                }
                if (ti != tj) {   // all four columns lie left of the diagonal: 128-bit read-modify-writes
#pragma unroll
                    for (int a = 0; a < 4; ++a) {
                        const int ia = ti * 4 + a;
                        if (ia < m) {
                            double2* p = reinterpret_cast<double2*>(Ls + tri(i1 + ia, i1 + tj * 4));
                            double2 u0 = p[0], u1 = p[1];
                            u0.x -= acc[a][0]; u0.y -= acc[a][1]; u1.x -= acc[a][2]; u1.y -= acc[a][3];
                            p[0] = u0; p[1] = u1;
                        }
                    }
                } else {
#pragma unroll
                    for (int a = 0; a < 4; ++a)
#pragma unroll
                        for (int c = 0; c <= a; ++c) {
                            const int ia = ti * 4 + a;
                            if (ia < m) Ls[tri(i1 + ia, i1 + tj * 4 + c)] -= acc[a][c];
                        }
                }
            }
        }
        __syncthreads();
    }

    // the last block row of inv(L) (the others were formed under the pivot chains above): all warps, one pair each
    if (k > NB) {
        const int I0 = ((k - 1) >> 4) << 4;
        const double* Dil = DiA + ((I0 >> 4) & 1) * NB * (NB + 1);
        double res[2][4];
        const bool act = warp < (I0 >> 4);
        if (act) chs_inv_compute(Ls, Dil, I0, k - I0, warp, lane, res);
        __syncthreads();
        if (act) chs_inv_store(Ls, I0, k - I0, warp, lane, res);
        __syncthreads();
    }
    // inv(L) to global memory with explicit zeros above the diagonal (k_gemm streams it unmasked)
    for (int r = warp; r < k; r += nwarps)
        for (int c = lane; c < k; c += 32) Xg[(size_t)r * kmax + c] = (c <= r) ? Ls[tri(r, c)] : 0.0;
    // y = X nu and cv = X' y = inv(S) nu
    double* nu = Pn;            // [k]
    double* ys = Pn + KM;       // [k]
    double* __restrict__ yv = v.yv + (size_t)b * kmax;
    for (int a = tid; a < k; a += CHS_T) nu[a] = yv[a];
    __syncthreads();
    // eight lanes per row, four rows per warp pass: the shuffle chains of the rows overlap
    for (int a0 = warp * 4; a0 < k; a0 += nwarps * 4) {   // warp-uniform trip count: the shuffles below name all 32 lanes
        const int a = a0 + (lane >> 3);
        double s = 0.0;
        if (a < k)
            for (int t = lane & 7; t <= a; t += 8) s += Ls[tri(a, t)] * nu[t];
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (a < k && (lane & 7) == 0) { yv[a] = s; ys[a] = s; }
    }
    __syncthreads();
    double* __restrict__ cv = v.cv + (size_t)b * kmax;
    for (int t = tid; t < k; t += CHS_T) {
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;   // four partial sums: the column is one dependent chain otherwise
        int a = t;
        for (; a + 3 < k; a += 4) {
            s0 += Ls[tri(a, t)] * ys[a];
            s1 += Ls[tri(a + 1, t)] * ys[a + 1];
            s2 += Ls[tri(a + 2, t)] * ys[a + 2];
            s3 += Ls[tri(a + 3, t)] * ys[a + 3];
        }
        for (; a < k; ++a) s0 += Ls[tri(a, t)] * ys[a];
        cv[t] = (s0 + s1) + (s2 + s3);
    }
    if (tid == 0 && s_bad) atomicOr(&v.stats[b].status, 2);
}

// ---------------------------------------------------------------------------------------
// Warp-per-filter variant for k <= 32 (the usual size of the hi update: k ~ 24).  The block-per-filter kernel above spends
// such a filter on two 16-wide panels with a dozen block barriers around a serial pivot chain that only warp 0 walks
// (27 us per CTA, 3 CTAs per SM by registers: 0.25 ms for 4096 filters).  Here lane i holds row i of S in registers
// for the whole factorisation (pivots by rsqrt, columns broadcast by shuffles - the diagonal-block scheme of k_chol_sm,
// 32 wide), lane c then forms column c of X = inv(L) by forward substitution against L in shared memory, and
// y = X nu, inv(S) nu = X' y come from the same shared tile.  No block barrier; four filters per CTA.
// ---------------------------------------------------------------------------------------
#define CHW_K 32
__global__ void __launch_bounds__(128) k_chol_w32(DevView v) {
    __shared__ double Ts[4][CHW_K][CHW_K + 1];   // S (transposing load), then L, then X
    __shared__ double rds[4][CHW_K];             // 1 / L[c][c]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int b = blockIdx.x * 4 + warp;
    if (b >= v.B) return;
    const int k = 2 * v.ksel[b];
    if (k == 0 || k > CHW_K) return;
    const int kmax = v.kmax;
    const unsigned full_mask = 0xffffffffu;
    const double* __restrict__ S = v.Sb + (size_t)b * kmax * kmax;
    double* __restrict__ Xg = v.Li + (size_t)b * kmax * kmax;
    double (*T)[CHW_K + 1] = Ts[warp];
    double* rd = rds[warp];
    // rows of S arrive coalesced (lane = column) and leave the shared tile transposed (lane = row); rows / columns past k
    // are padded with the identity so that the unrolled factorisation below is benign
    for (int r = 0; r < CHW_K; ++r) {
        double val = (r == lane) ? 1.0 : 0.0;
        if (r < k && lane <= r) val = S[(size_t)r * kmax + lane];
        T[r][lane] = val;
    }
    __syncwarp();
    double a[CHW_K];
#pragma unroll
    for (int c = 0; c < CHW_K; ++c) a[c] = (c <= lane) ? T[lane][c] : 0.0;
    __syncwarp();
    bool bad = false;
#pragma unroll
    for (int c = 0; c < CHW_K; ++c) {
        const double piv = __shfl_sync(full_mask, a[c], c);
        bad = bad || !(piv > 0.0);
        const double rs = rsqrt(piv);
        if (lane == c) rd[c] = rs;
        const double lic = (lane == c) ? piv * rs : a[c] * rs;
        a[c] = lic;
#pragma unroll
        for (int j = c + 1; j < CHW_K; ++j) {
            const double ljc = __shfl_sync(full_mask, lic, j);
            a[j] -= lic * ljc;
        }
    }
    // L (lower triangle; what the updates left in the strict upper part of a lane's row is never read)
#pragma unroll
    for (int c = 0; c < CHW_K; ++c) T[lane][c] = a[c];
    __syncwarp();
    // column `lane` of X = inv(L):  X[i][c] = -(sum_{c <= t < i} L[i][t] X[t][c]) / L[i][i],  X[c][c] = 1 / L[c][c]
    double x[CHW_K];
#pragma unroll
    for (int i = 0; i < CHW_K; ++i) {
        double sacc = 0.0;
#pragma unroll
        for (int t = 0; t < i; ++t) sacc += T[i][t] * x[t];
        const double rs = rd[i];
        x[i] = (i == lane) ? rs : ((i > lane) ? -sacc * rs : 0.0);
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < CHW_K; ++i) T[i][lane] = x[i];
    // inv(L) to global memory with explicit zeros above the diagonal, one coalesced row segment per instruction
#pragma unroll
    for (int i = 0; i < CHW_K; ++i)
        if (i < k && lane < k) Xg[(size_t)i * kmax + lane] = x[i];
    __syncwarp();
    // y = X nu (lane = row) and inv(S) nu = X' y (lane = column)
    double* __restrict__ yv = v.yv + (size_t)b * kmax;
    const double nu = (lane < k) ? yv[lane] : 0.0;
    double y = 0.0;
#pragma unroll
    for (int t = 0; t < CHW_K; ++t) {
        const double nt = __shfl_sync(full_mask, nu, t);
        if (t <= lane) y += T[lane][t] * nt;
    }
    if (lane >= k) y = 0.0;
    double s0 = 0.0, s1 = 0.0;
#pragma unroll
    for (int i = 0; i < CHW_K; i += 2) {
        const double y0 = __shfl_sync(full_mask, y, i), y1 = __shfl_sync(full_mask, y, i + 1);
        s0 += T[i][lane] * y0;
        s1 += T[i + 1][lane] * y1;
    }
    if (lane < k) {
        yv[lane] = y;
        v.cv[(size_t)b * kmax + lane] = s0 + s1;
    }
    if (bad && lane == 0) atomicOr(&v.stats[b].status, 2);
}

// ---------------------------------------------------------------------------------------
// Few filters with a large stacked innovation (large maps): the factorisation S = L L' and X = inv(L) run as the
// 64-wide blocked DMMA path of k_chol_big.cu (launch_chol_blocked64); the kernels below finish the job with
// y = X nu and inv(S) nu = X' y, spread over the whole GPU.
// ---------------------------------------------------------------------------------------
// y = X nu (one warp per row) and the explicit zeros k_gemm needs above the diagonal of X: k_gemm streams the rows of
// a 64-row tile up to the tile's last column, so only columns r < c < 64 (r / 64 + 1) are ever read.
// grid = (row chunks of 8, B); the result goes to cv as scratch (yv still holds nu for the other blocks).
__global__ void __launch_bounds__(256) k_mk_y(DevView v) {
    const int b = blockIdx.y;
    const int k = 2 * v.ksel[b];
    const int kmax = v.kmax;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int a = blockIdx.x * 8 + warp;
    if (a >= k) return;
    double* __restrict__ X = v.Li + (size_t)b * kmax * kmax;
    const double* __restrict__ nu = v.yv + (size_t)b * kmax;
    const int cend = min(k, ((a >> 6) + 1) << 6);
    for (int c = a + 1 + lane; c < cend; c += 32) X[(size_t)a * kmax + c] = 0.0;
    double s = 0.0;
    for (int t = lane; t <= a; t += 32) s += X[(size_t)a * kmax + t] * nu[t];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) v.cv[(size_t)b * kmax + a] = s;
}
// cv = X' y = inv(S) nu.  Column t needs sum_{a >= t} X[a][t] y[a]: one thread per column (coalesced across the
// threads), the row range split in chunks of CV_ROWS over grid.y (one CTA per column chunk was 0.2 ms of serial loop
// per update at k = 1000).  y is read from the cv scratch of k_mk_y; partial sums go to out[chunk][kmax] and are added
// up in a fixed order by k_mk_fin.  grid = (column chunks of 128, row chunks, B).
#define CV_ROWS 64
__global__ void __launch_bounds__(128) k_mk_cv(DevView v, double* __restrict__ out, long long out_stride) {
    __shared__ double ysh[CV_ROWS];
    const int b = blockIdx.z;
    const int k = 2 * v.ksel[b];
    const int a0 = blockIdx.y * CV_ROWS;
    const int t0 = blockIdx.x * blockDim.x;
    if (k == 0 || t0 >= k || a0 >= k) return;
    const int kmax = v.kmax;
    const double* __restrict__ X = v.Li + (size_t)b * kmax * kmax;
    const double* __restrict__ y = v.cv + (size_t)b * kmax;
    const int a1 = min(k, a0 + CV_ROWS);
    for (int a = a0 + threadIdx.x; a < a1; a += blockDim.x) ysh[a - a0] = y[a];
    __syncthreads();
    const int t = t0 + threadIdx.x;
    if (t >= k) return;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    int a = max(a0, t);
    for (; a + 3 < a1; a += 4) {
        s0 += X[(size_t)a * kmax + t] * ysh[a - a0];
        s1 += X[(size_t)(a + 1) * kmax + t] * ysh[a + 1 - a0];
        s2 += X[(size_t)(a + 2) * kmax + t] * ysh[a + 2 - a0];
        s3 += X[(size_t)(a + 3) * kmax + t] * ysh[a + 3 - a0];
    }
    for (; a < a1; ++a) s0 += X[(size_t)a * kmax + t] * ysh[a - a0];
    out[(size_t)b * out_stride + (size_t)blockIdx.y * kmax + t] = (s0 + s1) + (s2 + s3);
}
// yv <- y, cv <- inv(S) nu = sum over the row chunks of k_mk_cv (chunks below column t's own chunk hold nothing)
__global__ void k_mk_fin(DevView v, const double* __restrict__ tmp, long long tmp_stride) {
    const int b = blockIdx.y;
    const int k = 2 * v.ksel[b];
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= k) return;
    const size_t o = (size_t)b * v.kmax + t;
    const double yt = v.cv[o];
    double sacc = 0.0;
    for (int ch = t / CV_ROWS; ch * CV_ROWS < k; ++ch) sacc += tmp[(size_t)b * tmp_stride + (size_t)ch * v.kmax + t];
    v.yv[o] = yt;
    v.cv[o] = sacc;
}

static void launch_chol_lockstep(ekfslam_ctx* c) {
    DevView& v = c->v;
    cudaStream_t st = c->stream;
    const int kmax = v.kmax;
    // the launch loops only need to cover the largest stacked update of the batch: read it back (one small
    // synchronous copy; this path is for few filters with large maps, where empty launches cost more)
    cudaMemcpyAsync(c->kmax_host, v.kmaxdev, sizeof(int32_t), cudaMemcpyDeviceToHost, st);
    cudaStreamSynchronize(st);
    const int kact = min(v.kmax, max(0, (int)*c->kmax_host));
    KScope ks(c, KT_CHOL);  // timed as one stage; every launch is counted
    launch_chol_blocked64(c, kact);   // 64-wide panels, panel / trailing / triangular-inverse products on the tensor pipe
    if (kact > 0) {
        // scratch [row chunks][kmax] per filter at the head of its Sb block: the factor L (and the parked T blocks of the
        // blocked inverse) are dead once inv(L) exists (G holds the H P rows)
        double* tmp = v.Sb;
        const long long tstride = (long long)kmax * kmax;
        const int nch = (kact + CV_ROWS - 1) / CV_ROWS;
        dim3 gy((kact + 7) / 8, v.B), gc((kact + 127) / 128, nch, v.B), gf((kact + 127) / 128, v.B);
        k_mk_y<<<gy, 256, 0, st>>>(v);
        k_mk_cv<<<gc, 128, 0, st>>>(v, tmp, tstride);
        k_mk_fin<<<gf, 128, 0, st>>>(v, tmp, tstride);
        c->launches += 2;
    }
}

// ---------------------------------------------------------------------------------------
// Tensor-core GEMM of the update, 64x64 tiles, grid = (row tiles, column groups, B), each CTA walking its column tiles:
//   W[a] = sum_t X[a][t] * G[selrow(t)]       (X = inv(L), lower triangular, explicit zeros above the
//   diagonal; G_sel = the selected rows of G).  The last row tile also accumulates the state update
//   x+ = x + G_sel' inv(S) nu (mc/update.m:12) for its 64 columns, and column tile 0 then computes normJac(q+) and
//   normalises the quaternion (mc/update.m:18,24) when `finalize`.
// ---------------------------------------------------------------------------------------
// One K chunk (TK = 16 rows of the staged panels) of k_gemm for a warp's 8-row tiles [MT0, MT1): branch-free, fully
// unrolled.  HALF: tile MT0 sits on the diagonal and only needs K steps 0-1 (X = inv(L) has explicit zeros above it).
template <int MT0, int MT1, bool HALF>
__device__ __forceinline__ void gemm_chunk(const double* __restrict__ ap, const double* __restrict__ bp, double (&acc)[4][2][2]) {
#pragma unroll
    for (int k4 = 0; k4 < TK / 4; ++k4) {
        double af[4], bf[2];
#pragma unroll
        for (int mt = MT0; mt < MT1; ++mt) af[mt] = ap[mt * 8 * APAD + k4 * 4];
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) bf[nt] = bp[k4 * 4 * TPAD + nt * 8];
#pragma unroll
        for (int mt = MT0; mt < MT1; ++mt) {
            if (mt == MT0 && HALF && k4 >= 2) continue;
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) dmma(acc[mt][nt], af[mt], bf[nt]);
        }
    }
}

template <int mode>   // only mode 0 exists (the name k_gemm<0> is what the committed ncu profiles show)
__global__ void __launch_bounds__(256, 3) k_gemm(DevView v, int finalize, int kskip) {
    extern __shared__ __align__(16) double dsm[];
    const int b = blockIdx.z;
    const int k = 2 * v.ksel[b];                        // rows of the output
    const int kk = k;                                   // contraction length
    const int a0 = blockIdx.x * TM;
    if (a0 >= k || kk == 0 || k <= kskip) return;       // k <= kskip: handled by k_w_small
    const int n = v.nstate[b];
    const int ld = v.ld, kmax = v.kmax;
    const double* __restrict__ A = v.Li + (size_t)b * kmax * kmax;
    double* __restrict__ G = v.G + (size_t)b * kmax * ld;
    double* __restrict__ W = v.W + (size_t)b * v.wstride;
    const int* __restrict__ sel = v.sel + (size_t)b * v.N;

    double* As = dsm;                           // [NSTAGE][64][APAD]   As[i][t] = A[a0+i][t0+t]
    double* Bs = dsm + NSTAGE * TM * APAD;      // [NSTAGE][TK][TPAD]   Bs[t][j] = B[t0+t][c0+j]
    double* cs = Bs + NSTAGE * TK * TPAD;       // [kmax]               inv(S) nu
    double* xred = cs + kmax;                   // [256]                partial state-update sums
    int* grow = reinterpret_cast<int*>(xred + 256);  // [kmax]  G row of stacked row t: 2 sel[t/2] + (t&1)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wr = warp >> 2, wc = warp & 3, g = lane >> 2, q = lane & 3;
    const bool xrole = a0 + TM >= k;
    if (xrole)
        for (int t = tid; t < k; t += blockDim.x) cs[t] = v.cv[(size_t)b * kmax + t];
    for (int t = tid; t < k; t += blockDim.x) grow[t] = (2 * sel[t >> 1] + (t & 1)) * ld;   // element offset of the G row of stacked row t
    __syncthreads();

    // One CTA owns a 64-row tile of the output for ALL column tiles: the cp.async ring runs over the flattened
    // (column tile, K chunk) sequence, so the pipeline fills once per CTA instead of once per 64x64 tile (short K
    // loops - few stacked rows - were all pipeline fill).
    const int tend = min(k, a0 + TM);  // X[a][t] = 0 for t > a
    const int nk = (tend + TK - 1) / TK;
    // column tiles [cb0, cb1) of this CTA: gridDim.y CTAs share the column tiles of one row tile (1 = the CTA walks them
    // all; more = shorter CTAs, for launches where few filters have work)
    const int ncb_all = (n + TM - 1) / TM;
    const int cb0 = (int)(((long long)ncb_all * blockIdx.y) / gridDim.y), ncb = (int)(((long long)ncb_all * (blockIdx.y + 1)) / gridDim.y);
    if (cb0 >= ncb) return;
    const int total = (ncb - cb0) * nk;
    // this thread's two 16-byte pieces of an A stage (64 rows x 8 chunks) and of a B stage (16 rows x 32 chunks)
    const int ar = tid >> 3, acc2 = (tid & 7) * 2;
    const int br = tid >> 5, bcc = (tid & 31) * 2;
    // per-thread invariants of a stage load (the address arithmetic of four copies was ~200 instructions per chunk:
    // three times the tensor work of the chunk)
    const bool aok0 = a0 + ar < k, aok1 = a0 + ar + 32 < k;
    const double* ap0 = A + (size_t)(aok0 ? a0 + ar : 0) * kmax + acc2;
    const double* ap1 = A + (size_t)(aok1 ? a0 + ar + 32 : 0) * kmax + acc2;
    const double* gcol = G + bcc;
    unsigned ad0 = (unsigned)__cvta_generic_to_shared(As + ar * APAD + acc2);   // + st * TM * APAD * 8; second piece + 32 rows
    unsigned bd0 = (unsigned)__cvta_generic_to_shared(Bs + br * TPAD + bcc);    // + st * TK * TPAD * 8; second piece + 8 rows
    // opaque to the optimiser: left alone it REMATERIALISES these (block index, 64-bit products, ...) at every use
    asm volatile("" : "+l"(ap0), "+l"(ap1), "+l"(gcol), "+r"(ad0), "+r"(bd0));
    auto cpa = [](unsigned dst, const double* src, int bytes) {
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(bytes) : "memory");
    };
    auto load_stage = [&](int st, int cb, int it) {
        const int t0 = it * TK, c0 = cb * TM;
        const unsigned ad = ad0 + st * (TM * APAD * 8);
        const unsigned bd = bd0 + st * (TK * TPAD * 8);
        const bool tok = t0 + acc2 < kk;
        cpa(ad, (aok0 && tok) ? ap0 + t0 : ap0, (aok0 && tok) ? 16 : 0);
        cpa(ad + 32 * APAD * 8, (aok1 && tok) ? ap1 + t0 : ap1, (aok1 && tok) ? 16 : 0);
        const bool cok = c0 + bcc < ld;
#pragma unroll
        for (int j = 0; j < 2; ++j) {   // B: rows br, br + 8
            const int tt = t0 + br + 8 * j;
            const bool ok = cok && tt < kk;
            const double* src = gcol;
            if (ok) src = gcol + grow[tt] + c0;
            cpa(bd + j * (8 * TPAD * 8), src, ok ? 16 : 0);
        }
    };
    double acc[4][2][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    double xacc = 0.0;
    const int tmax_w = min(k, a0 + wr * 32 + 32);
    const int rbase = a0 + wr * 32;
    const int mt_hi = max(0, min(4, (k - rbase + 7) >> 3));

    int lcb = cb0, lit = 0;   // (column tile, chunk) of the next stage to load
#pragma unroll
    for (int st = 0; st < NSTAGE - 1; ++st) {
        if (lcb < ncb) { load_stage(st, lcb, lit); if (++lit == nk) { lit = 0; ++lcb; } }
        cp_async_commit();
    }
    int cb = cb0, it = 0;
    int cst = 0, lst = NSTAGE - 1;   // stage being consumed / stage being loaded (ring counters instead of j % NSTAGE)
    for (int j = 0; j < total; ++j) {
        cp_async_wait<NSTAGE - 2>();
        __syncthreads();
        if (lcb < ncb) { load_stage(lst, lcb, lit); if (++lit == nk) { lit = 0; ++lcb; } }
        cp_async_commit();
        if (++lst == NSTAGE) lst = 0;
        const double* as = As + cst * TM * APAD;
        const double* bs = Bs + cst * TK * TPAD;
        if (++cst == NSTAGE) cst = 0;
        if (xrole) {
            // state update G_sel' inv(S) nu for this column tile: thread (column tid & 63, quarter tid >> 6) takes four
            // of the chunk's 16 rows; the four partial sums meet in shared memory at the end of the column tile
            const int xc = tid & (TM - 1), t4 = (tid >> 6) * 4;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int tt = it * TK + t4 + t;
                if (tt < k) xacc += bs[(t4 + t) * TPAD + xc] * cs[tt];
            }
        }
        // 8-row tile mt of this warp (rows rbase + 8 mt ..) takes part in step tb when it exists (mt < mt_hi) and,
        // for the triangular A of mode 0, when tb <= its last row (mt >= mt_lo): a contiguous range.  Steps where all
        // four take part run branch-free (a predicated mma.sync costs a WARPSYNC/NOP pair and a predicate each).
        const double* ap = as + (wr * 32 + g) * APAD + q;
        const double* bp = bs + q * TPAD + wc * 16 + g;
        const int tb0 = it * TK;
        // Every chunk a warp needs runs one branch-free block over its existing 8-row tiles x all four K steps.  A has
        // explicit zeros above the diagonal and zero-filled columns beyond k, so the products a per-K-step triangular
        // dispatch would skip (a jump table per K step: ~20 instructions and an indirect branch for <= 8 DMMAs) are
        // multiplications by zero; the tensor pipe was 37 % busy and the issue slots 63 %, so trading issue for DMMAs wins.
        if (mt_hi > 0 && tb0 < tmax_w) {
            // d = chunk start relative to the warp's first row (a multiple of 16).  Left of the diagonal (d < 0) every
            // product is needed.  On the diagonal only part is: d = 0 -> tile 0 needs K steps 0-1; d = 16 -> tiles 0, 1
            // need nothing, tile 2 needs K steps 0-1.  The 8-row tiles beyond the last stacked row (mt >= mt_hi: the
            // lower warps of the last row tile, e.g. rows 96..102 of k = 103 fill ONE of their four tiles) are skipped as
            // well: they made those warps the longest of the CTA while 3/4 of their DMMAs multiplied zeros.  All blocks are
            // compile-time, one warp-uniform dispatch per chunk (a jump table per K step cost more than the DMMAs it saved).
            const int d = tb0 - rbase;
            switch (mt_hi) {
                case 4:
                    if (d < 0) gemm_chunk<0, 4, false>(ap, bp, acc);
                    else if (d == 0) gemm_chunk<0, 4, true>(ap, bp, acc);
                    else gemm_chunk<2, 4, true>(ap, bp, acc);
                    break;
                case 3:
                    if (d < 0) gemm_chunk<0, 3, false>(ap, bp, acc);
                    else if (d == 0) gemm_chunk<0, 3, true>(ap, bp, acc);
                    else gemm_chunk<2, 3, true>(ap, bp, acc);
                    break;
                case 2:
                    if (d < 0) gemm_chunk<0, 2, false>(ap, bp, acc);
                    else if (d == 0) gemm_chunk<0, 2, true>(ap, bp, acc);
                    break;
                default:
                    if (d < 0) gemm_chunk<0, 1, false>(ap, bp, acc);
                    else if (d == 0) gemm_chunk<0, 1, true>(ap, bp, acc);
                    break;
            }
        }
        if (++it < nk) continue;
        // ---- last chunk of column tile cb: store the 64x64 tile, fold the state update, restart the accumulators
        const int c0 = cb * TM;
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) {
            const int a = a0 + wr * 32 + mt * 8 + g;
            if (a < k) {
                // the 64 output columns of a column tile are one panel of W
                double* __restrict__ orow = W + w_at(v.wrows, a, c0) - c0;
#pragma unroll
                for (int nt = 0; nt < 2; ++nt) {
                    const int c = c0 + wc * 16 + nt * 8 + 2 * q;
                    if (c < ld) {  // ld is even: c+1 < ld as well; the padding columns [n, ld) are kept zero
                        double2 o;
                        o.x = (c < n) ? acc[mt][nt][0] : 0.0;
                        o.y = (c + 1 < n) ? acc[mt][nt][1] : 0.0;
                        *reinterpret_cast<double2*>(orow + c) = o;
                    }
                }
            }
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
        }
        if (xrole) {
            double* __restrict__ x = v.x + (size_t)b * ld;
            xred[tid] = xacc;
            xacc = 0.0;
            __syncthreads();
            if (tid < TM && c0 + tid < n) x[c0 + tid] += (xred[tid] + xred[tid + 64]) + (xred[tid + 128] + xred[tid + 192]);
            if (c0 == 0 && finalize) {
                // this block owns state entries 0..63, the quaternion among them
                __syncthreads();
                if (tid == 0) normjac_normalize(x, v.jnt + (size_t)b * 16);
            }
        }
        it = 0; ++cb;
    }
    cp_async_wait<0>();
}

// ---------------------------------------------------------------------------------------
// k_gemm(mode 0) for few stacked rows (k <= WS_K, the usual size of the hi update): W = inv(L) G_sel is a
// (k x k) x (k x n) product per filter - 64-row DMMA tiles would be mostly padding and every CTA mostly pipeline
// latency.  One block per filter, one state column per thread: the k entries of the column of G_sel stay in
// registers, inv(L) is broadcast from shared memory.  Same epilogue duties as k_gemm: x+ = x + G_sel' inv(S) nu,
// normJac(q+) and the quaternion normalisation.
// ---------------------------------------------------------------------------------------
#define WS_K 32    // k <= 32 (a second launch of this kernel for 32 < k <= 48 - 152 registers, 2 CTAs per SM - lost to the DMMA tiles
                   // of k_gemm: k_w_hi 0.47 -> 0.65 ms)
template <int KW, int KMIN, int MINB>
__global__ void __launch_bounds__(128, MINB) k_w_small(DevView v, int finalize) {
    const int b = blockIdx.x;
    const int k = 2 * v.ksel[b];
    if (k <= KMIN || k > KW) return;
    const int n = v.nstate[b], ld = v.ld, kmax = v.kmax;
    const double* __restrict__ Xg = v.Li + (size_t)b * kmax * kmax;
    const double* __restrict__ G = v.G + (size_t)b * kmax * ld;
    double* __restrict__ W = v.W + (size_t)b * v.wstride;
    const int* __restrict__ sel = v.sel + (size_t)b * v.N;
    __shared__ double Xs[KW][KW + 1];
    __shared__ double cs[KW];
    __shared__ int grow[KW];
    const int tid = threadIdx.x;
    for (int e = tid; e < KW * KW; e += blockDim.x) {
        const int a = e / KW, t = e - a * KW;
        Xs[a][t] = (a < k && t <= a) ? Xg[(size_t)a * kmax + t] : 0.0;
    }
    if (tid < KW) {
        cs[tid] = (tid < k) ? v.cv[(size_t)b * kmax + tid] : 0.0;
        grow[tid] = (tid < k) ? 2 * sel[tid >> 1] + (tid & 1) : 0;
    }
    __syncthreads();
    double* __restrict__ x = v.x + (size_t)b * ld;
    // A thread walks its columns one after the other, and every column started with a DRAM round trip for its k entries of
    // G before any arithmetic could begin (16 warps per SM, in-order issue: the launch ran at a third of the HBM rate).  Each
    // thread now requests the entries of its NEXT column as asynchronous copies into its own slots of a double-buffered
    // shared tile (only the thread itself reads them back: no barrier) while it works on the current one.
    extern __shared__ __align__(16) double gsm[];   // [2][KW][128]
    auto prefetch = [&](int buf, int c) {
        double* dst = gsm + (size_t)buf * KW * 128 + tid;
#pragma unroll
        for (int t = 0; t < KW; ++t)
            if (t < k) cp_async8(dst + t * 128, G + (size_t)grow[t] * ld + c);
        cp_async_commit();
    };
    if (tid < ld) prefetch(0, tid);
    int buf = 0;
    for (int c = tid; c < ld; c += blockDim.x, buf ^= 1) {
        cp_async_wait<0>();
        if (c + (int)blockDim.x < ld) prefetch(buf ^ 1, c + blockDim.x);
        double g[KW];
        const double* src = gsm + (size_t)buf * KW * 128 + tid;
#pragma unroll
        for (int t = 0; t < KW; ++t) g[t] = (t < k) ? src[t * 128] : 0.0;
        const bool incol = c < n;
        double xs = 0.0;
#pragma unroll
        for (int t = 0; t < KW; ++t) xs += g[t] * cs[t];
        double* __restrict__ wcol = W + w_at(v.wrows, 0, c);
#pragma unroll
        for (int a = 0; a < KW; ++a) {
            if (a < k) {
                double sacc = 0.0;
#pragma unroll
                for (int t = 0; t <= a; ++t) sacc += Xs[a][t] * g[t];
                wcol[(size_t)a * EKF_WPAD] = incol ? sacc : 0.0;   // the padding columns [n, ld) are kept zero
            }
        }
        if (incol) x[c] += xs;
    }
    if (finalize) {
        __syncthreads();
        if (tid == 0) normjac_normalize(x, v.jnt + (size_t)b * 16);
    }
}

// ---------------------------------------------------------------------------------------
// After k_gemm: fold this update's normalisation Jacobian Jt into W and do the bookkeeping.
//   mc/update.m:20-22 is  P+ = J (P - W'W) J' = J P J' - (W J')' (W J')  with J = blkdiag(I3, Jt, I): only columns
//   3..6 of W change; the covariance downdate applies J to the P tiles themselves.
// One block per filter.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_wfix(DevView v) {
    const int b = blockIdx.x;
    const int k = 2 * v.ksel[b];
    double* __restrict__ W = v.W + (size_t)b * v.wstride;
    __shared__ double Jt[16];
    if (threadIdx.x < 16) Jt[threadIdx.x] = v.jnt[(size_t)b * 16 + threadIdx.x];
    __syncthreads();
    for (int a = threadIdx.x; a < k; a += blockDim.x) w_fold_jt(W + w_at(v.wrows, a, 3), Jt);
    if (threadIdx.x < 16 && k > 0) v.jn[(size_t)b * 16 + threadIdx.x] = Jt[threadIdx.x];
    if (threadIdx.x == 0) v.ktot[b] = k;
}

static void gemm_attr(ekfslam_ctx* c, size_t w_sm) {
    ENSURE_DYN_SMEM(k_gemm<0>, w_sm, c->device);
}

void launch_update(ekfslam_ctx* c, int mask, int which_prior, int flags) {
    // flags: 1 = iterated-update innovation (see k_upd_S), 2 = not the final iteration (no quaternion
    // normalisation, no covariance downdate)
    DevView& v = c->v;
    cudaStream_t st = c->stream;
    const bool hi = (mask & EKFSLAM_F_HI) != 0;
    cudaMemsetAsync(v.kmaxdev, 0, sizeof(int32_t), st);
    {
        KScope ks(c, hi ? KT_UPD_S_HI : KT_UPD_S);
        const int slices = (v.B < 296) ? (int)((8 * 148 + v.B - 1) / v.B) : 1;   // few filters: spread the pair loop
        k_upd_S<<<v.B, 256, 0, st>>>(v, mask, which_prior, flags & 1, slices == 1);
        if (slices > 1) { dim3 gp(slices, v.B); k_upd_pairs<<<gp, 256, 0, st>>>(v); c->launches++; }
    }
    const size_t chol_sm = sizeof(double) * (2 * NB * (NB + 1) + (size_t)v.kmax * (NB + 1));
    const size_t chs_sm = CHS_SMEM(CHS_K);
    const size_t chss_sm = CHS_SMEM(CHS_KS);
    ENSURE_DYN_SMEM(k_chol, chol_sm, c->device);
    const size_t chsm_sm = CHS_SMEM(CHS_KM);
    ENSURE_DYN_SMEM((k_chol_sm<CHS_KM, 256, 0, 3>), chsm_sm, c->device);
    ENSURE_DYN_SMEM((k_chol_sm<CHS_K, 256, CHS_KM, 2>), chs_sm, c->device);
    ENSURE_DYN_SMEM((k_chol_sm<CHS_K, 256, 0, 2>), chs_sm, c->device);
    ENSURE_DYN_SMEM((k_chol_sm<CHS_K, 256, CHS_KS, 2>), chs_sm, c->device);
    ENSURE_DYN_SMEM((k_chol_sm<CHS_KM, 256, CHS_KS, 3>), chsm_sm, c->device);
    const size_t chl_sm = CHS_SMEM(CHS_KL);
    ENSURE_DYN_SMEM((k_chol_sm<CHS_KL, 512, CHS_K, 1>), chl_sm, c->device);
    // One block per filter fills the GPU once there are a few hundred filters (measured B=4096, k~98: block
    // 2.2 ms, lock-step 3.8 ms).  Few filters with a large stacked innovation (large maps): the single block is a
    // serial bottleneck (N=500, B=8: 7.1 of 11.5 ms per step), so every phase becomes its own launch over all
    // filters with the parallelism that phase has.
    if (chol_lockstep(v)) {
        launch_chol_lockstep(c);
    } else {
        KScope ks(c, hi ? KT_CHOL_HI : KT_CHOL);
        const bool use_mid = v.kmax > CHS_KM;
        // 144 < k <= 200: the few filters of a frame with that many stacked rows used to go through k_chol (S in global
        // memory, one 128-thread CTA each, ~0.28 ms of latency BEHIND the other variants); the resident kernel with 16
        // warps takes them on a second side stream, under the main variant
        const bool large = use_mid && v.kmax > CHS_K;
        auto fork_large = [&]() {   // after ev_fork has been recorded on st
            if (!large) return;
            cudaStreamWaitEvent(c->aux2_stream, c->ev_fork, 0);
            k_chol_sm<CHS_KL, 512, CHS_K, 1><<<v.B, 512, chl_sm, c->aux2_stream>>>(v);
            cudaEventRecord(c->ev_join2, c->aux2_stream);
            c->launches++;
        };
        auto join_large = [&]() { if (large) cudaStreamWaitEvent(st, c->ev_join2, 0); };
        if (hi) {   // few stacked rows are the rule: k <= 32, k <= CHS_KS, CHS_KS < k <= CHS_KM, and the rest
            if (use_mid) {
                // every variant is a chain of latencies that leaves the SMs mostly idle (one CTA per filter, a few hundred
                // filters each): the warp-per-filter kernel (k <= 32) and the rarely used 144-row variant run on one side
                // stream, the 48-row variant (and the 200-row one) on the other, the 112-row variant on the main stream -
                // back to back they took 0.22 ms
                cudaEventRecord(c->ev_fork, st);
                cudaStreamWaitEvent(c->aux_stream, c->ev_fork, 0);
                cudaStreamWaitEvent(c->aux2_stream, c->ev_fork, 0);
                k_chol_w32<<<(v.B + 3) / 4, 128, 0, c->aux_stream>>>(v);
                k_chol_sm<CHS_K, 256, CHS_KM, 2><<<v.B, 256, chs_sm, c->aux_stream>>>(v);
                cudaEventRecord(c->ev_join, c->aux_stream);
                k_chol_sm<CHS_KS, 128, CHW_K><<<v.B, 128, chss_sm, c->aux2_stream>>>(v);
                if (large) { k_chol_sm<CHS_KL, 512, CHS_K, 1><<<v.B, 512, chl_sm, c->aux2_stream>>>(v); c->launches++; }
                cudaEventRecord(c->ev_join2, c->aux2_stream);
                k_chol_sm<CHS_KM, 256, CHS_KS, 3><<<v.B, 256, chsm_sm, st>>>(v);
                cudaStreamWaitEvent(st, c->ev_join, 0);
                cudaStreamWaitEvent(st, c->ev_join2, 0);
                c->launches += 3;
            } else {
                // k <= 32: a warp per filter, no block barriers; the 48-row variant keeps 32 < k <= 48
                k_chol_w32<<<(v.B + 3) / 4, 128, 0, st>>>(v);
                k_chol_sm<CHS_KS, 128, CHW_K><<<v.B, 128, chss_sm, st>>>(v);
                k_chol_sm<CHS_K, 256, CHS_KS, 2><<<v.B, 256, chs_sm, st>>>(v);
                c->launches += 2;
            }
        } else {
            if (use_mid) {   // the common stacked sizes at 3 CTAs/SM, the rest in the large variant on the side stream
                cudaEventRecord(c->ev_fork, st);
                cudaStreamWaitEvent(c->aux_stream, c->ev_fork, 0);
                k_chol_sm<CHS_K, 256, CHS_KM, 2><<<v.B, 256, chs_sm, c->aux_stream>>>(v);
                cudaEventRecord(c->ev_join, c->aux_stream);
                fork_large();
                k_chol_sm<CHS_KM, 256, 0, 3><<<v.B, 256, chsm_sm, st>>>(v);
                cudaStreamWaitEvent(st, c->ev_join, 0);
                join_large();
                c->launches++;
            } else {
                k_chol_sm<CHS_K, 256, 0, 2><<<v.B, 256, chs_sm, st>>>(v);
            }
        }
        const int kres = large ? CHS_KL : CHS_K;   // largest k the resident variants took
        if (v.kmax > kres) { k_chol<<<v.B, 128, chol_sm, st>>>(v, kres); c->launches++; }
    }
    // (64-row tiles, column groups, filters): the li update has work in every filter -> long CTAs that walk all column
    // tiles; the hi update leaves few filters for this kernel (k_w_small takes k <= WS_K) -> two shorter CTAs per row tile
    // (hi: 2 / 3 / 5 / 10 column groups -> k_w_hi 0.43 / 0.44 / 0.47 / 0.56 ms)
    int cg = hi ? 2 : 1;
    // few filters (large maps): split the column tiles so that the grid still fills the GPU
    {
        const long long ctas = (long long)((v.kmax + TM - 1) / TM) * v.B;
        const int want = (int)((8LL * 148 + ctas - 1) / ctas);
        const int ncb_max = (v.nmax + TM - 1) / TM;
        if (want > cg) cg = want < ncb_max ? want : ncb_max;
    }
    dim3 gw((v.kmax + TM - 1) / TM, cg, v.B);
    const size_t w_sm = sizeof(double) * (NSTAGE * (TM * APAD + TK * TPAD) + v.kmax + 256) + sizeof(int) * v.kmax;
    gemm_attr(c, w_sm);
    {
        KScope ks(c, hi ? KT_W_HI : KT_W);
        const int fin = (flags & 2) ? 0 : 1;
        const size_t ws_sm = sizeof(double) * 2 * WS_K * 128;
        ENSURE_DYN_SMEM((k_w_small<WS_K, 0, 3>), ws_sm, c->device);
        k_w_small<WS_K, 0, 3><<<v.B, 128, ws_sm, st>>>(v, fin);
        c->launches++;
        // (a persistent variant over a device-built list of the (filter, row tile) pairs with work was measured in round 2:
        // li 1.51 -> 1.67 ms, hi 0.58 -> 0.55 ms - the CTAs that find nothing to do are not what this launch costs)
        k_gemm<0><<<gw, 256, w_sm, st>>>(v, fin, WS_K);
    }
    if (flags & 2) return;   // not the last iterate of an iterated update: W is recomputed
    { KScope ks(c, KT_WFIX); k_wfix<<<v.B, 128, 0, st>>>(v); }
    if (c->arm_out && (mask & EKFSLAM_F_HI)) { cudaEventRecord(c->ev_out, st); c->arm_out = 0; }  // x, flags, stats are final
    launch_downdate(c, (mask & EKFSLAM_F_HI) ? KT_DOWNDATE_HI : KT_DOWNDATE);
}
