// 1-point RANSAC (mc/ransac_hypotheses.m:3-47) — one thread block per filter.
//
// A hypothesis is fully determined by the feature it draws: xi = x + P H_p' inv(S_p) (z_p - h_p)
// (:22-26).  Rows 2p, 2p+1 of G = H*P (k_hp) are exactly (P H_p')', so
//     xi = x + g0 * G[2p,:] + g1 * G[2p+1,:],   [g0 g1]' = inv(S_p) (z_p - h_p).
// Hypotheses are scored warp-parallel in rounds of RW draws: warp w scores draw i0+w unless the
// drawn feature was already scored (its support is memoised — a repeated draw reproduces the
// same xi bit for bit).  Each lane re-projects matched features at xi
// (mc/compute_hypothesis_support_fast.m) and the inlier count is a ballot/popc reduction.
// After each round thread 0 replays the reference's sequential loop over those draws:
// "first strictly greater support wins" (:37), the adaptive hypothesis count (:40-41, from a
// host-libm table), the n_hyp==0 break (:42) and the i>n_hyp break (:45).
#include <cooperative_groups.h>
#include "model.cuh"
namespace cg = cooperative_groups;

#define RANSAC_WARPS 8
#define RANSAC_THREADS (RANSAC_WARPS * 32)
#ifndef RANSAC_MINB
#define RANSAC_MINB 4   // 64 registers: the kernel is latency-bound, 4 CTAs/SM instead of 2
#endif

// The state corrections of the hypotheses of ONE round (adaptive rule: 8 draws per round, ~7 scored per frame), built on
// demand by the whole block (mc/ransac_hypotheses.m:22-26):
//   xi - x = P H_pos' inv(S_pos) (z_pos - h_pos) = (g' H_pos) P          g = inv(S_pos) nu  (2-vector)
// i.e. ONE combination of the 13 rows of P that H_pos touches, so the 2N-row product G = H P that used to be computed up
// front for this (k_hp over all features) is gone.  Threads along the columns (coalesced rows of P); the 7 camera rows
// are loaded once per column and shared by the round's hypotheses; every load of a column is independent, so a round
// costs ~3 memory round trips (a warp per hypothesis walking its 613 columns took 20).  The combined row lands in row
// 2 pos of the G buffer, where score_hypothesis reads it.
struct HypRound {
    double coef[RANSAC_WARPS][16];   // g'H of the hypothesis of warp w (13 used; Cartesian: columns 10..12 of H are zero)
    int pos[RANSAC_WARPS];           // feature it draws, -1 = nothing to build
    int off[RANSAC_WARPS];           // state offset | Cartesian << 30
};
__device__ __forceinline__ void hyp_gain(const DevView& v, size_t t, double& g0, double& g1) {
    const double s00 = v.S[4 * t], s01 = v.S[4 * t + 1], s10 = v.S[4 * t + 2], s11 = v.S[4 * t + 3];
    const double n0 = v.z[2 * t] - v.h[2 * t], n1 = v.z[2 * t + 1] - v.h[2 * t + 1];
    const double det = s00 * s11 - s01 * s10;
    g0 = (s11 * n0 - s01 * n1) / det;
    g1 = (-s10 * n0 + s00 * n1) / det;
}
__device__ __forceinline__ void build_round_rows(const DevView& v, int b, int n, const HypRound& hr, double* G) {
    const int ld = v.ld;
    const double* __restrict__ P = v.P + (size_t)b * v.nmax * ld;
    for (int c = threadIdx.x; c < n; c += blockDim.x) {
        double cam[7];
#pragma unroll
        for (int r = 0; r < 7; ++r) cam[r] = P[(size_t)r * ld + c];
#pragma unroll
        for (int w = 0; w < RANSAC_WARPS; ++w) {
            const int pos = hr.pos[w];
            if (pos < 0) continue;
            const int off = hr.off[w] & 0x3fffffff;
            const size_t r3 = (hr.off[w] >> 30) ? 0 : 3;   // Cartesian features re-read their first rows for the three missing ones
            const double* __restrict__ Pf = P + (size_t)off * ld + c;
            const double* hs = hr.coef[w];
            double p6[6];
#pragma unroll
            for (int r = 0; r < 3; ++r) { p6[r] = Pf[(size_t)r * ld]; p6[3 + r] = Pf[(r3 + r) * ld]; }
            double d = 0.0;
#pragma unroll
            for (int r = 0; r < 7; ++r) d += hs[r] * cam[r];
#pragma unroll
            for (int r = 0; r < 6; ++r) d += hs[7 + r] * p6[r];
            G[(size_t)(2 * pos) * ld + c] = d;
        }
    }
}

// Support of the hypothesis drawn at feature `pos` (mc/ransac_hypotheses.m:22-33), one warp: lanes re-project the
// matched features at xi; the inlier mask goes to mask[nwords].  Returns the support (same value in every lane).
// rows == 2: rows 2 pos, 2 pos + 1 of G = H P are there (k_hp over the IC features - the fixed-budget configurations
//            score nearly every matched feature, one batched pass beats ~90 row builds):  xi = x + g0 Ga + g1 Gb;
// rows == 1: row 2 pos holds the combined correction (build_round_rows):                  xi = x + Ga.
__device__ __forceinline__ int score_hypothesis(const DevView& v, const DevCam& cam, int b, int pos, const double* xs,
                                                const double* G, const int* moff, const int* mtype,
                                                const double* zs, int nm, double thr, unsigned* mask, int lane, int rows) {
    const int N = v.N, ld = v.ld;
    double f0 = 1.0, f1 = 0.0;
    if (rows == 2) hyp_gain(v, (size_t)b * N + pos, f0, f1);
    const double* Ga = G + (size_t)(2 * pos) * ld;   // (rows == 1: written by this block just before - plain loads)
    const double* Gb = Ga + ld;
    const bool two = rows == 2;
    double c7[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) c7[k] = two ? xs[k] + (Ga[k] * f0 + Gb[k] * f1) : xs[k] + Ga[k];
    double R[9];
    q2r_dev(c7 + 3, R);
    int support = 0;
    for (int j0 = 0; j0 < nm; j0 += 32) {
        const int j = j0 + lane;
        bool inl = false;
        if (j < nm) {
            const int off = moff[j];
            const int ty = mtype[j];
            const int w = (ty == EKFSLAM_FEAT_INVERSEDEPTH) ? 6 : 3;
            double y[6];
#pragma unroll
            for (int k = 0; k < 6; ++k)
                y[k] = (k < w) ? (two ? xs[off + k] + (Ga[off + k] * f0 + Gb[off + k] * f1) : xs[off + k] + Ga[off + k]) : 0.0;
            const double res = support_residual_dev(cam, c7, R, y, ty, zs[2 * j], zs[2 * j + 1]);
            inl = res < thr;
        }
        const unsigned m = __ballot_sync(0xffffffffu, inl);
        support += __popc(m);
        if (lane == 0) mask[j0 >> 5] = m;
    }
    return support;
}

__global__ void __launch_bounds__(RANSAC_THREADS, RANSAC_MINB) k_ransac(DevView v, DevCam cam, ekfslam_params prm, int prebuilt) {
    extern __shared__ unsigned char smem_raw[];
    const int b = blockIdx.x;
    const int n = v.nstate[b];
    const int nf = v.nfeat[b];
    const int N = v.N;
    const int ld = v.ld;
    const int nwords = (N + 31) / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // shared layout
    double* xs = reinterpret_cast<double*>(smem_raw);              // [ld]
    double* zs = xs + ld;                                          // [N][2] z of matched list entries
    int* mlist = reinterpret_cast<int*>(zs + 2 * N);               // [N] matched (HAS_Z) feature indices
    int* moff = mlist + N;                                         // [N] state offset of matched entries
    int* mtype = moff + N;                                         // [N]
    int* iclist = mtype + N;                                       // [N] IC feature indices
    int* memo = iclist + N;                                        // [N] support per feature, -1 = unscored
    unsigned* rmask = reinterpret_cast<unsigned*>(memo + N);       // [RW][nwords]
    unsigned* bestmask = rmask + RANSAC_WARPS * nwords;            // [nwords]  (+ [N][nwords] masks of the fixed-budget path)
    int* dl = reinterpret_cast<int*>(bestmask + nwords + N * nwords);  // [N] distinct drawn features (fixed-budget path)
    __shared__ int s_nm, s_nic, s_done, s_best, s_roundbest, s_nhyp, s_iters, s_scored, s_status;
    __shared__ int rpos[RANSAC_WARPS], rsup[RANSAC_WARPS];
    __shared__ HypRound hround;

    const double* __restrict__ xp = v.xp + (size_t)b * ld;
    double* G = v.G + (size_t)b * v.kmax * ld;
    const uint8_t* __restrict__ fl = v.flags + (size_t)b * N;

    for (int j = tid; j < n; j += blockDim.x) xs[j] = xp[j];
    for (int j = tid; j < N; j += blockDim.x) memo[j] = -1;
    for (int j = tid; j < nwords; j += blockDim.x) bestmask[j] = 0u;
    if (warp == 0) {
        // matched (HAS_Z) and individually compatible (IC) lists in feature order: ballot + prefix popcount
        int nm = 0, nic = 0;
        for (int i0 = 0; i0 < nf; i0 += 32) {
            const int i = i0 + lane;
            const uint8_t f = (i < nf) ? fl[i] : 0;
            const bool hz = (f & EKFSLAM_F_HAS_Z) != 0, ic = (f & EKFSLAM_F_IC) != 0;
            const unsigned mz = __ballot_sync(0xffffffffu, hz), mi = __ballot_sync(0xffffffffu, ic);
            const unsigned below = (1u << lane) - 1u;
            if (hz) {
                const int s = nm + __popc(mz & below);
                mlist[s] = i; moff[s] = v.foff[b * N + i]; mtype[s] = v.ftype[b * N + i];
                zs[2 * s] = v.z[2 * (b * N + i)]; zs[2 * s + 1] = v.z[2 * (b * N + i) + 1];
            }
            if (ic) iclist[nic + __popc(mi & below)] = i;
            nm += __popc(mz); nic += __popc(mi);
        }
        if (lane == 0) {
            s_nm = nm; s_nic = nic; s_done = (nic == 0); s_best = 0; s_roundbest = -1; s_nhyp = prm.max_hyp; s_iters = 0; s_scored = 0;
            s_status = 0;
        }
    }
    __syncthreads();
    const int nm = s_nm, nic = s_nic;
    const int n_loop = (prm.fixed_hyp > 0) ? prm.fixed_hyp : prm.max_hyp;
    const double thr = prm.std_z;
    const double* __restrict__ ub = v.u + (size_t)b * v.n_u;

    if (prm.fixed_hyp > 0 && nic > 0) {
        // ---- fixed hypothesis budget (BASELINE configs 2 and 5: 256 / 512 draws per frame): no adaptive break, so the
        // outcome is "the earliest draw that reaches the maximum support".  All draws are known up front: every DISTINCT
        // drawn feature is scored once, warp-parallel, without the per-round sequential replay of the adaptive path.
        int* need = memo;                                   // reuse: 0/1 drawn flag, then support
        unsigned* masks = reinterpret_cast<unsigned*>(bestmask + nwords);   // [N][nwords] inlier mask per feature
        __shared__ int s_nd;
        __shared__ unsigned long long s_key;
        const int ndraw = min(n_loop, v.n_u);
        for (int j = tid; j < N; j += blockDim.x) need[j] = 0;
        if (tid == 0) { s_nd = 0; s_key = 0ull; }
        __syncthreads();
        for (int it = tid; it < ndraw; it += blockDim.x) {
            int r = (int)floor(ub[it] * (double)nic);
            r = min(r, nic - 1);
            need[iclist[r]] = 1;
        }
        __syncthreads();
        if (warp == 0) {
            int nd = 0;
            for (int i0 = 0; i0 < nf; i0 += 32) {
                const int i = i0 + lane;
                const bool on = (i < nf) && need[i] != 0;
                const unsigned m = __ballot_sync(0xffffffffu, on);
                if (on) dl[nd + __popc(m & ((1u << lane) - 1u))] = i;
                nd += __popc(m);
            }
            if (lane == 0) s_nd = nd;
        }
        __syncthreads();
        const int nd = s_nd;
        for (int d = warp; d < nd; d += RANSAC_WARPS) {
            const int pos = dl[d];
            const int support = score_hypothesis(v, cam, b, pos, xs, G, moff, mtype, zs, nm, thr, masks + pos * nwords, lane, 2);
            if (lane == 0) need[pos] = support;             // need[] now holds the support of every drawn feature
        }
        __syncthreads();
        // earliest draw with the maximum support: key = support << 32 | (0xffffffff - draw index), block-wide max
        unsigned long long key = 0ull;
        for (int it = tid; it < ndraw; it += blockDim.x) {
            int r = (int)floor(ub[it] * (double)nic);
            r = min(r, nic - 1);
            const unsigned long long kq = ((unsigned long long)(unsigned)need[iclist[r]] << 32) | (unsigned long long)(0xffffffffu - (unsigned)it);
            key = kq > key ? kq : key;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
            key = other > key ? other : key;
        }
        if (lane == 0) atomicMax(&s_key, key);
        __syncthreads();
        const int best = (int)(s_key >> 32);
        const int bestit = (int)(0xffffffffu - (unsigned)(s_key & 0xffffffffull));
        if (best > 0) {
            int r = (int)floor(ub[bestit] * (double)nic);
            r = min(r, nic - 1);
            const int bp = iclist[r];
            for (int j = tid; j < nwords; j += blockDim.x) bestmask[j] = masks[bp * nwords + j];
        }
        if (tid == 0) {
            s_best = best; s_iters = ndraw; s_scored = nd; s_done = 1;
            s_status = (n_loop > v.n_u) ? 1 : 0;            // uniform stream exhausted
        }
        __syncthreads();
    }
    for (int i0 = 0; !s_done; i0 += RANSAC_WARPS) {
        // ---- which feature does draw i0+warp select?  (mc/select_random_match.m:12-16)
        const int it = i0 + warp;  // 0-based draw index
        int pos = -1;
        if (it < n_loop && it < v.n_u) {
            int r = (int)floor(ub[it] * (double)nic);
            r = min(r, nic - 1);
            pos = iclist[r];
        }
        if (lane == 0) { rpos[warp] = pos; rsup[warp] = -1; }
        __syncthreads();
        bool score = (pos >= 0) && (memo[pos] < 0);
        for (int w2 = 0; w2 < warp && score; ++w2)
            if (rpos[w2] == pos) score = false;
        if (!prebuilt) {
            // the round's state corrections, built by the whole block
            if (score) {
                const size_t t = (size_t)b * N + pos;
                double g0, g1;
                hyp_gain(v, t, g0, g1);
                const double* __restrict__ H = v.Hc + t * EKF_HSTRIDE;
                if (lane < 13) hround.coef[warp][lane] = g0 * H[lane] + g1 * H[EKF_HC + lane];
                if (lane == 0) { hround.pos[warp] = pos; hround.off[warp] = v.foff[t] | (v.ftype[t] == EKFSLAM_FEAT_INVERSEDEPTH ? 0 : (1 << 30)); }
            } else if (lane == 0) hround.pos[warp] = -1;
            __syncthreads();
            build_round_rows(v, b, n, hround, G);
            __syncthreads();
        }
        if (score) {
            const int support = score_hypothesis(v, cam, b, pos, xs, G, moff, mtype, zs, nm, thr, rmask + warp * nwords, lane, prebuilt ? 2 : 1);
            if (lane == 0) rsup[warp] = support;
        }
        __syncthreads();
        // ---- sequential replay of the reference loop over this round's draws
        if (tid == 0) {
            int best = s_best, bestw = -1, iters = s_iters, scored = s_scored, done = 0, status = s_status;
            int nh = s_nhyp;
            const bool adaptive = prm.fixed_hyp <= 0;
            for (int w2 = 0; w2 < RANSAC_WARPS; ++w2) {
                const int i1 = i0 + w2 + 1;  // 1-based loop counter of the reference
                if (i1 > n_loop) { done = 1; break; }               // for i = 1:n_hyp ran out
                if (i1 > v.n_u) { status |= 1; done = 1; break; }   // uniform stream exhausted
                const int p = rpos[w2];
                iters = i1;
                int sup = memo[p];
                if (sup < 0) { sup = rsup[w2]; memo[p] = sup; ++scored; }
                if (sup > best) {                                    // :37
                    best = sup; bestw = w2;
                    if (adaptive) {
                        nh = v.nhyp_tab[EKF_TRI(nic, min(sup, nic))];  // :40-41
                        if (nh == 0) { done = 1; break; }              // :42
                    }
                }
                if (adaptive && i1 > nh) { done = 1; break; }        // :45
            }
            s_best = best; s_iters = iters; s_scored = scored; s_status = status; s_nhyp = nh;
            s_roundbest = bestw;
            s_done = done;
        }
        __syncthreads();
        const int bw = s_roundbest;
        if (bw >= 0)
            for (int j = tid; j < nwords; j += blockDim.x) bestmask[j] = rmask[bw * nwords + j];
        __syncthreads();
    }

    // ---- mc/set_as_most_supported_hypothesis.m:6-27 (only if some hypothesis had support > 0)
    if (s_best > 0) {
        for (int j = tid; j < nm; j += blockDim.x) {
            const int i = mlist[j];
            const bool inl = (bestmask[j >> 5] >> (j & 31)) & 1u;
            uint8_t f = v.flags[(size_t)b * N + i];
            f = inl ? (f | EKFSLAM_F_LI) : (f & ~EKFSLAM_F_LI);
            v.flags[(size_t)b * N + i] = f;
        }
    }
    if (tid == 0) {
        ekfslam_stats& st = v.stats[b];
        st.n_ic = nic; st.ransac_iters = s_iters; st.ransac_scored = s_scored; st.max_support = s_best;
        st.status = s_status; st.n_li = 0; st.n_hi = 0; st.reserved = 0;
    }
}

// ---------------------------------------------------------------------------------------
// Latency path (few filters, fixed hypothesis budget - BASELINE config 2: ONE filter, 256 hypotheses per frame):
// a thread-block CLUSTER of RANSAC_CLUSTER CTAs per filter.  Every CTA builds the (identical) match / draw lists, the
// distinct drawn features are dealt round robin to the CTAs of the cluster (8 warps each), and CTA 0 collects the
// supports and the winner's inlier mask through distributed shared memory (cluster.map_shared_rank) - no global
// scratch, no second launch.  Same outcome as the fixed-budget branch of k_ransac: "the earliest draw that reaches
// the maximum support" (mc/ransac_hypotheses.m:37 with :41-45 disabled).
// ---------------------------------------------------------------------------------------
#define RANSAC_CLUSTER 8
__global__ void __launch_bounds__(RANSAC_THREADS) k_ransac_fixed_cluster(DevView v, DevCam cam, ekfslam_params prm, int prebuilt) {
    cg::cluster_group cluster = cg::this_cluster();
    const int C = (int)cluster.num_blocks();
    const int rank = (int)cluster.block_rank();
    extern __shared__ unsigned char smem_raw[];
    const int b = blockIdx.x / C;
    const int n = v.nstate[b], nf = v.nfeat[b], N = v.N, ld = v.ld;
    const int nwords = (N + 31) / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double* xs = reinterpret_cast<double*>(smem_raw);              // [ld]
    double* zs = xs + ld;                                          // [N][2]
    int* mlist = reinterpret_cast<int*>(zs + 2 * N);               // [N]
    int* moff = mlist + N;                                         // [N]
    int* mtype = moff + N;                                         // [N]
    int* iclist = mtype + N;                                       // [N]
    int* need = iclist + N;                                        // [N] drawn flag, then support (of the features this CTA scored)
    int* dl = need + N;                                            // [N] distinct drawn features, feature order
    int* own = dl + N;                                             // [N] cluster rank that scores feature i
    unsigned* masks = reinterpret_cast<unsigned*>(own + N);        // [N][nwords] inlier mask per scored feature
    __shared__ int s_nm, s_nic, s_nd;
    __shared__ unsigned long long s_key;

    const double* __restrict__ xp = v.xp + (size_t)b * ld;
    double* G = v.G + (size_t)b * v.kmax * ld;
    const uint8_t* __restrict__ fl = v.flags + (size_t)b * N;
    for (int j = tid; j < n; j += blockDim.x) xs[j] = xp[j];
    for (int j = tid; j < N; j += blockDim.x) { need[j] = 0; own[j] = 0; }
    if (tid == 0) { s_nd = 0; s_key = 0ull; }
    if (warp == 0) {
        int nm = 0, nic = 0;
        for (int i0 = 0; i0 < nf; i0 += 32) {
            const int i = i0 + lane;
            const uint8_t f = (i < nf) ? fl[i] : 0;
            const bool hz = (f & EKFSLAM_F_HAS_Z) != 0, ic = (f & EKFSLAM_F_IC) != 0;
            const unsigned mz = __ballot_sync(0xffffffffu, hz), mi = __ballot_sync(0xffffffffu, ic);
            const unsigned below = (1u << lane) - 1u;
            if (hz) {
                const int s2 = nm + __popc(mz & below);
                mlist[s2] = i; moff[s2] = v.foff[b * N + i]; mtype[s2] = v.ftype[b * N + i];
                zs[2 * s2] = v.z[2 * (b * N + i)]; zs[2 * s2 + 1] = v.z[2 * (b * N + i) + 1];
            }
            if (ic) iclist[nic + __popc(mi & below)] = i;
            nm += __popc(mz); nic += __popc(mi);
        }
        if (lane == 0) { s_nm = nm; s_nic = nic; }
    }
    __syncthreads();
    const int nm = s_nm, nic = s_nic;
    const int n_loop = prm.fixed_hyp;
    const int ndraw = min(n_loop, v.n_u);
    const double thr = prm.std_z;
    const double* __restrict__ ub = v.u + (size_t)b * v.n_u;
    if (nic > 0) {
        for (int it = tid; it < ndraw; it += blockDim.x) {
            int r = (int)floor(ub[it] * (double)nic);
            r = min(r, nic - 1);
            need[iclist[r]] = 1;
        }
        __syncthreads();
        if (warp == 0) {
            int nd = 0;
            for (int i0 = 0; i0 < nf; i0 += 32) {
                const int i = i0 + lane;
                const bool on = (i < nf) && need[i] != 0;
                const unsigned m = __ballot_sync(0xffffffffu, on);
                if (on) {
                    const int d = nd + __popc(m & ((1u << lane) - 1u));
                    dl[d] = i;
                    own[i] = (d / RANSAC_WARPS) % C;
                }
                nd += __popc(m);
            }
            if (lane == 0) s_nd = nd;
        }
        __syncthreads();
        const int nd = s_nd;
        for (int d = rank * RANSAC_WARPS + warp; d < nd; d += C * RANSAC_WARPS) {
            const int pos = dl[d];
            const int support = score_hypothesis(v, cam, b, pos, xs, G, moff, mtype, zs, nm, thr, masks + pos * nwords, lane, 2);
            if (lane == 0) need[pos] = support;
        }
    }
    cluster.sync();                                                // every CTA's supports / masks are in its shared memory
    if (rank == 0) {
        int best = 0;
        if (nic > 0) {
            const int nd = s_nd;
            for (int d = tid; d < nd; d += blockDim.x) {
                const int pos = dl[d], o = own[pos];
                if (o != 0) need[pos] = cluster.map_shared_rank(need, o)[pos];
            }
            __syncthreads();
            unsigned long long key = 0ull;
            for (int it = tid; it < ndraw; it += blockDim.x) {
                int r = (int)floor(ub[it] * (double)nic);
                r = min(r, nic - 1);
                const unsigned long long kq = ((unsigned long long)(unsigned)need[iclist[r]] << 32) | (unsigned long long)(0xffffffffu - (unsigned)it);
                key = kq > key ? kq : key;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
                key = other > key ? other : key;
            }
            if (lane == 0) atomicMax(&s_key, key);
            __syncthreads();
            best = (int)(s_key >> 32);
            if (best > 0) {
                const int bestit = (int)(0xffffffffu - (unsigned)(s_key & 0xffffffffull));
                int r = (int)floor(ub[bestit] * (double)nic);
                r = min(r, nic - 1);
                const int bp = iclist[r];
                const unsigned* bm = cluster.map_shared_rank(masks, own[bp]) + bp * nwords;
                // mc/set_as_most_supported_hypothesis.m:6-27
                for (int j = tid; j < nm; j += blockDim.x) {
                    const int i = mlist[j];
                    const bool inl = (bm[j >> 5] >> (j & 31)) & 1u;
                    uint8_t f = v.flags[(size_t)b * N + i];
                    f = inl ? (f | EKFSLAM_F_LI) : (f & ~EKFSLAM_F_LI);
                    v.flags[(size_t)b * N + i] = f;
                }
            }
        }
        if (tid == 0) {
            ekfslam_stats& st = v.stats[b];
            st.n_ic = nic; st.ransac_iters = nic > 0 ? ndraw : 0; st.ransac_scored = nic > 0 ? s_nd : 0; st.max_support = best;
            st.status = (nic > 0 && n_loop > v.n_u) ? 1 : 0; st.n_li = 0; st.n_hi = 0; st.reserved = 0;
        }
    }
    cluster.sync();                                                // remote shared memory stays valid until CTA 0 is done
}

static size_t ransac_smem_bytes(const DevView& v) {
    const int nwords = (v.N + 31) / 32;
    return sizeof(double) * (v.ld + 2 * v.N) + sizeof(int) * (6 * v.N) +
           sizeof(unsigned) * ((RANSAC_WARPS + 1) * nwords + v.N * nwords) + 16;
}

static size_t ransac_cluster_smem_bytes(const DevView& v) {
    const int nwords = (v.N + 31) / 32;
    return sizeof(double) * (v.ld + 2 * v.N) + sizeof(int) * (7 * v.N) + sizeof(unsigned) * (v.N * nwords) + 16;
}

void launch_ransac(ekfslam_ctx* c) {
    // fixed hypothesis budget (BASELINE configs 2 / 5: 256 / 512 draws): nearly every matched feature is drawn, so the
    // rows H P of the IC features come from one k_hp pass; adaptive rule (~7 scored hypotheses): built on demand
    const int prebuilt = c->prm.fixed_hyp > 0 ? 1 : 0;
    if (prebuilt) launch_hp(c, EKFSLAM_F_HAS_H | EKFSLAM_F_IC, 0);
    KScope ks(c, KT_RANSAC);
    // few filters + fixed hypothesis budget (the latency path): one cluster of CTAs per filter
    if (c->prm.fixed_hyp > 0 && (long long)c->v.B * RANSAC_CLUSTER <= 2LL * c->sm_count) {
        const size_t sm = ransac_cluster_smem_bytes(c->v);
        ENSURE_DYN_SMEM(k_ransac_fixed_cluster, sm, c->device);
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(c->v.B * RANSAC_CLUSTER));
        cfg.blockDim = dim3(RANSAC_THREADS);
        cfg.dynamicSmemBytes = sm;
        cfg.stream = c->stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = RANSAC_CLUSTER; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        cudaLaunchKernelEx(&cfg, k_ransac_fixed_cluster, c->v, c->cam, c->prm, prebuilt);
        return;
    }
    const size_t sm = ransac_smem_bytes(c->v);
    ENSURE_DYN_SMEM(k_ransac, sm, c->device);
    k_ransac<<<c->v.B, RANSAC_THREADS, sm, c->stream>>>(c->v, c->cam, c->prm, prebuilt);
}
