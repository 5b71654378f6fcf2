// Covariance downdate  P <- J P J' - W'W  (mc/update.m:13-22) on 64x64 tiles of the lower triangle.
//
// W holds the ktot rows of one update per filter.  Every row already carries the normalisation
// Jacobian (W <- W J', k_wfix), so J = blkdiag(I3, Jn, I) only has to be applied to the P
// tile itself: columns 3..6 of tile column 0 and rows 3..6 of tile (0,0).  0.5P + 0.5P' (:14) is the identity
// because the lower triangle is authoritative and every tile is stored together with its mirror image.
//
// Two kernels, same arithmetic and summation order (k ascending, DMMA m8n8k4):
//   k_downdate_ws2  (default) persistent, warp-specialised, 2 CTAs per SM: a producer warp streams the W panels with
//                   bulk asynchronous copies (cp.async.bulk -> SASS UBLKCP, one per panel and stage thanks to the
//                   panel-major W layout) on a 4-stage mbarrier ring that keeps running across tile boundaries; 8
//                   consumer warps issue the DMMAs; 4 epilogue warps prefetch the next P tile into shared memory and
//                   store the finished tile and its mirror image while the consumers are already in the next K loop.
//   k_downdate_tile (the fallback for shapes whose tile list does not fit the persistent kernel's shared memory:
//                   n_max > 4352 for the li update, n_max > 4608 for the hi update) one CTA per tile, cp.async (LDGSTS) ring.
#include <cstdlib>
#include "model.cuh"
#include "tc_common.cuh"

#define WS_CONSUMERS 8
#define XP_ 66   // row pitch (doubles) of the shared P tile buffer X of k_downdate_ws2 (= XP below)

// ---- shared epilogue pieces ---------------------------------------------------------------------------
// bit mt*2+nt of the mask: the warp's 8x8 DMMA tile (mt, nt) has work (inside n x n, not strictly above the
// diagonal of a diagonal tile)
__device__ __forceinline__ unsigned tile_mask(int i0, int j0, int wr, int wc, int n, bool diag) {
    unsigned m = 0;
#pragma unroll
    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
            const int r0 = i0 + wr * 32 + mt * 8, c0 = j0 + wc * 16 + nt * 8;
            const bool on = (r0 < n) && (c0 < n) && !(diag && c0 > r0 + 7);
            m |= (on ? 1u : 0u) << (mt * 2 + nt);
        }
    return m;
}

// P tile -> accumulator layout (lane g = lane>>2, q = lane&3 holds rows .. + g, columns .. + 2q, 2q+1)
__device__ __forceinline__ void load_p_frags(const double* __restrict__ P, int ld, int n, int i0, int j0, int wr, int wc,
                                             int g, int q, double (&pf)[4][2][2]) {
#pragma unroll
    for (int mt = 0; mt < 4; ++mt) {
        const int gi = i0 + wr * 32 + mt * 8 + g;
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
            const int gj = j0 + wc * 16 + nt * 8 + 2 * q;
            double2 val = make_double2(0.0, 0.0);
            if (gi < n && gj < ld) val = *reinterpret_cast<const double2*>(P + (size_t)gi * ld + gj);
            pf[mt][nt][0] = val.x; pf[mt][nt][1] = val.y;
        }
    }
}

// J on the P tile of tile column 0: the warps holding columns 0..7 (wc == 0, nt == 0) exchange them through
// a [64][9] strip; 64 threads apply [c3 c4 c5 c6] <- [c3 c4 c5 c6] Jn' per row and, for tile (0,0), rows 3..6 <-
// Jn * rows of the 8x8 corner.  `sync` is the barrier over the participating warps.
template <typename Sync>
__device__ __forceinline__ void apply_j_col0(double* strip, const double* __restrict__ Jn, bool diag, int wr, int wc, int g,
                                             int q, int tid, double (&pf)[4][2][2], Sync sync) {
    if (wc == 0) {
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) {
            strip[(wr * 32 + mt * 8 + g) * 9 + 2 * q] = pf[mt][0][0];
            strip[(wr * 32 + mt * 8 + g) * 9 + 2 * q + 1] = pf[mt][0][1];
        }
    }
    sync();
    if (tid < TM) {
        const int r = tid;
        const double c3 = strip[r * 9 + 3], c4 = strip[r * 9 + 4], c5 = strip[r * 9 + 5], c6 = strip[r * 9 + 6];
#pragma unroll
        for (int a = 0; a < 4; ++a)
            strip[r * 9 + 3 + a] = c3 * Jn[a * 4 + 0] + c4 * Jn[a * 4 + 1] + c5 * Jn[a * 4 + 2] + c6 * Jn[a * 4 + 3];
    }
    sync();
    if (diag) {
        if (tid < 8) {
            const int c = tid;
            const double r3 = strip[3 * 9 + c], r4 = strip[4 * 9 + c], r5 = strip[5 * 9 + c], r6 = strip[6 * 9 + c];
#pragma unroll
            for (int a = 0; a < 4; ++a)
                strip[(3 + a) * 9 + c] = Jn[a * 4 + 0] * r3 + Jn[a * 4 + 1] * r4 + Jn[a * 4 + 2] * r5 + Jn[a * 4 + 3] * r6;
        }
        sync();
    }
    if (wc == 0) {
#pragma unroll
        for (int mt = 0; mt < 4; ++mt) {
            pf[mt][0][0] = strip[(wr * 32 + mt * 8 + g) * 9 + 2 * q];
            pf[mt][0][1] = strip[(wr * 32 + mt * 8 + g) * 9 + 2 * q + 1];
        }
    }
    sync();  // the strip is free again
}

// C = P - acc, stored with its mirror image straight from the accumulator fragments (lanes with equal q cover
// 64-byte runs).  Diagonal tiles: the lower triangle is authoritative, the upper one its mirror.
__device__ __forceinline__ void store_tile(double* __restrict__ P, int ld, int n, int i0, int j0, int wr, int wc, int g, int q,
                                           bool diag, unsigned onmask, const double (&pf)[4][2][2],
                                           const double (&acc)[8][2]) {
#pragma unroll
    for (int mt = 0; mt < 4; ++mt) {
        const int gi = i0 + wr * 32 + mt * 8 + g;
        if (gi >= n) continue;
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) {
            if (!(onmask & (1u << (mt * 2 + nt)))) continue;
            const int gj = j0 + wc * 16 + nt * 8 + 2 * q;
            const double c0 = pf[mt][nt][0] - acc[mt * 2 + nt][0];
            const double c1 = pf[mt][nt][1] - acc[mt * 2 + nt][1];
            if (!diag) {
                if (gj + 1 < n) {
                    *reinterpret_cast<double2*>(P + (size_t)gi * ld + gj) = make_double2(c0, c1);
                    P[(size_t)gj * ld + gi] = c0;
                    P[(size_t)(gj + 1) * ld + gi] = c1;
                } else if (gj < n) {
                    P[(size_t)gi * ld + gj] = c0;
                    P[(size_t)gj * ld + gi] = c0;
                }
            } else {
                if (gj <= gi && gj < n) {
                    P[(size_t)gi * ld + gj] = c0;
                    if (gj < gi) P[(size_t)gj * ld + gi] = c0;
                }
                if (gj + 1 <= gi && gj + 1 < n) {
                    P[(size_t)gi * ld + gj + 1] = c1;
                    if (gj + 1 < gi) P[(size_t)(gj + 1) * ld + gi] = c1;
                }
            }
        }
    }
}


// ---- K chunk: acc += A' B over n4 steps of 4 rows of the staged panels ------------------------------------
// `a` / `b` point at this lane's first fragment element of the stage (q*TPAD + warp offset + g).  A warp whose
// eight 8x8 DMMA tiles all have work (the common case) runs branch-free, fully unrolled code; the compiler
// otherwise brackets every predicated mma.sync with WARPSYNC/NOP and re-derives the predicate per tile, which
// made the DMMA one instruction in ten (ncu, round 1).
__device__ __forceinline__ void mma_step_full(const double* __restrict__ a, const double* __restrict__ b, double (&acc)[8][2]) {
    double af[4], bf[2];
#pragma unroll
    for (int mt = 0; mt < 4; ++mt) af[mt] = a[mt * 8];
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) bf[nt] = b[nt * 8];
#pragma unroll
    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int nt = 0; nt < 2; ++nt) dmma(acc[mt * 2 + nt], af[mt], bf[nt]);
}
__device__ __forceinline__ void mma_chunk(const double* __restrict__ a, const double* __restrict__ b, int n4, unsigned onmask,
                                          double (&acc)[8][2]) {
    if (onmask == 0xffu) {
        if (n4 == TK / 4) {
#pragma unroll
            for (int k4 = 0; k4 < TK / 4; ++k4) mma_step_full(a + k4 * 4 * TPAD, b + k4 * 4 * TPAD, acc);
        } else {
#pragma unroll 1
            for (int k4 = 0; k4 < n4; ++k4) mma_step_full(a + k4 * 4 * TPAD, b + k4 * 4 * TPAD, acc);
        }
    } else if (onmask != 0u) {
#pragma unroll 1
        for (int k4 = 0; k4 < n4; ++k4) {
            double af[4], bf[2];
#pragma unroll
            for (int mt = 0; mt < 4; ++mt) af[mt] = a[k4 * 4 * TPAD + mt * 8];
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) bf[nt] = b[k4 * 4 * TPAD + nt * 8];
#pragma unroll
            for (int mt = 0; mt < 4; ++mt)
#pragma unroll
                for (int nt = 0; nt < 2; ++nt)
                    if (onmask & (1u << (mt * 2 + nt))) dmma(acc[mt * 2 + nt], af[mt], bf[nt]);
        }
    }
}

// ---- balanced warp layouts for the tiles a 2x4 grid of 32x16 warp tiles serves badly (k_downdate_ws2) -------
// A full diagonal tile needs 36 of its 64 8x8 blocks; in the 2x4 grid two warps have all 8 of theirs and two have none, so
// the tile takes as long as a full one.  An off-diagonal tile of the last tile row has n - i0 < 64 rows: the upper-row warps
// have 8 blocks, the lower-row warps 2.  At n = 613 these are 18 of the 55 tiles of a filter.
//   TRI:   8x8 block (r, c), c <= r, of the diagonal tile -> fixed per-warp lists of <= 5 blocks in at most two block rows
//          (one A fragment per block row); A and B fragments both come from the tile's single W panel.
//   STRIP: warp w owns block column w and all NRB existing block rows (one B fragment, NRB A fragments).
template <int RA, int CA, int NA, int RB, int CB, int NBK>
struct TriW {
    static __device__ __forceinline__ void step(const double* __restrict__ p, double (&acc)[8][2]) {
        const double af0 = p[RA * 8];
        double af1 = 0.0;
        if (NBK > 0) af1 = p[RB * 8];
        double bf[NA + NBK];
#pragma unroll
        for (int i = 0; i < NA; ++i) bf[i] = p[(CA + i) * 8];
#pragma unroll
        for (int i = 0; i < NBK; ++i) bf[NA + i] = p[(CB + i) * 8];
#pragma unroll
        for (int i = 0; i < NA; ++i) dmma(acc[i], af0, bf[i]);
#pragma unroll
        for (int i = 0; i < NBK; ++i) dmma(acc[NA + i], af1, bf[NA + i]);
    }
    static __device__ __forceinline__ void chunk(const double* __restrict__ p, int n4, double (&acc)[8][2]) {
        if (n4 == TK / 4) {
#pragma unroll
            for (int k4 = 0; k4 < TK / 4; ++k4) step(p + k4 * 4 * TPAD, acc);
        } else {
#pragma unroll 1
            for (int k4 = 0; k4 < n4; ++k4) step(p + k4 * 4 * TPAD, acc);
        }
    }
    // X <- X - acc for this warp's blocks (x = X + g * XP + 2 q)
    static __device__ __forceinline__ void update(double* __restrict__ x, const double (&acc)[8][2]) {
#pragma unroll
        for (int i = 0; i < NA + NBK; ++i) {
            const int r = (i < NA) ? RA : RB, c = (i < NA) ? CA + i : CB + i - NA;
            double2* xp = reinterpret_cast<double2*>(x + r * 8 * XP_ + c * 8);
            double2 pv = *xp;
            pv.x -= acc[i][0];
            pv.y -= acc[i][1];
            *xp = pv;
        }
    }
};
// warp -> block list of the lower triangle of an 8x8 block grid: row 7: w0 (cols 0-4), w1 (5-7); row 6: w2 (0-4), w3 (5-6);
// row 5: w4 (0-4), w5 (5); row 4: w6 (0-4); row 3: w5 (0-3); row 2: w3 (0-2); row 1: w1 (0-1); row 0: w7.  36 blocks, <= 5 each.
typedef TriW<7, 0, 5, 0, 0, 0> TriW0;
typedef TriW<7, 5, 3, 1, 0, 2> TriW1;
typedef TriW<6, 0, 5, 0, 0, 0> TriW2;
typedef TriW<6, 5, 2, 2, 0, 3> TriW3;
typedef TriW<5, 0, 5, 0, 0, 0> TriW4;
typedef TriW<5, 5, 1, 3, 0, 4> TriW5;
typedef TriW<4, 0, 5, 0, 0, 0> TriW6;
typedef TriW<0, 0, 1, 0, 0, 0> TriW7;
#define TRI_DISPATCH(warp, CALL)           \
    switch (warp) {                        \
        case 0: CALL(TriW0); break;        \
        case 1: CALL(TriW1); break;        \
        case 2: CALL(TriW2); break;        \
        case 3: CALL(TriW3); break;        \
        case 4: CALL(TriW4); break;        \
        case 5: CALL(TriW5); break;        \
        case 6: CALL(TriW6); break;        \
        default: CALL(TriW7); break;       \
    }

template <int NRB>
struct StripW {
    static __device__ __forceinline__ void step(const double* __restrict__ a, const double* __restrict__ b, double (&acc)[8][2]) {
        const double bf = b[0];
        double af[NRB];
#pragma unroll
        for (int rb = 0; rb < NRB; ++rb) af[rb] = a[rb * 8];
#pragma unroll
        for (int rb = 0; rb < NRB; ++rb) dmma(acc[rb], af[rb], bf);
    }
    static __device__ __forceinline__ void chunk(const double* __restrict__ a, const double* __restrict__ b, int n4, double (&acc)[8][2]) {
        if (n4 == TK / 4) {
#pragma unroll
            for (int k4 = 0; k4 < TK / 4; ++k4) step(a + k4 * 4 * TPAD, b + k4 * 4 * TPAD, acc);
        } else {
#pragma unroll 1
            for (int k4 = 0; k4 < n4; ++k4) step(a + k4 * 4 * TPAD, b + k4 * 4 * TPAD, acc);
        }
    }
    // x = X + g * XP + warp * 8 + 2 q
    static __device__ __forceinline__ void update(double* __restrict__ x, const double (&acc)[8][2]) {
#pragma unroll
        for (int rb = 0; rb < NRB; ++rb) {
            double2* xp = reinterpret_cast<double2*>(x + rb * 8 * XP_);
            double2 pv = *xp;
            pv.x -= acc[rb][0];
            pv.y -= acc[rb][1];
            *xp = pv;
        }
    }
};
#define STRIP_DISPATCH(nrb, CALL)                 \
    switch (nrb) {                                \
        case 1: CALL(StripW<1>); break;           \
        case 2: CALL(StripW<2>); break;           \
        case 3: CALL(StripW<3>); break;           \
        case 4: CALL(StripW<4>); break;           \
        case 5: CALL(StripW<5>); break;           \
        case 6: CALL(StripW<6>); break;           \
        case 7: CALL(StripW<7>); break;           \
        default: CALL(StripW<8>); break;          \
    }

// ---- one CTA per tile, cp.async ring ------------------------------------------------------------------
__global__ void __launch_bounds__(256, 3) k_downdate_tile(DevView v) {
    extern __shared__ __align__(16) double dsm[];
    const int b = blockIdx.y;
    const int k = v.ktot[b];
    if (k == 0) return;
    const int n = v.nstate[b];
    const int e = blockIdx.x;
    int ti = (int)((sqrtf(8.0f * e + 1.0f) - 1.0f) * 0.5f);
    while ((ti + 1) * (ti + 2) / 2 <= e) ++ti;
    while (ti * (ti + 1) / 2 > e) --ti;
    const int tj = e - ti * (ti + 1) / 2;
    const int i0 = ti * TM, j0 = tj * TM;
    if (i0 >= n) return;
    const int ld = v.ld, kmax = v.wrows;   // W panel stride (rows)
    const double* __restrict__ W = v.W + (size_t)b * v.wstride;
    double* __restrict__ P = v.P + (size_t)b * v.nmax * ld;
    const bool diag = (ti == tj);
    double* As = dsm;                            // [NSTAGE][TK][TPAD]
    double* Bs = dsm + NSTAGE * TK * TPAD;       // [NSTAGE][TK][TPAD]
    double* strip = Bs + NSTAGE * TK * TPAD;     // [64][9]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wr = warp >> 2, wc = warp & 3, g = lane >> 2, q = lane & 3;

    double pf[4][2][2];
    load_p_frags(P, ld, n, i0, j0, wr, wc, g, q, pf);
    const int nk = (k + TK - 1) / TK;
    const int lr = tid >> 5, lcc = (tid & 31) * 2;
    const bool cola = (i0 + lcc < ld), colb = (j0 + lcc < ld);
    const double* __restrict__ wa = W + w_at(kmax, lr, i0 + lcc);   // panel-major W: row stride EKF_WPAD inside a panel
    const double* __restrict__ wb = W + w_at(kmax, lr, j0 + lcc);
    const int soff = lr * TPAD + lcc;
    auto load_stage = [&](int st, int t0) {
        double* as = As + st * TK * TPAD + soff;
        double* bs = Bs + st * TK * TPAD + soff;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int tt = t0 + lr + 8 * j;
            const bool oka = (tt < k) && cola;
            cp_async16(as + 8 * j * TPAD, oka ? wa + (size_t)(t0 + 8 * j) * EKF_WPAD : W, oka ? 16 : 0);
            if (!diag) {
                const bool okb = (tt < k) && colb;
                cp_async16(bs + 8 * j * TPAD, okb ? wb + (size_t)(t0 + 8 * j) * EKF_WPAD : W, okb ? 16 : 0);
            }
        }
    };
    double acc[8][2];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i][0] = acc[i][1] = 0.0;
    const unsigned onmask = tile_mask(i0, j0, wr, wc, n, diag);
    const int aoff = q * TPAD + wr * 32 + g, boff = q * TPAD + wc * 16 + g;

#pragma unroll
    for (int st = 0; st < NSTAGE - 1; ++st) {
        if (st < nk) load_stage(st, st * TK);
        cp_async_commit();
    }
    for (int it = 0; it < nk; ++it) {
        cp_async_wait<NSTAGE - 2>();
        __syncthreads();
        if (it + NSTAGE - 1 < nk) load_stage((it + NSTAGE - 1) % NSTAGE, (it + NSTAGE - 1) * TK);
        cp_async_commit();
        const double* as = As + (it % NSTAGE) * TK * TPAD;
        const double* bs = diag ? as : Bs + (it % NSTAGE) * TK * TPAD;
        mma_chunk(as + aoff, bs + boff, min(TK / 4, (k - it * TK + 3) >> 2), onmask, acc);  // the tail panel stops at k (rounded to 4)
    }
    cp_async_wait<0>();
    if (tj == 0)
        apply_j_col0(strip, v.jn + (size_t)b * 16, diag, wr, wc, g, q, tid, pf, [] { __syncthreads(); });
    store_tile(P, ld, n, i0, j0, wr, wc, g, q, diag, onmask, pf, acc);
}

// ---- persistent, warp-specialised, with epilogue warps (default) ----------------------------------------
// Roles per CTA (13 warps, 2 CTAs per SM); X = one shared [64][XP] tile buffer:
//   warp  8     producer: streams the W panels with bulk copies through the mbarrier ring (one per panel and stage).
//   warps 0-7   consumers: K loop; then J on tile column 0 of X (the prefetched P tile), X <- X - acc, and straight on
//               to the next tile.
//   warps 9-12  epilogue: row-coalesced stores of the tile and of its mirror image (read
//               transposed from X), then the bulk-copy prefetch of the NEXT tile's P into X, which completes
//               (mbarrier pfull) while the consumers run that tile's K loop.
// The round-1 kernel kept the P loads and the stores in the consumer warps, so each CTA alternated between a DMMA
// phase and a load/store phase and the two CTAs of an SM drifted into the same phase (ablation in DESIGN.md §3.1:
// consumers without copies 3.42 ms = DMMA 2.03 + stores 1.39); here both phases run concurrently inside every CTA
// and no P value is held in registers across the K loop.
#define WS2_EPI 4
#define WS2_THREADS ((WS_CONSUMERS + 1 + WS2_EPI) * 32)
#define XP XP_  // row pitch of X in doubles (66): rows stay 16-byte aligned for bulk copies and double2 access

__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 2, 128;" ::: "memory"); }
__device__ __forceinline__ void cons_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// bulk-copy prefetch of the P tile of `t` into X: 16 rows per epilogue warp, one row per lane (a bulk copy is a
// uniform-datapath instruction, so the copies of one warp issue one after the other; four warps issue in parallel)
__device__ __forceinline__ void epi_prefetch_p(double* X, const double* __restrict__ P, int ld, const DTile& t, int ew, int lane,
                                               unsigned long long* pfull) {
    const int nrows = min(TM, t.n - t.i0);
    const unsigned rowbytes = (unsigned)(min(TM, ld - t.j0) * 8);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // X was last read through the generic proxy
    if (ew == 0 && lane == 0) mbar_arrive_expect_tx(pfull, (unsigned)nrows * rowbytes);
    const int r = ew * 16 + lane;
    if (lane < 16 && r < nrows) bulk_g2s(X + r * XP, P + (size_t)(t.i0 + r) * ld + t.j0, rowbytes, pfull);
}

// S = stages of the W ring, NX = P tile buffers.  <4,1>: deep ring for long K loops (li update); <2,2>: short K loops
// (small k, the kernel streams P): the next-but-one P tile is prefetched while the current one is being stored.
template <int S, int NX>
__global__ void __launch_bounds__(WS2_THREADS, 2) k_downdate_ws2(DevView v, int T, int b0, long long total, int M) {
    extern __shared__ __align__(16) double dsm[];
    double* As = dsm;                                   // [S][TK][TPAD]
    double* Bs = dsm + S * TK * TPAD;           // [S][TK][TPAD]
    double* X0 = Bs + S * TK * TPAD;            // [NX][64][XP]
    unsigned long long* full = reinterpret_cast<unsigned long long*>(X0 + NX * TM * XP);   // [S]
    unsigned long long* empty = full + S;                                     // [S]
    unsigned long long* pfull = empty + S;   // [NX] P tile landed in X[j]
    unsigned long long* cfull = pfull + NX;  // [NX] X[j] holds P - acc
    int2* meta = reinterpret_cast<int2*>(cfull + NX);                                  // [M]  {ktot, n}
    unsigned* lut = reinterpret_cast<unsigned*>(meta + M);                            // [T]  ti<<16|tj
    const int ld = v.ld, kmax = v.wrows;   // W panel stride (rows)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long G = gridDim.x;
    for (int m = tid; m < M; m += blockDim.x) {
        const long long t = blockIdx.x + (long long)m * G;
        int2 kn = make_int2(0, 0);
        if (t < total) { const int b = b0 + (int)(t / T); kn = make_int2(v.ktot[b], v.nstate[b]); }
        meta[m] = kn;
    }
    for (int e = tid; e < T; e += blockDim.x) {
        int ti = (int)((sqrtf(8.0f * e + 1.0f) - 1.0f) * 0.5f);
        while ((ti + 1) * (ti + 2) / 2 <= e) ++ti;
        while (ti * (ti + 1) / 2 > e) --ti;
        lut[e] = ((unsigned)ti << 16) | (unsigned)(e - ti * (ti + 1) / 2);
    }
    if (tid == 0) {
        for (int s2 = 0; s2 < S; ++s2) { mbar_init(full + s2, 32); mbar_init(empty + s2, WS_CONSUMERS); }
        for (int j = 0; j < NX; ++j) mbar_init(pfull + j, 1);
        for (int j = 0; j < NX; ++j) mbar_init(cfull + j, WS_CONSUMERS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int own = (int)((total - blockIdx.x + G - 1) / G);
    const int Mreal = own < M ? own : M;

    if (warp == WS_CONSUMERS) {
        // ================= producer warp =================
        // W is panel-major (common.cuh, w_at): the K chunk of a 64-column panel is one contiguous range that already
        // has the padded [TK][TPAD] shared-memory layout -> one bulk copy per panel and stage, issued by lane 0.
        unsigned cnt = 0;
        for (int m = 0; m < Mreal; ++m) {
            const DTile L = decode_tile(meta, lut, m, Mreal, blockIdx.x + (long long)m * G, T);
            if (L.nk == 0) continue;
            const double* __restrict__ W = v.W + (size_t)(b0 + L.b) * v.wstride;
            const double* __restrict__ wa = W + w_at(kmax, 0, L.i0);
            const double* __restrict__ wb = W + w_at(kmax, 0, L.j0);
            for (int st = 0; st < L.nk; ++st, ++cnt) {
                const unsigned slot = cnt % S, ph = (cnt / S) & 1u;
                mbar_wait(empty + slot, ph ^ 1u);
                const int t0 = st * TK;
                const int nvalid = min(TK, L.k - t0);
                double* da = As + slot * TK * TPAD;
                double* db = Bs + slot * TK * TPAD;
                if (lane == 0) {
                    const unsigned bytes = (unsigned)(nvalid * TPAD * 8);
                    mbar_arrive_expect_tx(full + slot, L.diag ? bytes : 2u * bytes);
                    bulk_g2s(da, wa + (size_t)t0 * TPAD, bytes, full + slot);
                    if (!L.diag) bulk_g2s(db, wb + (size_t)t0 * TPAD, bytes, full + slot);
                } else {
                    if (nvalid & 3) {   // rows between k and the next multiple of 4 are zero
                        const int nz = (((nvalid + 3) & ~3) - nvalid) * TPAD;
                        for (int e = lane - 1; e < nz; e += 31) {
                            da[nvalid * TPAD + e] = 0.0;
                            if (!L.diag) db[nvalid * TPAD + e] = 0.0;
                        }
                    }
                    mbar_arrive(full + slot);
                }
            }
        }
        return;
    }

    if (warp < WS_CONSUMERS) {
        // ================= consumer warps: 2 (rows) x 4 (cols), 32 x 16 each =================
        const int wr = warp >> 2, wc = warp & 3, g = lane >> 2, q = lane & 3;
        const int aoff = q * TPAD + wr * 32 + g, boff = q * TPAD + wc * 16 + g;
        const int xoff = (wr * 32 + g) * XP + wc * 16 + 2 * q;
        unsigned cnt = 0, tiles = 0;
        for (int cm = 0; cm < Mreal; ++cm) {
            const DTile C = decode_tile(meta, lut, cm, Mreal, blockIdx.x + (long long)cm * G, T);
            if (C.nk == 0) continue;
            // warp layout of this tile: 0 = 2x4 grid of 32x16 (full tiles; masked path for the partial last diagonal tile),
            // 1 = STRIP (off-diagonal tile with fewer than 64 rows), 2 = TRI (full diagonal tile)
            const bool full_rows = C.i0 + TM <= C.n;
            const int layout = C.diag ? (full_rows ? 2 : 0) : (full_rows ? 0 : 1);
            const int nrb = (min(TM, C.n - C.i0) + 7) >> 3;
            const unsigned onmask = tile_mask(C.i0, C.j0, wr, wc, C.n, C.diag);
            double acc[8][2];
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i][0] = acc[i][1] = 0.0;
            for (int it = 0; it < C.nk; ++it, ++cnt) {
                const unsigned slot = cnt % S, ph = (cnt / S) & 1u;
                mbar_wait(full + slot, ph);
                const double* as = As + slot * TK * TPAD;
                const double* bs = C.diag ? as : Bs + slot * TK * TPAD;
                const int n4 = min(TK / 4, (C.k - it * TK + 3) >> 2);
                if (layout == 0) {
                    mma_chunk(as + aoff, bs + boff, n4, onmask, acc);
                } else if (layout == 1) {
#define CALL_(W) W::chunk(as + q * TPAD + g, bs + q * TPAD + warp * 8 + g, n4, acc)
                    STRIP_DISPATCH(nrb, CALL_)
#undef CALL_
                } else {
#define CALL_(W) W::chunk(as + q * TPAD + g, n4, acc)
                    TRI_DISPATCH(warp, CALL_)
#undef CALL_
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(empty + slot);
            }
            double* X = X0 + (tiles % NX) * TM * XP;
            mbar_wait(pfull + tiles % NX, (tiles / NX) & 1u);   // this tile's P has landed (and an earlier tile has left X)
            if (C.col0) {
                // J P J' on the P tile itself (W already carries J, see k_wfix): columns 3..6 of tile column 0, rows 3..6
                // of tile (0,0)
                const double* __restrict__ Jn = v.jn + (size_t)(b0 + C.b) * 16;
                if (tid < TM) {
                    double* xr = X + tid * XP;
                    const double c3 = xr[3], c4 = xr[4], c5 = xr[5], c6 = xr[6];
#pragma unroll
                    for (int a = 0; a < 4; ++a) xr[3 + a] = c3 * Jn[a * 4 + 0] + c4 * Jn[a * 4 + 1] + c5 * Jn[a * 4 + 2] + c6 * Jn[a * 4 + 3];
                }
                cons_bar();
                if (C.diag) {
                    if (tid < 8) {
                        const double r3 = X[3 * XP + tid], r4 = X[4 * XP + tid], r5 = X[5 * XP + tid], r6 = X[6 * XP + tid];
#pragma unroll
                        for (int a = 0; a < 4; ++a)
                            X[(3 + a) * XP + tid] = Jn[a * 4 + 0] * r3 + Jn[a * 4 + 1] * r4 + Jn[a * 4 + 2] * r5 + Jn[a * 4 + 3] * r6;
                    }
                    cons_bar();
                }
            }
            if (layout == 0) {
#pragma unroll
                for (int mt = 0; mt < 4; ++mt)
#pragma unroll
                    for (int nt = 0; nt < 2; ++nt) {
                        double2* xp = reinterpret_cast<double2*>(X + xoff + (mt * 8) * XP + nt * 8);
                        double2 pv = *xp;
                        pv.x -= acc[mt * 2 + nt][0];
                        pv.y -= acc[mt * 2 + nt][1];
                        *xp = pv;
                    }
            } else if (layout == 1) {
#define CALL_(W) W::update(X + g * XP + warp * 8 + 2 * q, acc)
                STRIP_DISPATCH(nrb, CALL_)
#undef CALL_
            } else {
#define CALL_(W) W::update(X + g * XP + 2 * q, acc)
                TRI_DISPATCH(warp, CALL_)
#undef CALL_
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(cfull + tiles % NX);
            ++tiles;
        }
        return;
    }

    // ================= epilogue warps =================
    const int et = tid - (WS_CONSUMERS + 1) * 32, ew = et >> 5;
    unsigned tiles = 0;
    // two cursors over this CTA's tile list: pm = next tile whose P has to be prefetched, cm = tile being stored
    int pm = -1;
    DTile Pn;
    auto next_valid = [&](int m, DTile& t) {
        do { ++m; t = decode_tile(meta, lut, m, Mreal, blockIdx.x + (long long)m * G, T); } while (m < Mreal && t.nk == 0);
        return m;
    };
#pragma unroll
    for (int j = 0; j < NX; ++j) {
        pm = next_valid(pm, Pn);
        if (pm < Mreal) epi_prefetch_p(X0 + j * TM * XP, v.P + (size_t)(b0 + Pn.b) * v.nmax * ld, ld, Pn, ew, lane, pfull + j);
    }
    DTile C;
    int cm = next_valid(-1, C);
    while (cm < Mreal) {
        double* __restrict__ P = v.P + (size_t)(b0 + C.b) * v.nmax * ld;
        double* X = X0 + (tiles % NX) * TM * XP;
        const int n = C.n, i0 = C.i0, j0 = C.j0;
        mbar_wait(cfull + tiles % NX, (tiles / NX) & 1u);
        // stores: one 512-byte row segment (tile) / two 256-byte segments (mirror image) per warp instruction
        const int c = 2 * lane;
        if (!C.diag) {
#pragma unroll 4
            for (int p = 0; p < 16; ++p) {
                const int r = ew + 4 * p;
                if (i0 + r < n) {
                    const double2 val = *reinterpret_cast<const double2*>(X + r * XP + c);
                    double* o = P + (size_t)(i0 + r) * ld + j0 + c;
                    if (j0 + c + 1 < n) *reinterpret_cast<double2*>(o) = val;
                    else if (j0 + c < n) o[0] = val.x;
                }
                if (j0 + r < n) {   // mirror image: row j0 + r of P, columns i0 ..
                    double* mrow = P + (size_t)(j0 + r) * ld + i0;
                    if (i0 + lane < n) mrow[lane] = X[lane * XP + r];
                    if (i0 + lane + 32 < n) mrow[lane + 32] = X[(lane + 32) * XP + r];
                }
            }
        } else {
#pragma unroll 4
            for (int p = 0; p < 16; ++p) {
                const int r = ew + 4 * p;
                if (i0 + r < n) {
                    const double a = (c <= r) ? X[r * XP + c] : X[c * XP + r];
                    const double bq = (c + 1 <= r) ? X[r * XP + c + 1] : X[(c + 1) * XP + r];
                    double* o = P + (size_t)(i0 + r) * ld + i0 + c;
                    if (i0 + c + 1 < n) *reinterpret_cast<double2*>(o) = make_double2(a, bq);
                    else if (i0 + c < n) o[0] = a;
                }
            }
        }
        epi_bar();   // every epilogue thread is done reading X
        if (pm < Mreal) {
            pm = next_valid(pm, Pn);
            if (pm < Mreal) epi_prefetch_p(X, v.P + (size_t)(b0 + Pn.b) * v.nmax * ld, ld, Pn, ew, lane, pfull + tiles % NX);
        }
        ++tiles;
        cm = next_valid(cm, C);
    }
}

void launch_downdate(ekfslam_ctx* c, int slot) {
    DevView& v = c->v;
    const int sms = c->sm_count;   // of the context's own device (a process may drive several GPUs)
    const int nt = (v.nmax + TM - 1) / TM;
    const int T = nt * (nt + 1) / 2;
    KScope ks(c, slot);
    // ring depth / P buffers by update kind: the hi update and the camera-state update stack few rows (short K loops,
    // the kernel streams P), the li update many.
    const bool cfgB = slot != KT_DOWNDATE;
    const int S = cfgB ? 2 : 4, NX = cfgB ? 2 : 1;
    // filters are processed in groups small enough for the per-CTA tile metadata (8 B per tile) to stay
    // within the shared-memory budget of two CTAs per SM
    const long long ctas_full = (long long)sms * 2;
    const size_t fixed = sizeof(double) * (2 * S * TK * TPAD + NX * TM * XP) + sizeof(unsigned long long) * (2 * S + 2 * NX) +
                         sizeof(unsigned) * T;
    const size_t budget = 111 * 1024;
    if (fixed + 64 * sizeof(int2) <= budget) {
        const long long Mcap = (long long)((budget - fixed) / sizeof(int2));
        long long bgroup = (Mcap * ctas_full) / T;
        if (bgroup < 1) bgroup = 1;
        const char* eg = getenv("EKFSLAM_DD_GROUP");   // =g: at most g filters per launch (exercises the grouping in tests)
        const long long force_group = eg ? atoll(eg) : 0;
        if (force_group > 0 && force_group < bgroup) bgroup = force_group;
        for (long long b0 = 0; b0 < v.B; b0 += bgroup) {
            const long long nb = (v.B - b0 < bgroup) ? (v.B - b0) : bgroup;
            const long long total = (long long)T * nb;
            const long long ctas = total < ctas_full ? total : ctas_full;
            const int M = (int)((total + ctas - 1) / ctas);
            const size_t sm2 = fixed + sizeof(int2) * M;
            if (cfgB) ENSURE_DYN_SMEM((k_downdate_ws2<2, 2>), sm2, c->device);
            else ENSURE_DYN_SMEM((k_downdate_ws2<4, 1>), sm2, c->device);
            if (cfgB) k_downdate_ws2<2, 2><<<(unsigned)ctas, WS2_THREADS, sm2, c->stream>>>(v, T, (int)b0, total, M);
            else k_downdate_ws2<4, 1><<<(unsigned)ctas, WS2_THREADS, sm2, c->stream>>>(v, T, (int)b0, total, M);
            if (b0 > 0) c->launches++;
        }
        return;
    }
    // the tile table does not fit (li <4,1>: T > 2412, i.e. n_max > 4352; hi <2,2>: T > 2672, n_max > 4608): one CTA per tile
    const size_t sm = sizeof(double) * (2 * NSTAGE * TK * TPAD + TM * 9);
    ENSURE_DYN_SMEM(k_downdate_tile, sm, c->device);
    dim3 gd(T, v.B);
    k_downdate_tile<<<gd, 256, sm, c->stream>>>(v);
}
