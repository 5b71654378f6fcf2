// Shared building blocks of the tensor-core kernels (k_w, k_downdate*): DMMA wrapper, cp.async ring
// helpers, mbarrier / bulk-copy wrappers, lower-triangle tile decoding; and the 16-wide warp Cholesky of the
// update's diagonal blocks.
#pragma once
#include "common.cuh"

// ---------------------------------------------------------------------------------------
// fp64 tensor-core building blocks.  mma.sync m8n8k4 f64 (SASS DMMA.8x8x4) fragment layout, lane
// l, g = l>>2, q = l&3:  A[g][q],  B[q][g],  C[g][2q], C[g][2q+1].
// Both GEMMs below use 64x64 block tiles, 8 warps in a 2x4 grid, 32x16 per warp (4x2 DMMA tiles),
// K panels of 16 staged through a 3-deep cp.async (LDGSTS) ring.
// ---------------------------------------------------------------------------------------
#define TM 64
#define TK 16
#define TPAD 68    // row stride (doubles) of a K-major panel [TK][64]: stride % 16 == 4 -> conflict-free frags
#define APAD 20    // row stride of a row-major A panel [64][TK]: same property
#define NSTAGE 3

__device__ __forceinline__ void dmma(double (&c)[2], double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}
__device__ __forceinline__ void cp_async16(double* smem_dst, const double* gmem_src, int src_bytes) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem_src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async8(double* smem_dst, const double* gmem_src) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---------------------------------------------------------------------------------------
// 16x16 Cholesky + inverse by ONE warp (the diagonal blocks of k_chol, k_chol_sm and k_cb_diagpanel), the block held in
// registers (lane i = row i, lanes 16..31 mirror 0..15 so that every shuffle is full-warp), column c broadcast by
// shuffles, one rsqrt per pivot in place of the sqrt and every division.  Blk: shared, the lower triangle in (the upper
// one is not read), L out with zeros above the diagonal; rows past the data must be padded with the identity.
// Di [16][17]: inv(L), all 16 x 16 entries written (zeros above the diagonal).  Returns true for a pivot that is not > 0.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ bool chol16_warp(double* __restrict__ Blk, int pitch, double* __restrict__ Di) {
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31, i = lane & 15;
    double a[16], rd[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) a[c] = (c <= i) ? Blk[i * pitch + c] : 0.0;
    bool bad = false;
#pragma unroll
    for (int c = 0; c < 16; ++c) {
        const double piv = __shfl_sync(full, a[c], c);
        bad = bad || !(piv > 0.0);
        const double rs = rsqrt(piv);
        rd[c] = rs;
        const double lic = (i == c) ? piv * rs : a[c] * rs;  // rows above the diagonal carry don't-care values
        a[c] = lic;
#pragma unroll
        for (int j = c + 1; j < 16; ++j) {
            const double ljc = __shfl_sync(full, lic, j);
            a[j] -= lic * ljc;
        }
    }
    if (lane < 16) {
#pragma unroll
        for (int c = 0; c < 16; ++c) Blk[i * pitch + c] = (c <= i) ? a[c] : 0.0;
    }
    __syncwarp();
    // column c = lane of inv(L) by forward substitution; every lane reads the same L entry at the same time (broadcast)
    const int c = i;
    double x[16];
#pragma unroll
    for (int ii = 0; ii < 16; ++ii) {
        double sacc = 0.0;
#pragma unroll
        for (int t = 0; t < ii; ++t) sacc += Blk[ii * pitch + t] * x[t];
        x[ii] = (ii == c) ? rd[ii] : ((ii > c) ? -sacc * rd[ii] : 0.0);
    }
    if (lane < 16) {
#pragma unroll
        for (int ii = 0; ii < 16; ++ii) Di[ii * 17 + c] = x[ii];
    }
    return bad;
}


struct DTile {
    int b, i0, j0, k, n, nk;
    bool diag, col0;
};

// tile m of this CTA (global tile t = blockIdx.x + m*G): metadata comes from shared memory
// (meta[m] = {k, n} of the tile's filter, lut[e] = ti<<16|tj), never from a dependent global load
__device__ __forceinline__ DTile decode_tile(const int2* meta, const unsigned* lut, int m, int M, long long t, int T,
                                             int tile = TM) {
    DTile d;
    d.nk = 0; d.b = 0; d.i0 = 0; d.j0 = 0; d.k = 0; d.n = 0; d.diag = false; d.col0 = false;
    if (m >= M) return d;
    d.b = (int)(t / T);
    const unsigned e = lut[(int)(t - (long long)d.b * T)];
    const int ti = (int)(e >> 16), tj = (int)(e & 0xffffu);
    d.i0 = ti * tile; d.j0 = tj * tile;
    d.diag = (ti == tj); d.col0 = (tj == 0);
    const int2 kn = meta[m];
    d.k = kn.x; d.n = kn.y;
    d.nk = (d.i0 < d.n) ? (d.k + TK - 1) / TK : 0;
    return d;
}


__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(double* smem_dst, const double* gmem_src, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

