// Closed-loop support on the device (SURVEY §8f ranks 2-3):
//   * the synthetic world: candidate pixels for the features currently in each map and corner detections for
//     new features, from resident world points + camera trajectory + counter-based noise - the stand-in for
//     the reference's image front-end (mc/matching.m FAST/FREAK search, mc/initialize_a_feature.m:22-57), so a
//     whole sequence runs with zero per-frame host-to-device traffic;
//   * the decision part of mc/map_management.m:7-35 (deletion list, measured count, number of features to
//     initialise); the state / covariance surgery itself is k_delete_features, k_id2cart, k_add_feature
//     (k_model.cu).
// numpy mirror of the world: ekf-slam_b200/synth.py (SynthWorld).
#include "model.cuh"

// ---------------------------------------------------------------------------------------
// counter-based uniforms: key (seed, filter, frame, world point, channel) -> [0,1)   (synth.world_uniform)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
    x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull;
    x ^= x >> 27; x *= 0x94D049BB133111EBull;
    x ^= x >> 31;
    return x;
}
__device__ __forceinline__ double world_u01(unsigned long long seed, int b, int t, int w, int c) {
    unsigned long long k = mix64(seed + 0x9E3779B97F4A7C15ull * ((unsigned long long)b + 1ull));
    k = mix64(k + (unsigned long long)t);
    k = mix64(k + (unsigned long long)w);
    k = mix64(k + (unsigned long long)c);
    return (double)(k >> 11) * (1.0 / 9007199254740992.0);
}

// distorted pixel of world point p seen from pose (r, q); returns depth along the optical axis
__device__ __forceinline__ double world_project(const DevCam& cam, const double* __restrict__ p, const double* __restrict__ pose,
                                                double& ud, double& vd) {
    double R[9];
    q2r_dev(pose + 3, R);
    const double d0 = p[0] - pose[0], d1 = p[1] - pose[1], d2 = p[2] - pose[2];
    const double hx = R[0] * d0 + R[3] * d1 + R[6] * d2;   // R' d
    const double hy = R[1] * d0 + R[4] * d1 + R[7] * d2;
    const double hz = R[2] * d0 + R[5] * d1 + R[8] * d2;
    const double fku = cam.f / cam.dx, fkv = cam.f / cam.dy;
    distort_dev(cam, cam.Cx + hx / hz * fku, cam.Cy + hy / hz * fkv, ud, vd);
    return hz;
}

// Box-Muller pair from noise channels c1 and c1 + 1
__device__ __forceinline__ void world_gauss(const DevWorld& w, int b, int t, int id, double& n0, double& n1, int c1 = 1) {
    const double u1 = world_u01(w.seed, b + w.b_offset, t, id, c1);
    const double u2 = world_u01(w.seed, b + w.b_offset, t, id, c1 + 1);
    const double rad = sqrt(-2.0 * log(1.0 - u1));
    double s, c;
    sincos(2.0 * 3.14159265358979323846 * u2, &s, &c);
    n0 = rad * c;
    n1 = rad * s;
}

// ---------------------------------------------------------------------------------------
// candidates of frame t for every feature of every map: one thread per (filter, feature slot)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_synth_candidates(DevView v, DevCam cam, DevWorld w, int t) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= v.B * v.N) return;
    const int b = e / v.N, i = e - b * v.N;
    double zx = 0.0, zy = 0.0;
    uint8_t fl = 0;
    if (i < v.nfeat[b]) {
        const int id = v.tag[e];
        if (id >= 0 && id < w.M) {
            double ud, vd;
            const double dep = world_project(cam, w.points + ((size_t)b * w.M + id) * 3, w.poses + ((size_t)t * v.B + b) * 7, ud, vd);
            const bool vis = dep > 0.0 && ud > 0.0 && ud < cam.nCols && vd > 0.0 && vd < cam.nRows;
            if (vis) {
                const double u0 = world_u01(w.seed, b + w.b_offset, t, id, 0);
                const double p_out = (id % w.flaky_mod == w.flaky_mod - 1) ? w.p_flaky : w.p_outlier;
                if (u0 < p_out) {
                    zx = ud + (2.0 * world_u01(w.seed, b + w.b_offset, t, id, 3) - 1.0) * w.gross_px;
                    zy = vd + (2.0 * world_u01(w.seed, b + w.b_offset, t, id, 4) - 1.0) * w.gross_px;
                } else {
                    double n0, n1;
                    world_gauss(w, b, t, id, n0, n1);
                    zx = ud + n0 * w.noise_px;
                    zy = vd + n1 * w.noise_px;
                }
                fl = EKFSLAM_F_CAND;
            }
        }
    }
    v.zc[2 * (size_t)e] = zx;
    v.zc[2 * (size_t)e + 1] = zy;
    v.mflags[e] = fl;
}

// ---------------------------------------------------------------------------------------
// corner detections in the image of frame t: per filter the first K world points (by id) that are visible
// inside the excluded band (mc/initialize_a_feature.m:8,24-27) and not yet in the map, at integer pixels.
// One block per filter; M <= WORLD_MAX_M.
// ---------------------------------------------------------------------------------------
#define WORLD_MAX_M 2048
__global__ void __launch_bounds__(128) k_synth_detect(DevView v, DevCam cam, DevWorld w, int t, int K,
                                                      double* __restrict__ det_uv, int32_t* __restrict__ det_tag,
                                                      int32_t* __restrict__ det_n) {
    __shared__ uint8_t ok[WORLD_MAX_M];
    __shared__ float px[WORLD_MAX_M][2];   // integer pixel values: exact in fp32
    const int b = blockIdx.x;
    for (int id = threadIdx.x; id < w.M; id += blockDim.x) ok[id] = 1;
    __syncthreads();
    const int nf = v.nfeat[b];
    for (int i = threadIdx.x; i < nf; i += blockDim.x) {
        const int id = v.tag[(size_t)b * v.N + i];
        if (id >= 0 && id < w.M) ok[id] = 0;
    }
    __syncthreads();
    for (int id = threadIdx.x; id < w.M; id += blockDim.x) {
        if (!ok[id]) continue;
        double ud, vd;
        const double dep = world_project(cam, w.points + ((size_t)b * w.M + id) * 3, w.poses + ((size_t)t * v.B + b) * 7, ud, vd);
        bool good = dep > 0.0 && ud > 0.0 && ud < cam.nCols && vd > 0.0 && vd < cam.nRows;
        if (good) {
            double n0, n1;
            world_gauss(w, b, t, id, n0, n1);
            const double pu = floor(ud + n0 * w.noise_px + 0.5), pv = floor(vd + n1 * w.noise_px + 0.5);
            good = !(pu < w.band || pu > cam.nCols - w.band || pv < w.band || pv > cam.nRows - w.band);
            px[id][0] = (float)pu;
            px[id][1] = (float)pv;
        }
        ok[id] = good ? 1 : 0;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int n = 0;
        for (int id = 0; id < w.M && n < K; ++id) {
            if (!ok[id]) continue;
            det_uv[((size_t)b * K + n) * 2] = (double)px[id][0];
            det_uv[((size_t)b * K + n) * 2 + 1] = (double)px[id][1];
            det_tag[(size_t)b * K + n] = id;
            ++n;
        }
        det_n[b] = n;
        for (int j = n; j < K; ++j) {
            det_uv[((size_t)b * K + j) * 2] = 0.0;
            det_uv[((size_t)b * K + j) * 2 + 1] = 0.0;
            det_tag[(size_t)b * K + j] = -1;
        }
    }
}

// ---------------------------------------------------------------------------------------
// mc/map_management.m:7-14,27-35, the decisions: deletion list (`delete_features` is missing upstream: the rule
// of the published toolbox - predicted more than 5 times, matched in fewer than half of them), `measured` over
// the surviving features, and how many detections to initialise (attempt cap 50, mc/initialize_features.m:5).
// One warp per filter.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_mm_plan(DevView v, int min_features, const int32_t* __restrict__ det_n, int K,
                                                 uint8_t* __restrict__ del, int32_t* __restrict__ quota) {
    const int b = blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (b >= v.B) return;
    const int nf = v.nfeat[b];
    int measured = 0;
    for (int i = lane; i < v.N; i += 32) {
        const size_t e = (size_t)b * v.N + i;
        uint8_t d = 0;
        if (i < nf) {
            const int tp = v.counters[2 * e], tm = v.counters[2 * e + 1];
            d = (2 * tm < tp && tp > 5) ? 1 : 0;     // times_measured < 0.5*times_predicted && times_predicted > 5
            if (!d && (v.flags[e] & (EKFSLAM_F_LI | EKFSLAM_F_HI))) ++measured;
        }
        del[e] = d;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) measured += __shfl_xor_sync(0xffffffffu, measured, o);
    if (lane == 0) {
        int need = 0;
        if (measured == 0) need = min_features;
        else if (measured < min_features) need = min_features - measured;
        quota[b] = min(min(need, det_n[b]), min(K, 50));
    }
}

// RANSAC uniform stream of frame t (the rand(1) of mc/select_random_match.m:12): u[b][i] = U(seed, b, t, i, channel 7)
__global__ void k_synth_uniforms(DevView v, DevWorld w, int t) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= v.B * v.n_u) return;
    const int b = e / v.n_u, i = e - b * v.n_u;
    v.u[e] = world_u01(w.seed, b + w.b_offset, t, i, 7);
}

// ---------------------------------------------------------------------------------------
// landmark observations of frame t (ekfslam_world_landmark_obs): one thread per (filter, landmark slot).  Landmark j
// with j < nlm[b] and a tag in [0, M) is that world point, seen as the candidates see it (visibility, outlier model,
// pixel noise) but on noise channels 8..12, so its noise is independent of the candidate of the same point.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_synth_landmark_obs(int B, DevCam cam, DevWorld w, DevLm lm, int t) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B * EKFSLAM_LM_MAX) return;
    const int b = e / EKFSLAM_LM_MAX, j = e - b * EKFSLAM_LM_MAX;
    double zx = 0.0, zy = 0.0;
    uint8_t has = 0;
    const int id = lm.tag[e];
    if (j < lm.nlm[b] && id >= 0 && id < w.M) {
        double ud, vd;
        const double dep = world_project(cam, w.points + ((size_t)b * w.M + id) * 3, w.poses + ((size_t)t * B + b) * 7, ud, vd);
        if (dep > 0.0 && ud > 0.0 && ud < cam.nCols && vd > 0.0 && vd < cam.nRows) {
            const double u0 = world_u01(w.seed, b + w.b_offset, t, id, 8);
            const double p_out = (id % w.flaky_mod == w.flaky_mod - 1) ? w.p_flaky : w.p_outlier;
            if (u0 < p_out) {
                zx = ud + (2.0 * world_u01(w.seed, b + w.b_offset, t, id, 11) - 1.0) * w.gross_px;
                zy = vd + (2.0 * world_u01(w.seed, b + w.b_offset, t, id, 12) - 1.0) * w.gross_px;
            } else {
                double n0, n1;
                world_gauss(w, b, t, id, n0, n1, 9);
                zx = ud + n0 * w.noise_px;
                zy = vd + n1 * w.noise_px;
            }
            has = 1;
        }
    }
    lm.uv[2 * (size_t)e] = zx;
    lm.uv[2 * (size_t)e + 1] = zy;
    lm.has[e] = has;
}

void launch_world_landmark_obs(ekfslam_ctx* c, int t) {
    const int tot = c->v.B * EKFSLAM_LM_MAX;
    KScope ks(c, KT_WORLD);
    k_synth_landmark_obs<<<(tot + 127) / 128, 128, 0, c->stream>>>(c->v.B, c->cam, c->world, c->lm, t);
}

void launch_world_uniforms(ekfslam_ctx* c, int t) {
    const int tot = c->v.B * c->v.n_u;
    KScope ks(c, KT_WORLD);
    k_synth_uniforms<<<(tot + 255) / 256, 256, 0, c->stream>>>(c->v, c->world, t);
}

void launch_world_candidates(ekfslam_ctx* c, int t) {
    const int tot = c->v.B * c->v.N;
    KScope ks(c, KT_WORLD);
    k_synth_candidates<<<(tot + 127) / 128, 128, 0, c->stream>>>(c->v, c->cam, c->world, t);
}

void launch_world_detect(ekfslam_ctx* c, int t) {
    KScope ks(c, KT_WORLD);
    k_synth_detect<<<c->v.B, 128, 0, c->stream>>>(c->v, c->cam, c->world, t, c->det_K, c->det_uv, c->det_tag, c->det_n);
}

void launch_mm_plan(ekfslam_ctx* c, int min_features) {
    KScope ks(c, KT_ADD_FEATURES);
    k_mm_plan<<<(c->v.B + 3) / 4, 128, 0, c->stream>>>(c->v, min_features, c->det_n, c->det_K, c->mm_del, c->mm_quota);
}
