// C ABI of libekfslam.so (include/ekfslam.h): context management, host<->device marshalling
// of the reference's `filter` / `features_info` structs, and the stage sequencing of the
// filter step.  Host logic only — every arithmetic stage is a CUDA kernel; there is no CPU
// fallback (a missing device is an error).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <climits>
#include <string>
#include <vector>

#include "common.cuh"

static thread_local std::string g_err;
extern "C" { static void step_graph_destroy(ekfslam_ctx* c); }   // defined with ekfslam_step_graph

static int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define CK(call)                                                                              \
    do {                                                                                      \
        cudaError_t _e = (call);                                                              \
        if (_e != cudaSuccess)                                                                \
            return fail(EKFSLAM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorName(_e) + \
                                              " (" + cudaGetErrorString(_e) + ")");           \
    } while (0)

#define NEED_CTX(c)                                                     \
    do {                                                                \
        if (!(c)) return fail(EKFSLAM_ERR_INVALID, "null context");     \
        CK(cudaSetDevice((c)->device));                                 \
    } while (0)

// ---- per-kernel timing ---------------------------------------------------------------------
struct KTimer {
    struct Rec { cudaEvent_t a, b; int slot; };
    std::vector<Rec> pending;
    std::vector<cudaEvent_t> pool;
    double ms[KT_COUNT];
    long long count[KT_COUNT];
    cudaEvent_t cur[KT_COUNT];
};

static cudaEvent_t kt_event(KTimer* t) {
    if (!t->pool.empty()) { cudaEvent_t e = t->pool.back(); t->pool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    if (cudaEventCreate(&e) != cudaSuccess) { cudaGetLastError(); return nullptr; }   // this launch goes untimed
    return e;
}

void kt_begin(ekfslam_ctx* c, int slot) {
    KTimer* t = c->timer;
    t->cur[slot] = kt_event(t);
    if (t->cur[slot]) cudaEventRecord(t->cur[slot], c->stream);
}

// completed pairs at the head of the list are folded into the totals as soon as the list grows: a long run that never
// queries ekfslam_kernel_time keeps a bounded number of events alive
static void kt_drain_completed(KTimer* t) {
    size_t done = 0;
    while (done < t->pending.size() && cudaEventQuery(t->pending[done].b) == cudaSuccess) {
        KTimer::Rec& r = t->pending[done];
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) { t->ms[r.slot] += ms; t->count[r.slot]++; }
        t->pool.push_back(r.a);
        t->pool.push_back(r.b);
        ++done;
    }
    cudaGetLastError();   // cudaErrorNotReady of the first unfinished pair is not an error
    if (done) t->pending.erase(t->pending.begin(), t->pending.begin() + done);
}

void kt_end(ekfslam_ctx* c, int slot) {
    KTimer* t = c->timer;
    KTimer::Rec r;
    r.a = t->cur[slot]; r.b = r.a ? kt_event(t) : nullptr; r.slot = slot;
    if (!r.a || !r.b) { if (r.a) t->pool.push_back(r.a); return; }
    cudaEventRecord(r.b, c->stream);
    t->pending.push_back(r);
    if (t->pending.size() > 1024) kt_drain_completed(t);
}

static void kt_collect(ekfslam_ctx* c) {
    KTimer* t = c->timer;
    if (!t) return;
    for (auto& r : t->pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) { t->ms[r.slot] += ms; t->count[r.slot]++; }
        t->pool.push_back(r.a);
        t->pool.push_back(r.b);
    }
    t->pending.clear();
}

static const char* KT_NAMES[KT_COUNT] = {"k_begin_frame", "k_predict", "k_features", "k_hp", "k_innov", "k_ransac",
                                         "k_upd_S", "k_chol", "k_w", "k_downdate_hi", "k_downdate", "k_symmetrize",
                                         "k_add_features", "k_wfix", "k_w_hi", "k_chol_hi", "k_upd_S_hi",
                                         "k_hp_rescue", "k_world", "k_eval"};

template <typename T>
static cudaError_t dalloc(T** p, size_t count, int64_t* total) {
    const size_t bytes = count * sizeof(T);
    cudaError_t e = cudaMalloc((void**)p, bytes ? bytes : 1);
    if (e == cudaSuccess) {
        *total += (int64_t)bytes;
        e = cudaMemset(*p, 0, bytes ? bytes : 1);
    }
    return e;
}

extern "C" {

const char* ekfslam_last_error(void) { return g_err.c_str(); }
int ekfslam_version(void) { return 100; }

int ekfslam_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

void ekfslam_default_camera(ekfslam_camera* cam) {
    // mc/initialize_cam.m:3-10
    const double d = 0.0112;
    cam->k1 = 6.333e-2; cam->k2 = 1.390e-2;
    cam->Cx = 1.7945 / d; cam->Cy = 1.4433 / d;
    cam->f = 2.1735; cam->dx = d; cam->dy = d;
    cam->nRows = 240; cam->nCols = 320;
}

void ekfslam_default_params(ekfslam_params* p) {
    p->std_a = 0.007; p->std_alpha = 0.007; p->std_z = 1.0;  // mc/mono_slam.m:29-31
    p->delta_t = 1.0;                                         // mc/predict_state_and_covariance.m:5
    p->chi2_gate = 5.9915;                                    // mc/rescue_hi_inliers.m:3
    p->p_spurious_free = 0.99;                                // mc/ransac_hypotheses.m:3
    p->max_hyp = 1000;                                        // mc/ransac_hypotheses.m:9
    p->fixed_hyp = 0;
}

static void set_devcam(ekfslam_ctx* c, const ekfslam_camera* cam) {
    DevCam& d = c->cam;
    d.k1 = cam->k1; d.k2 = cam->k2; d.Cx = cam->Cx; d.Cy = cam->Cy; d.f = cam->f; d.dx = cam->dx; d.dy = cam->dy;
    d.fku = cam->f * (1.0 / cam->dx);  // f*ku, ku = 1/dx (mc/compute_hypothesis_support_fast.m:35-38)
    d.fkv = cam->f * (1.0 / cam->dy);
    d.nRows = (double)cam->nRows; d.nCols = (double)cam->nCols;
}

// mc/ransac_hypotheses.m:40-41 tabulated with the HOST libm for every (num_IC_matches, support):
//   epsilon = 1 - support/nIC;  n_hyp = ceil(log(1-p)/log(1-(1-epsilon)))
// Ratios such as support/nIC = 0.9 sit on an integer boundary of the ceil(); evaluating the two
// log() calls with the same libm as the CPU oracle keeps the hypothesis count identical.
static void build_nhyp_table(std::vector<int32_t>& tab, int N, double p) {
    tab.assign((size_t)(N + 1) * (N + 2) / 2, 0);
    const double num = std::log(1.0 - p);
    for (int nic = 1; nic <= N; ++nic)
        for (int s = 0; s <= nic; ++s) {
            const double epsilon = 1.0 - ((double)s / (double)nic);
            const double den = 1.0 - (1.0 - epsilon);
            double v;
            if (den <= 0.0) v = 0.0;  // log(0) = -Inf -> ceil(-0) = 0
            else {
                const double lden = std::log(den);
                v = (lden == 0.0) ? (double)INT_MAX : std::ceil(num / lden);
            }
            if (!(v < (double)INT_MAX)) v = (double)INT_MAX;
            if (v < 0.0) v = 0.0;
            tab[EKF_TRI(nic, s)] = (int32_t)v;
        }
}

int ekfslam_create(ekfslam_ctx** out, int device, int B, int N_max, int n_max) {
    if (!out) return fail(EKFSLAM_ERR_INVALID, "out is null");
    *out = nullptr;
    if (B <= 0 || N_max <= 0 || n_max < EKF_XV) return fail(EKFSLAM_ERR_INVALID, "B, N_max must be > 0 and n_max >= 13");
    if (B > 65535) return fail(EKFSLAM_ERR_INVALID, "B must be <= 65535 per context");
    if (n_max > EKF_XV + 6 * N_max) return fail(EKFSLAM_ERR_INVALID, "n_max exceeds 13 + 6*N_max");
    const int ndev = ekfslam_device_count();
    if (ndev <= 0) return fail(EKFSLAM_ERR_NODEVICE, "no CUDA device visible: libekfslam has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(EKFSLAM_ERR_INVALID, "device index out of range");
    CK(cudaSetDevice(device));
    ekfslam_ctx* c = new (std::nothrow) ekfslam_ctx();
    if (!c) return fail(EKFSLAM_ERR_NOMEM, "host allocation failed");
    memset(c, 0, sizeof(*c));
    c->device = device;
    DevView& v = c->v;
    v.B = B; v.N = N_max; v.nmax = n_max;
    // Row pitch of x / P / G in doubles: a multiple of 32 (256 B).  With the minimal pitch (multiple of 8: 616 at n = 613) the
    // 512-byte row segments of the 64x64 covariance tiles straddle 128-byte lines on every other row; measured on the
    // HBM-bound hi downdate at the bench shape: pitch 616 -> 4.22 ms, 624 -> 4.08 ms, 640 -> 3.78 ms.
    v.ld = (n_max + 31) / 32 * 32;
    v.kmax = 2 * N_max;
    v.n_u = 0;
    c->u_cap = 0;
    const size_t Bz = (size_t)B;
#define DA(ptr, count)                                                                           \
    do {                                                                                         \
        cudaError_t _e = dalloc(&(ptr), (count), &c->bytes);                                     \
        if (_e != cudaSuccess) {                                                                 \
            std::string m = std::string("cudaMalloc " #ptr ": ") + cudaGetErrorString(_e);       \
            ekfslam_destroy(c);                                                                  \
            return fail(_e == cudaErrorMemoryAllocation ? EKFSLAM_ERR_NOMEM : EKFSLAM_ERR_CUDA, m); \
        }                                                                                        \
    } while (0)
    DA(v.x, Bz * v.ld);
    DA(v.xp, Bz * v.ld);
    DA(v.P, Bz * v.nmax * v.ld);
    DA(v.G, Bz * v.kmax * v.ld);
    v.wrows = v.kmax;
    v.wstride = (long long)((v.ld + 63) / 64) * v.wrows * EKF_WPAD;
    DA(v.W, Bz * (size_t)v.wstride);
    DA(v.Sb, Bz * v.kmax * v.kmax);
    DA(v.Li, Bz * v.kmax * v.kmax);
    DA(v.yv, Bz * v.kmax);
    DA(v.jn, Bz * 16);
    DA(v.jnt, Bz * 16);
    DA(v.ktot, Bz);
    DA(v.kmaxdev, 1);
    DA(v.cv, Bz * v.kmax);
    DA(v.h, Bz * v.N * 2);
    DA(v.Hc, Bz * v.N * EKF_HSTRIDE);
    DA(v.S, Bz * v.N * 4);
    DA(v.z, Bz * v.N * 2);
    DA(v.zc, Bz * v.N * 2);
    DA(v.ftype, Bz * v.N);
    DA(v.flags, Bz * v.N);
    DA(v.mflags, Bz * v.N);
    DA(v.foff, Bz * v.N);
    DA(v.nstate, Bz);
    DA(v.nfeat, Bz);
    DA(v.counters, Bz * v.N * 2);
    DA(v.tag, Bz * v.N);
    DA(c->mm_del, Bz * v.N);
    DA(c->mm_quota, Bz);
    DA(c->det_n, Bz);
    DA(v.sel, Bz * v.N);
    DA(v.ksel, Bz);
    DA(v.stats, Bz);
    DA(v.nhyp_tab, (size_t)(v.N + 1) * (v.N + 2) / 2);
#undef DA
    ekfslam_camera cam;
    ekfslam_default_camera(&cam);
    set_devcam(c, &cam);
    ekfslam_default_params(&c->prm);
    std::vector<int32_t> tab;
    build_nhyp_table(tab, v.N, c->prm.p_spurious_free);
    cudaError_t e = cudaMemcpy(v.nhyp_tab, tab.data(), tab.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->aux_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->aux2_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_join2, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMallocHost((void**)&c->kmax_host, sizeof(int32_t));
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_in, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_out, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_main, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        ekfslam_destroy(c);
        return fail(EKFSLAM_ERR_CUDA, std::string("context init: ") + cudaGetErrorString(e));
    }
    c->stream = c->own_stream;
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (c->sm_count <= 0) c->sm_count = 148;
    *out = c;
    return EKFSLAM_OK;
}

int ekfslam_destroy(ekfslam_ctx* c) {
    if (!c) return EKFSLAM_OK;
    cudaSetDevice(c->device);
    if (c->own_zc) { c->v.zc = c->own_zc; c->v.mflags = c->own_mflags; c->v.u = c->own_u; c->own_zc = nullptr; }
    DevView& v = c->v;
    void* ptrs[] = {v.x, v.xp, v.P, v.G, v.W, v.Sb, v.Li, v.yv, v.jn, v.jnt, v.ktot, v.kmaxdev, v.cv, v.h, v.Hc, v.S, v.z, v.zc, v.u, v.ftype,
                    v.flags, v.mflags, v.foff, v.nstate, v.nfeat, v.counters, v.tag, v.sel, v.ksel, v.stats, v.nhyp_tab,
                    c->mm_del, c->mm_quota, c->det_n, c->det_uv, c->det_tag, c->world_points, c->world_poses,
                    c->ev.rec, c->ev.tot, c->ev.ferr, c->ev.fnees, c->ev.mp, c->ev.mc};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (c->timer) {
        cudaStreamSynchronize(c->stream);
        kt_collect(c);
        for (cudaEvent_t e : c->timer->pool) cudaEventDestroy(e);
        delete c->timer;
        c->timer = nullptr;
    }
    step_graph_destroy(c);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->aux_stream) cudaStreamDestroy(c->aux_stream);
    if (c->aux2_stream) cudaStreamDestroy(c->aux2_stream);
    if (c->ev_join2) cudaEventDestroy(c->ev_join2);
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    if (c->ev_in) cudaEventDestroy(c->ev_in);
    if (c->ev_out) cudaEventDestroy(c->ev_out);
    if (c->ev_main) cudaEventDestroy(c->ev_main);
    if (c->pin) cudaFree(c->pin);
    if (c->kmax_host) cudaFreeHost(c->kmax_host);
    delete c;
    return EKFSLAM_OK;
}

int ekfslam_set_stream(ekfslam_ctx* c, void* s) {
    NEED_CTX(c);
    c->stream = s ? (cudaStream_t)s : c->own_stream;
    return EKFSLAM_OK;
}

int ekfslam_set_camera(ekfslam_ctx* c, const ekfslam_camera* cam) {
    NEED_CTX(c);
    if (!cam) return fail(EKFSLAM_ERR_INVALID, "cam is null");
    if (!(cam->dx > 0) || !(cam->dy > 0) || cam->nRows <= 0 || cam->nCols <= 0)
        return fail(EKFSLAM_ERR_INVALID, "camera: dx, dy, nRows, nCols must be positive");
    set_devcam(c, cam);
    return EKFSLAM_OK;
}

int ekfslam_set_params(ekfslam_ctx* c, const ekfslam_params* p) {
    NEED_CTX(c);
    if (!p) return fail(EKFSLAM_ERR_INVALID, "params is null");
    if (p->max_hyp <= 0 || p->fixed_hyp < 0 || !(p->p_spurious_free > 0 && p->p_spurious_free < 1))
        return fail(EKFSLAM_ERR_INVALID, "params: max_hyp > 0, fixed_hyp >= 0, 0 < p_spurious_free < 1");
    const bool retab = p->p_spurious_free != c->prm.p_spurious_free;
    c->prm = *p;
    if (retab) {
        std::vector<int32_t> tab;
        build_nhyp_table(tab, c->v.N, p->p_spurious_free);
        CK(cudaMemcpyAsync(c->v.nhyp_tab, tab.data(), tab.size() * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
    return EKFSLAM_OK;
}

int ekfslam_synchronize(ekfslam_ctx* c) {
    NEED_CTX(c);
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaGetLastError());
    return EKFSLAM_OK;
}

int ekfslam_dims(const ekfslam_ctx* c, int* B, int* N_max, int* n_max, int* ld) {
    if (!c) return fail(EKFSLAM_ERR_INVALID, "null context");
    if (B) *B = c->v.B;
    if (N_max) *N_max = c->v.N;
    if (n_max) *n_max = c->v.nmax;
    if (ld) *ld = c->v.ld;
    return EKFSLAM_OK;
}

int ekfslam_enable_timing(ekfslam_ctx* c, int on) {
    NEED_CTX(c);
    CK(cudaStreamSynchronize(c->stream));
    if (on && !c->timer) {
        c->timer = new KTimer();
        memset(c->timer->ms, 0, sizeof(c->timer->ms));
        memset(c->timer->count, 0, sizeof(c->timer->count));
    } else if (on && c->timer) {
        kt_collect(c);
        memset(c->timer->ms, 0, sizeof(c->timer->ms));
        memset(c->timer->count, 0, sizeof(c->timer->count));
    } else if (!on && c->timer) {
        kt_collect(c);
        for (cudaEvent_t e : c->timer->pool) cudaEventDestroy(e);
        delete c->timer;
        c->timer = nullptr;
    }
    return EKFSLAM_OK;
}

int ekfslam_kernel_count(void) { return KT_COUNT; }

int ekfslam_kernel_time(ekfslam_ctx* c, int slot, char* name, int name_cap, double* ms, int64_t* launches) {
    NEED_CTX(c);
    if (slot < 0 || slot >= KT_COUNT) return fail(EKFSLAM_ERR_INVALID, "kernel slot out of range");
    if (!c->timer) return fail(EKFSLAM_ERR_STATE, "timing is not enabled");
    CK(cudaStreamSynchronize(c->stream));
    kt_collect(c);
    if (name && name_cap > 0) { strncpy(name, KT_NAMES[slot], name_cap - 1); name[name_cap - 1] = 0; }
    if (ms) *ms = c->timer->ms[slot];
    if (launches) *launches = c->timer->count[slot];
    return EKFSLAM_OK;
}

int ekfslam_bind_frame(ekfslam_ctx* c, const void* d_zc, const void* d_fl, const void* d_u, int n_u) {
    NEED_CTX(c);
    if (!d_zc || !d_fl || !d_u || n_u <= 0) return fail(EKFSLAM_ERR_INVALID, "bind_frame: null pointer or n_u <= 0");
    if (!c->own_zc) { c->own_zc = c->v.zc; c->own_mflags = c->v.mflags; c->own_u = c->v.u; c->own_n_u = c->v.n_u; }
    c->v.zc = (double*)d_zc; c->v.mflags = (uint8_t*)d_fl; c->v.u = (double*)d_u; c->v.n_u = n_u;
    return EKFSLAM_OK;
}

int ekfslam_unbind_frame(ekfslam_ctx* c) {
    NEED_CTX(c);
    if (c->own_zc) {
        c->v.zc = c->own_zc; c->v.mflags = c->own_mflags; c->v.u = c->own_u; c->v.n_u = c->own_n_u;
        c->own_zc = nullptr; c->own_mflags = nullptr; c->own_u = nullptr;
    }
    return EKFSLAM_OK;
}

int64_t ekfslam_device_bytes(const ekfslam_ctx* c) { return c ? c->bytes : 0; }
int64_t ekfslam_launch_count(const ekfslam_ctx* c) { return c ? c->launches : 0; }

static int check_range(const ekfslam_ctx* c, int b0, int nb) {
    if (b0 < 0 || nb <= 0 || b0 + nb > c->v.B) return fail(EKFSLAM_ERR_INVALID, "filter range [b0, b0+nb) out of bounds");
    return EKFSLAM_OK;
}

// ---- filter struct <-> device ------------------------------------------------------------
int ekfslam_upload_state(ekfslam_ctx* c, int b0, int nb, int which, const double* x, const double* P,
                         const int32_t* nstate) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    DevView& v = c->v;
    if (nstate) {
        for (int i = 0; i < nb; ++i)
            if (nstate[i] < EKF_XV || nstate[i] > v.nmax) return fail(EKFSLAM_ERR_INVALID, "nstate out of [13, n_max]");
        CK(cudaMemcpyAsync(v.nstate + b0, nstate, sizeof(int32_t) * nb, cudaMemcpyHostToDevice, c->stream));
    }
    if (x) {
        double* dst = (which ? v.xp : v.x) + (size_t)b0 * v.ld;
        CK(cudaMemcpy2DAsync(dst, sizeof(double) * v.ld, x, sizeof(double) * v.nmax, sizeof(double) * v.nmax, nb,
                             cudaMemcpyHostToDevice, c->stream));
    }
    if (P) {
        // host: nb matrices of n_max x n_max (ld n_max); device rows padded to ld (padding stays zero)
        double* dst = v.P + (size_t)b0 * v.nmax * v.ld;
        CK(cudaMemcpy2DAsync(dst, sizeof(double) * v.ld, P, sizeof(double) * v.nmax, sizeof(double) * v.nmax,
                             (size_t)nb * v.nmax, cudaMemcpyHostToDevice, c->stream));
        launch_symmetrize(c, b0, nb);  // lower triangle is authoritative (see k_symmetrize)
    }
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

int ekfslam_download_state(ekfslam_ctx* c, int b0, int nb, int which, double* x, double* P, int32_t* nstate) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    DevView& v = c->v;
    if (nstate) CK(cudaMemcpyAsync(nstate, v.nstate + b0, sizeof(int32_t) * nb, cudaMemcpyDeviceToHost, c->stream));
    if (x) {
        const double* src = (which ? v.xp : v.x) + (size_t)b0 * v.ld;
        CK(cudaMemcpy2DAsync(x, sizeof(double) * v.nmax, src, sizeof(double) * v.ld, sizeof(double) * v.nmax, nb,
                             cudaMemcpyDeviceToHost, c->stream));
    }
    if (P) {
        const double* src = v.P + (size_t)b0 * v.nmax * v.ld;
        CK(cudaMemcpy2DAsync(P, sizeof(double) * v.nmax, src, sizeof(double) * v.ld, sizeof(double) * v.nmax,
                             (size_t)nb * v.nmax, cudaMemcpyDeviceToHost, c->stream));
    }
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

// ---- features_info <-> device --------------------------------------------------------------
int ekfslam_upload_feature_types(ekfslam_ctx* c, int b0, int nb, const uint8_t* type, const int32_t* nfeat) {
    NEED_CTX(c);
    if (c->own_zc) return fail(EKFSLAM_ERR_STATE, "frame buffers are bound to caller memory (ekfslam_unbind_frame first)");
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    if (!type || !nfeat) return fail(EKFSLAM_ERR_INVALID, "type / nfeat is null");
    DevView& v = c->v;
    std::vector<int32_t> off((size_t)nb * v.N, 0), ns(nb);
    for (int i = 0; i < nb; ++i) {
        if (nfeat[i] < 0 || nfeat[i] > v.N) return fail(EKFSLAM_ERR_INVALID, "nfeat out of [0, N_max]");
        int pos = EKF_XV;  // mc/calculate_Hi_inverse_depth.m:22 (index_of_insertion, 0-based)
        for (int f = 0; f < nfeat[i]; ++f) {
            const uint8_t t = type[(size_t)i * v.N + f];
            if (t != EKFSLAM_FEAT_INVERSEDEPTH && t != EKFSLAM_FEAT_CARTESIAN)
                return fail(EKFSLAM_ERR_INVALID, "feature type must be 1 (inversedepth) or 2 (cartesian)");
            off[(size_t)i * v.N + f] = pos;
            pos += (t == EKFSLAM_FEAT_INVERSEDEPTH) ? 6 : 3;
        }
        if (pos > v.nmax) return fail(EKFSLAM_ERR_INVALID, "features do not fit in n_max");
        ns[i] = pos;
    }
    const size_t o = (size_t)b0 * v.N;
    CK(cudaMemcpyAsync(v.ftype + o, type, (size_t)nb * v.N, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(v.foff + o, off.data(), sizeof(int32_t) * nb * v.N, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(v.nfeat + b0, nfeat, sizeof(int32_t) * nb, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(v.nstate + b0, ns.data(), sizeof(int32_t) * nb, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemsetAsync(v.flags + o, 0, (size_t)nb * v.N, c->stream));
    CK(cudaMemsetAsync(v.mflags + o, 0, (size_t)nb * v.N, c->stream));
    CK(cudaMemsetAsync(v.counters + 2 * o, 0, sizeof(int32_t) * 2 * nb * v.N, c->stream));
    CK(cudaMemsetAsync(v.tag + o, 0xff, sizeof(int32_t) * nb * v.N, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

static int upload_zc(ekfslam_ctx* c, int b0, int nb, const double* z, const uint8_t* fl, bool sync) {
    if (c->own_zc) return fail(EKFSLAM_ERR_STATE, "frame buffers are bound to caller memory (ekfslam_unbind_frame first)");
    DevView& v = c->v;
    const size_t o = (size_t)b0 * v.N;
    if (z) CK(cudaMemcpyAsync(v.zc + 2 * o, z, sizeof(double) * 2 * nb * v.N, cudaMemcpyHostToDevice, c->stream));
    if (fl) CK(cudaMemcpyAsync(v.mflags + o, fl, (size_t)nb * v.N, cudaMemcpyHostToDevice, c->stream));
    if (sync) CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

int ekfslam_upload_matches(ekfslam_ctx* c, int b0, int nb, const double* z, const uint8_t* flags) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    if (!z || !flags) return fail(EKFSLAM_ERR_INVALID, "z / flags is null");
    return upload_zc(c, b0, nb, z, flags, true);
}

int ekfslam_upload_candidates(ekfslam_ctx* c, int b0, int nb, const double* zc, const uint8_t* has) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    if (!zc || !has) return fail(EKFSLAM_ERR_INVALID, "zc / has is null");
    // normalise any non-zero byte to the CAND bit
    std::vector<uint8_t> fl((size_t)nb * c->v.N);
    for (size_t i = 0; i < fl.size(); ++i) fl[i] = has[i] ? EKFSLAM_F_CAND : 0;
    return upload_zc(c, b0, nb, zc, fl.data(), true);
}

static int ensure_u(ekfslam_ctx* c, int n_u) {
    if (c->own_zc) return fail(EKFSLAM_ERR_STATE, "frame buffers are bound to caller memory (ekfslam_unbind_frame first)");
    DevView& v = c->v;
    if (n_u > c->u_cap) {
        if (v.u) { CK(cudaStreamSynchronize(c->stream)); CK(cudaFree(v.u)); v.u = nullptr; }
        CK(cudaMalloc((void**)&v.u, sizeof(double) * (size_t)v.B * n_u));
        CK(cudaMemsetAsync(v.u, 0, sizeof(double) * (size_t)v.B * n_u, c->stream));
        c->bytes += (int64_t)sizeof(double) * v.B * (n_u - c->u_cap);
        c->u_cap = n_u;
    }
    return EKFSLAM_OK;
}

int ekfslam_upload_uniforms(ekfslam_ctx* c, int b0, int nb, const double* u, int n_u) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    if (!u || n_u <= 0) return fail(EKFSLAM_ERR_INVALID, "u is null or n_u <= 0");
    DevView& v = c->v;
    if (n_u != v.n_u && !(b0 == 0 && nb == v.B) && v.n_u != 0)
        return fail(EKFSLAM_ERR_INVALID, "changing n_u requires uploading all B filters at once");
    if (int r = ensure_u(c, n_u)) return r;
    v.n_u = n_u;
    CK(cudaMemcpyAsync(v.u + (size_t)b0 * n_u, u, sizeof(double) * (size_t)nb * n_u, cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

int ekfslam_download_features(ekfslam_ctx* c, int b0, int nb, double* h, double* Hc, double* S, double* z,
                              uint8_t* flags, int32_t* offs, int32_t* counters) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    DevView& v = c->v;
    const size_t o = (size_t)b0 * v.N, cnt = (size_t)nb * v.N;
    if (h) CK(cudaMemcpyAsync(h, v.h + 2 * o, sizeof(double) * 2 * cnt, cudaMemcpyDeviceToHost, c->stream));
    if (Hc) CK(cudaMemcpyAsync(Hc, v.Hc + EKF_HSTRIDE * o, sizeof(double) * EKF_HSTRIDE * cnt, cudaMemcpyDeviceToHost, c->stream));
    if (S) CK(cudaMemcpyAsync(S, v.S + 4 * o, sizeof(double) * 4 * cnt, cudaMemcpyDeviceToHost, c->stream));
    if (z) CK(cudaMemcpyAsync(z, v.z + 2 * o, sizeof(double) * 2 * cnt, cudaMemcpyDeviceToHost, c->stream));
    if (flags) CK(cudaMemcpyAsync(flags, v.flags + o, cnt, cudaMemcpyDeviceToHost, c->stream));
    if (offs) CK(cudaMemcpyAsync(offs, v.foff + o, sizeof(int32_t) * cnt, cudaMemcpyDeviceToHost, c->stream));
    if (counters) CK(cudaMemcpyAsync(counters, v.counters + 2 * o, sizeof(int32_t) * 2 * cnt, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

int ekfslam_upload_features(ekfslam_ctx* c, int b0, int nb, const double* h, const double* Hc, const double* S,
                            const double* z, const uint8_t* flags) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    DevView& v = c->v;
    const size_t o = (size_t)b0 * v.N, cnt = (size_t)nb * v.N;
    if (h) CK(cudaMemcpyAsync(v.h + 2 * o, h, sizeof(double) * 2 * cnt, cudaMemcpyHostToDevice, c->stream));
    if (Hc) CK(cudaMemcpyAsync(v.Hc + EKF_HSTRIDE * o, Hc, sizeof(double) * EKF_HSTRIDE * cnt, cudaMemcpyHostToDevice, c->stream));
    if (S) CK(cudaMemcpyAsync(v.S + 4 * o, S, sizeof(double) * 4 * cnt, cudaMemcpyHostToDevice, c->stream));
    if (z) CK(cudaMemcpyAsync(v.z + 2 * o, z, sizeof(double) * 2 * cnt, cudaMemcpyHostToDevice, c->stream));
    if (flags) CK(cudaMemcpyAsync(v.flags + o, flags, cnt, cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

int ekfslam_download_feature_types(ekfslam_ctx* c, int b0, int nb, uint8_t* type, int32_t* nfeat) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    DevView& v = c->v;
    if (type) CK(cudaMemcpyAsync(type, v.ftype + (size_t)b0 * v.N, (size_t)nb * v.N, cudaMemcpyDeviceToHost, c->stream));
    if (nfeat) CK(cudaMemcpyAsync(nfeat, v.nfeat + b0, sizeof(int32_t) * nb, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

int ekfslam_download_stats(ekfslam_ctx* c, int b0, int nb, ekfslam_stats* stats) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    if (!stats) return fail(EKFSLAM_ERR_INVALID, "stats is null");
    CK(cudaMemcpyAsync(stats, c->v.stats + b0, sizeof(ekfslam_stats) * nb, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

// ---- stages ---------------------------------------------------------------------------------
#define LAUNCHED()                                                                                     \
    do {                                                                                               \
        cudaError_t _e = cudaGetLastError();                                                           \
        if (_e != cudaSuccess) return fail(EKFSLAM_ERR_CUDA, std::string("kernel launch: ") + cudaGetErrorString(_e)); \
    } while (0)

int ekfslam_begin_frame(ekfslam_ctx* c) {
    NEED_CTX(c);
    launch_begin_frame(c);
    LAUNCHED();
    return EKFSLAM_OK;
}

int ekfslam_predict(ekfslam_ctx* c) {
    NEED_CTX(c);
    launch_predict(c);
    LAUNCHED();
    return EKFSLAM_OK;
}

int ekfslam_features(ekfslam_ctx* c, int which, int parts) {
    NEED_CTX(c);
    if (parts < 1 || parts > 3) return fail(EKFSLAM_ERR_INVALID, "parts must be 1 (h), 2 (H) or 3 (both)");
    launch_features(c, which ? 1 : 0, parts);
    LAUNCHED();
    return EKFSLAM_OK;
}

int ekfslam_hp(ekfslam_ctx* c, int need, int forbid) {
    NEED_CTX(c);
    launch_hp(c, need, forbid);
    LAUNCHED();
    return EKFSLAM_OK;
}

int ekfslam_innovation(ekfslam_ctx* c) {
    NEED_CTX(c);
    launch_innov_gather(c, 0);
    LAUNCHED();
    return EKFSLAM_OK;
}

int ekfslam_measure(ekfslam_ctx* c, int which) {
    NEED_CTX(c);
    launch_features(c, which ? 1 : 0, 3);
    launch_innov_gather(c, 0);   // S_i from 13x13 gathers of P: the full rows H P are built where they are consumed
    LAUNCHED();               // (ekfslam_ransac: per hypothesis; ekfslam_update_li / ekfslam_hp: per update)
    return EKFSLAM_OK;
}

// mode: 1 = gate the staged candidates, 2 = apply the staged explicit matches
static int gate_mode(ekfslam_ctx* c, int mode) {
    launch_innov(c, mode);
    LAUNCHED();
    return EKFSLAM_OK;
}

int ekfslam_gate(ekfslam_ctx* c) {
    NEED_CTX(c);
    return gate_mode(c, 1);
}

int ekfslam_apply_matches(ekfslam_ctx* c) {
    NEED_CTX(c);
    return gate_mode(c, 2);
}

int ekfslam_ransac(ekfslam_ctx* c) {
    NEED_CTX(c);
    if (c->v.n_u <= 0) return fail(EKFSLAM_ERR_STATE, "ransac: no uniform stream uploaded (ekfslam_upload_uniforms)");
    launch_ransac(c);
    LAUNCHED();
    return EKFSLAM_OK;
}

int ekfslam_update_masked(ekfslam_ctx* c, int mask, int which_prior) {
    NEED_CTX(c);
    if (!(mask & 0xff)) return fail(EKFSLAM_ERR_INVALID, "empty mask");
    launch_update(c, mask, which_prior ? 1 : 0);
    LAUNCHED();
    return EKFSLAM_OK;
}

int ekfslam_update_li(ekfslam_ctx* c) {
    NEED_CTX(c);
    launch_hp(c, EKFSLAM_F_HAS_H | EKFSLAM_F_LI, 0);   // G rows of the low-innovation inliers
    return ekfslam_update_masked(c, EKFSLAM_F_LI, 1);
}

int ekfslam_update_iterated(ekfslam_ctx* c, int mask, int which_prior, int n_iter) {
    NEED_CTX(c);
    if (!(mask & 0xff)) return fail(EKFSLAM_ERR_INVALID, "empty mask");
    if (n_iter < 1 || n_iter > 64) return fail(EKFSLAM_ERR_INVALID, "n_iter must be in [1, 64]");
    DevView& v = c->v;
    const size_t xbytes = sizeof(double) * (size_t)v.B * v.ld;
    // the prior lives in xp; the running iterate x_j in x (x_0 = prior)
    if (which_prior) CK(cudaMemcpyAsync(v.x, v.xp, xbytes, cudaMemcpyDeviceToDevice, c->stream));
    else CK(cudaMemcpyAsync(v.xp, v.x, xbytes, cudaMemcpyDeviceToDevice, c->stream));
    for (int j = 0; j < n_iter; ++j) {
        launch_features(c, 0, 3);         // h(x_j), H_j for every feature (stale-h rule as in the reference)
        launch_hp(c, mask & 0xff, 0);     // G = H_j P^-  (P is untouched until the last iteration)
        launch_update(c, mask, 1, 1 | (j + 1 < n_iter ? 2 : 0));
    }
    LAUNCHED();
    return EKFSLAM_OK;
}

int ekfslam_rescue(ekfslam_ctx* c) {
    NEED_CTX(c);
    launch_features(c, 0, 3);                            // h, H of ALL features at x_k_k (:6-7)
    launch_innov_gather(c, 3);                           // chi2 gate of the candidates (IC && !LI) -> HI (:11-20)
    launch_hp(c, EKFSLAM_F_HAS_H | EKFSLAM_F_HI, 0, KT_HP_RESCUE);   // G rows of the rescued features for ekfslam_update_hi
    LAUNCHED();
    return EKFSLAM_OK;
}

int ekfslam_update_hi(ekfslam_ctx* c) { return ekfslam_update_masked(c, EKFSLAM_F_HI, 0); }

int ekfslam_step(ekfslam_ctx* c, int reset, int match_mode) {
    NEED_CTX(c);
    if (match_mode < 0 || match_mode > 2) return fail(EKFSLAM_ERR_INVALID, "match_mode must be 0, 1 or 2");
    if (c->v.n_u <= 0) return fail(EKFSLAM_ERR_STATE, "step: no uniform stream uploaded");
    if (reset) launch_begin_frame(c);
    launch_predict(c);
    launch_features(c, 1, 3);
    launch_innov_gather(c, 0);                              // S_i from 13x13 gathers of P: no G rows needed yet
    if (c->wait_inputs) { cudaStreamWaitEvent(c->stream, c->ev_in, 0); c->wait_inputs = 0; }
    if (match_mode) launch_innov(c, match_mode);
    launch_ransac(c);                                    // builds the G rows of the hypotheses it scores
    {
        // G rows of the low-innovation inliers only (with a fixed hypothesis budget launch_ransac has already built the
        // rows of every individually compatible feature, a superset)
        if (c->prm.fixed_hyp <= 0) launch_hp(c, EKFSLAM_F_HAS_H | EKFSLAM_F_LI, 0);
        launch_update(c, EKFSLAM_F_LI, 1);
        launch_features(c, 0, 3);
        launch_innov_gather(c, 3);                                        // chi2 gate from 13x13 gathers of p_k_k
        launch_hp(c, EKFSLAM_F_HAS_H | EKFSLAM_F_HI, 0, KT_HP_RESCUE);    // G rows only for the hi inliers
        launch_update(c, EKFSLAM_F_HI, 0);
    }
    LAUNCHED();
    return EKFSLAM_OK;
}

// ---- the filter step as a CUDA graph (latency path: few filters, ~25 small launches per frame) -----------------
struct StepGraph {
    cudaGraphExec_t exec;
    DevView v; ekfslam_params prm; DevCam cam;
    int reset, match_mode;
    int64_t launches;
};

static void step_graph_destroy(ekfslam_ctx* c) {
    StepGraph* g = (StepGraph*)c->step_graph;
    if (g) { if (g->exec) cudaGraphExecDestroy(g->exec); delete g; c->step_graph = nullptr; }
}

int ekfslam_step_graph(ekfslam_ctx* c, int reset, int match_mode) {
    NEED_CTX(c);
    DevView& v = c->v;
    // not capturable: per-kernel timing (event queries), the lock-step Cholesky (host read-back of the largest stacked
    // size), the host-buffer step's cross-stream events
    if (c->timer || chol_lockstep(v) || c->wait_inputs || c->arm_out) return ekfslam_step(c, reset, match_mode);
    if (match_mode < 0 || match_mode > 2) return fail(EKFSLAM_ERR_INVALID, "match_mode must be 0, 1 or 2");
    if (v.n_u <= 0) return fail(EKFSLAM_ERR_STATE, "step: no uniform stream uploaded");
    StepGraph* g = (StepGraph*)c->step_graph;
    if (g && (memcmp(&g->v, &v, sizeof(DevView)) || memcmp(&g->prm, &c->prm, sizeof(ekfslam_params)) ||
              memcmp(&g->cam, &c->cam, sizeof(DevCam)) || g->reset != reset || g->match_mode != match_mode)) {
        step_graph_destroy(c);
        g = nullptr;
    }
    if (!g) {
        g = new (std::nothrow) StepGraph();
        if (!g) return fail(EKFSLAM_ERR_NOMEM, "host allocation failed");
        memset(g, 0, sizeof(*g));
        memcpy(&g->v, &v, sizeof(DevView)); memcpy(&g->prm, &c->prm, sizeof(ekfslam_params)); memcpy(&g->cam, &c->cam, sizeof(DevCam));
        g->reset = reset; g->match_mode = match_mode;
        const int64_t l0 = c->launches;
        cudaGraph_t graph = nullptr;
        cudaError_t e = cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeRelaxed);
        if (e != cudaSuccess) { delete g; return fail(EKFSLAM_ERR_CUDA, std::string("cudaStreamBeginCapture: ") + cudaGetErrorString(e)); }
        const int rs = ekfslam_step(c, reset, match_mode);
        e = cudaStreamEndCapture(c->stream, &graph);
        g->launches = c->launches - l0;
        c->launches = l0;                                  // nothing has executed yet
        if (rs != EKFSLAM_OK || e != cudaSuccess || !graph) {
            if (graph) cudaGraphDestroy(graph);
            delete g;
            cudaGetLastError();
            if (rs != EKFSLAM_OK) return rs;
            return fail(EKFSLAM_ERR_CUDA, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e));
        }
        e = cudaGraphInstantiate(&g->exec, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) { delete g; return fail(EKFSLAM_ERR_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e)); }
        c->step_graph = g;
    }
    CK(cudaGraphLaunch(g->exec, c->stream));
    c->launches += g->launches;
    return EKFSLAM_OK;
}

// device-resident frame -> the context's OWN frame buffers by copy (unlike ekfslam_bind_frame the buffer addresses the
// kernels see do not change, so a captured step graph stays valid)
int ekfslam_stage_frame(ekfslam_ctx* c, const void* d_zc, const void* d_fl, const void* d_u, int n_u) {
    NEED_CTX(c);
    if (!d_zc || !d_fl || !d_u || n_u <= 0) return fail(EKFSLAM_ERR_INVALID, "stage_frame: null pointer or n_u <= 0");
    if (c->own_zc) return fail(EKFSLAM_ERR_STATE, "frame buffers are bound to caller memory (ekfslam_unbind_frame first)");
    DevView& v = c->v;
    if (int r = ensure_u(c, n_u)) return r;
    v.n_u = n_u;
    const size_t bn = (size_t)v.B * v.N;
    CK(cudaMemcpyAsync(v.zc, d_zc, sizeof(double) * 2 * bn, cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaMemcpyAsync(v.mflags, d_fl, bn, cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaMemcpyAsync(v.u, d_u, sizeof(double) * (size_t)v.B * n_u, cudaMemcpyDeviceToDevice, c->stream));
    return EKFSLAM_OK;
}

int ekfslam_step_host(ekfslam_ctx* c, int match_mode, const double* zc, const uint8_t* fl, const double* u, int n_u,
                      double* x_out, uint8_t* flags_out, ekfslam_stats* stats_out) {
    NEED_CTX(c);
    if (match_mode != 1 && match_mode != 2) return fail(EKFSLAM_ERR_INVALID, "match_mode must be 1 (gate) or 2 (explicit)");
    if (!zc || !fl || !u || n_u <= 0) return fail(EKFSLAM_ERR_INVALID, "zc / flags / u is null or n_u <= 0");
    DevView& v = c->v;
    if (int r = ensure_u(c, n_u)) return r;
    v.n_u = n_u;
    if (c->own_zc) return fail(EKFSLAM_ERR_STATE, "frame buffers are bound to caller memory (ekfslam_unbind_frame first)");
    // inputs: copy stream, ordered after whatever the compute stream still has queued
    const size_t bn = (size_t)v.B * v.N;
    CK(cudaEventRecord(c->ev_main, c->stream));
    CK(cudaStreamWaitEvent(c->copy_stream, c->ev_main, 0));
    CK(cudaMemcpyAsync(v.zc, zc, sizeof(double) * 2 * bn, cudaMemcpyHostToDevice, c->copy_stream));
    CK(cudaMemcpyAsync(v.mflags, fl, bn, cudaMemcpyHostToDevice, c->copy_stream));
    CK(cudaMemcpyAsync(v.u, u, sizeof(double) * (size_t)v.B * n_u, cudaMemcpyHostToDevice, c->copy_stream));
    CK(cudaEventRecord(c->ev_in, c->copy_stream));
    c->wait_inputs = 1;
    c->arm_out = 1;
    const int rs = ekfslam_step(c, 1, match_mode);
    c->wait_inputs = 0;
    if (rs) { c->arm_out = 0; return rs; }
    if (c->arm_out) { CK(cudaEventRecord(c->ev_out, c->stream)); c->arm_out = 0; }   // not recorded inside the step
    // outputs: x_k_k, flags and stats are final before the last covariance downdate (it only writes P)
    CK(cudaStreamWaitEvent(c->copy_stream, c->ev_out, 0));
    if (x_out)
        CK(cudaMemcpy2DAsync(x_out, sizeof(double) * v.nmax, v.x, sizeof(double) * v.ld, sizeof(double) * v.nmax, v.B,
                             cudaMemcpyDeviceToHost, c->copy_stream));
    if (flags_out) CK(cudaMemcpyAsync(flags_out, v.flags, bn, cudaMemcpyDeviceToHost, c->copy_stream));
    if (stats_out) CK(cudaMemcpyAsync(stats_out, v.stats, sizeof(ekfslam_stats) * v.B, cudaMemcpyDeviceToHost, c->copy_stream));
    CK(cudaStreamSynchronize(c->copy_stream));
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

int ekfslam_reset_filters(ekfslam_ctx* c, int b0, int nb, const double* xv, const double* Pxv) {
    NEED_CTX(c);
    if (c->own_zc) return fail(EKFSLAM_ERR_STATE, "frame buffers are bound to caller memory (ekfslam_unbind_frame first)");
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    if (!xv || !Pxv) return fail(EKFSLAM_ERR_INVALID, "xv / Pxv is null");
    DevView& v = c->v;
    const size_t need = sizeof(double) * (13 + 169);
    if (need > c->pin_bytes) {
        if (c->pin) { CK(cudaStreamSynchronize(c->stream)); CK(cudaFree(c->pin)); c->pin = nullptr; c->pin_bytes = 0; }
        CK(cudaMalloc(&c->pin, need));
        c->pin_bytes = need;
    }
    double* d = (double*)c->pin;
    CK(cudaMemcpyAsync(d, xv, sizeof(double) * 13, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(d + 13, Pxv, sizeof(double) * 169, cudaMemcpyHostToDevice, c->stream));
    const size_t o = (size_t)b0 * v.N;
    CK(cudaMemsetAsync(v.x + (size_t)b0 * v.ld, 0, sizeof(double) * (size_t)nb * v.ld, c->stream));
    CK(cudaMemsetAsync(v.xp + (size_t)b0 * v.ld, 0, sizeof(double) * (size_t)nb * v.ld, c->stream));
    CK(cudaMemsetAsync(v.P + (size_t)b0 * v.nmax * v.ld, 0, sizeof(double) * (size_t)nb * v.nmax * v.ld, c->stream));
    CK(cudaMemsetAsync(v.ftype + o, 0, (size_t)nb * v.N, c->stream));
    CK(cudaMemsetAsync(v.flags + o, 0, (size_t)nb * v.N, c->stream));
    CK(cudaMemsetAsync(v.mflags + o, 0, (size_t)nb * v.N, c->stream));
    CK(cudaMemsetAsync(v.foff + o, 0, sizeof(int32_t) * nb * v.N, c->stream));
    CK(cudaMemsetAsync(v.counters + 2 * o, 0, sizeof(int32_t) * 2 * nb * v.N, c->stream));
    CK(cudaMemsetAsync(v.tag + o, 0xff, sizeof(int32_t) * nb * v.N, c->stream));
    CK(cudaMemsetAsync(v.stats + b0, 0, sizeof(ekfslam_stats) * nb, c->stream));
    launch_reset_filters(c, b0, nb, d, d + 13);
    LAUNCHED();
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

int ekfslam_add_features(ekfslam_ctx* c, int b0, int nb, const double* uvd, const uint8_t* add, double std_pxl,
                         double initial_rho, double std_rho) {
    NEED_CTX(c);
    if (c->own_zc) return fail(EKFSLAM_ERR_STATE, "frame buffers are bound to caller memory (ekfslam_unbind_frame first)");
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    if (!uvd) return fail(EKFSLAM_ERR_INVALID, "uvd is null");
    // staging buffers for the pixels / mask (grown on demand, freed with the context)
    const size_t need = sizeof(double) * 2 * (size_t)nb + (size_t)nb;
    if (need > c->pin_bytes) {
        if (c->pin) { CK(cudaStreamSynchronize(c->stream)); CK(cudaFree(c->pin)); c->pin = nullptr; c->pin_bytes = 0; }
        CK(cudaMalloc(&c->pin, need));
        c->pin_bytes = need;
    }
    double* d_uvd = (double*)c->pin;
    uint8_t* d_add = (uint8_t*)(d_uvd + 2 * (size_t)nb);
    CK(cudaMemcpyAsync(d_uvd, uvd, sizeof(double) * 2 * nb, cudaMemcpyHostToDevice, c->stream));
    if (add) CK(cudaMemcpyAsync(d_add, add, nb, cudaMemcpyHostToDevice, c->stream));
    launch_add_features(c, b0, nb, d_uvd, 2, add ? d_add : nullptr, nullptr, 0, nullptr, 0, std_pxl, initial_rho, std_rho);
    LAUNCHED();
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

static int ensure_scratch(ekfslam_ctx* c, size_t need) {
    if (need > c->pin_bytes) {
        if (c->pin) { CK(cudaStreamSynchronize(c->stream)); CK(cudaFree(c->pin)); c->pin = nullptr; c->pin_bytes = 0; }
        CK(cudaMalloc(&c->pin, need));
        c->pin_bytes = need;
    }
    return EKFSLAM_OK;
}

int ekfslam_inversedepth_2_cartesian(ekfslam_ctx* c, double threshold, int force_index, int32_t* converted) {
    NEED_CTX(c);
    DevView& v = c->v;
    if (v.nmax > 512 * 8) return fail(EKFSLAM_ERR_INVALID, "inversedepth_2_cartesian supports n_max <= 4096");
    if (force_index >= v.N) return fail(EKFSLAM_ERR_INVALID, "force_index out of range");
    if (int r = ensure_scratch(c, sizeof(int32_t) * (size_t)v.B)) return r;
    launch_id2cart(c, threshold, force_index, (int32_t*)c->pin);
    LAUNCHED();
    if (converted) CK(cudaMemcpyAsync(converted, c->pin, sizeof(int32_t) * v.B, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

int ekfslam_delete_features(ekfslam_ctx* c, int b0, int nb, const uint8_t* del) {
    NEED_CTX(c);
    if (c->own_zc) return fail(EKFSLAM_ERR_STATE, "frame buffers are bound to caller memory (ekfslam_unbind_frame first)");
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    if (!del) return fail(EKFSLAM_ERR_INVALID, "del is null");
    DevView& v = c->v;
    if (v.nmax > 512 * 8) return fail(EKFSLAM_ERR_INVALID, "delete_features supports n_max <= 4096");
    if (int r = ensure_scratch(c, (size_t)nb * v.N)) return r;
    CK(cudaMemcpyAsync(c->pin, del, (size_t)nb * v.N, cudaMemcpyHostToDevice, c->stream));
    launch_delete_features(c, b0, nb, (const uint8_t*)c->pin);
    LAUNCHED();
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

// ---- closed loop: detection list, map management, synthetic world ------------------------------
static int ensure_det(ekfslam_ctx* c, int K) {
    if (K <= 0 || K > 1024) return fail(EKFSLAM_ERR_INVALID, "K must be in [1, 1024]");
    if (c->det_uv && c->det_K == K) return EKFSLAM_OK;
    CK(cudaStreamSynchronize(c->stream));
    if (c->det_uv) { cudaFree(c->det_uv); cudaFree(c->det_tag); c->det_uv = nullptr; c->det_tag = nullptr; }
    const size_t BK = (size_t)c->v.B * K;
    CK(cudaMalloc((void**)&c->det_uv, sizeof(double) * 2 * BK));
    CK(cudaMalloc((void**)&c->det_tag, sizeof(int32_t) * BK));
    CK(cudaMemsetAsync(c->det_uv, 0, sizeof(double) * 2 * BK, c->stream));
    CK(cudaMemsetAsync(c->det_tag, 0xff, sizeof(int32_t) * BK, c->stream));
    CK(cudaMemsetAsync(c->det_n, 0, sizeof(int32_t) * c->v.B, c->stream));
    c->det_K = K;
    return EKFSLAM_OK;
}

int ekfslam_upload_detections(ekfslam_ctx* c, int b0, int nb, int K, const double* uv, const int32_t* tag,
                              const int32_t* n) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    if (!uv || !n) return fail(EKFSLAM_ERR_INVALID, "uv / n is null");
    for (int i = 0; i < nb; ++i)
        if (n[i] < 0 || n[i] > K) return fail(EKFSLAM_ERR_INVALID, "n out of [0, K]");
    if (int r = ensure_det(c, K)) return r;
    CK(cudaMemcpyAsync(c->det_uv + 2 * (size_t)b0 * K, uv, sizeof(double) * 2 * nb * K, cudaMemcpyHostToDevice, c->stream));
    if (tag) CK(cudaMemcpyAsync(c->det_tag + (size_t)b0 * K, tag, sizeof(int32_t) * nb * K, cudaMemcpyHostToDevice, c->stream));
    else CK(cudaMemsetAsync(c->det_tag + (size_t)b0 * K, 0xff, sizeof(int32_t) * nb * K, c->stream));
    CK(cudaMemcpyAsync(c->det_n + b0, n, sizeof(int32_t) * nb, cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

int ekfslam_download_detections(ekfslam_ctx* c, int b0, int nb, int K, double* uv, int32_t* tag, int32_t* n) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    if (!c->det_uv || K != c->det_K) return fail(EKFSLAM_ERR_STATE, "no detection list of this K on the device");
    if (uv) CK(cudaMemcpyAsync(uv, c->det_uv + 2 * (size_t)b0 * K, sizeof(double) * 2 * nb * K, cudaMemcpyDeviceToHost, c->stream));
    if (tag) CK(cudaMemcpyAsync(tag, c->det_tag + (size_t)b0 * K, sizeof(int32_t) * nb * K, cudaMemcpyDeviceToHost, c->stream));
    if (n) CK(cudaMemcpyAsync(n, c->det_n + b0, sizeof(int32_t) * nb, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

int ekfslam_upload_feature_meta(ekfslam_ctx* c, int b0, int nb, const int32_t* counters, const int32_t* tag) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    DevView& v = c->v;
    const size_t o = (size_t)b0 * v.N, cnt = (size_t)nb * v.N;
    if (counters) CK(cudaMemcpyAsync(v.counters + 2 * o, counters, sizeof(int32_t) * 2 * cnt, cudaMemcpyHostToDevice, c->stream));
    if (tag) CK(cudaMemcpyAsync(v.tag + o, tag, sizeof(int32_t) * cnt, cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

int ekfslam_download_feature_tags(ekfslam_ctx* c, int b0, int nb, int32_t* tag) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    if (!tag) return fail(EKFSLAM_ERR_INVALID, "tag is null");
    CK(cudaMemcpyAsync(tag, c->v.tag + (size_t)b0 * c->v.N, sizeof(int32_t) * (size_t)nb * c->v.N, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

int ekfslam_download_candidates(ekfslam_ctx* c, int b0, int nb, double* zc, uint8_t* fl) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    DevView& v = c->v;
    const size_t o = (size_t)b0 * v.N, cnt = (size_t)nb * v.N;
    if (zc) CK(cudaMemcpyAsync(zc, v.zc + 2 * o, sizeof(double) * 2 * cnt, cudaMemcpyDeviceToHost, c->stream));
    if (fl) CK(cudaMemcpyAsync(fl, v.mflags + o, cnt, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

int ekfslam_map_management(ekfslam_ctx* c, int min_number_of_features_in_image) {
    NEED_CTX(c);
    DevView& v = c->v;
    if (min_number_of_features_in_image < 0) return fail(EKFSLAM_ERR_INVALID, "min_number_of_features_in_image < 0");
    if (c->own_zc) return fail(EKFSLAM_ERR_STATE, "frame buffers are bound to caller memory (ekfslam_unbind_frame first)");
    if (!c->det_uv) return fail(EKFSLAM_ERR_STATE, "map_management: no detection list (ekfslam_upload_detections / ekfslam_world_detect)");
    if (v.nmax > 512 * 8) return fail(EKFSLAM_ERR_INVALID, "map_management supports n_max <= 4096");
    launch_mm_plan(c, min_number_of_features_in_image);           // deletion list, measured, quota     (:7-14, :27-35)
    launch_delete_features(c, 0, v.B, c->mm_del);                  // delete_a_feature.m                 (:7)
    launch_begin_frame(c);                                         // update_features_info.m             (:17)
    launch_id2cart(c, 0.1, -1, nullptr);                           // inversedepth_2_cartesian.m         (:22)
    const int K = c->det_K < 50 ? c->det_K : 50;
    for (int j = 0; j < K; ++j)                                    // initialize_features                (:27-35)
        launch_add_features(c, 0, v.B, c->det_uv + 2 * (size_t)j, 2 * c->det_K, nullptr, c->mm_quota, j,
                            c->det_tag + j, c->det_K, c->prm.std_z, 1.0, 1.0);
    LAUNCHED();
    return EKFSLAM_OK;
}

int ekfslam_world_upload(ekfslam_ctx* c, int M, int T, const double* points, const double* poses,
                         const ekfslam_world_params* wp) {
    NEED_CTX(c);
    if (!points || !poses || !wp) return fail(EKFSLAM_ERR_INVALID, "points / poses / params is null");
    if (M <= 0 || M > 2048 || T < 0) return fail(EKFSLAM_ERR_INVALID, "M must be in [1, 2048] and T >= 0");
    if (wp->flaky_mod <= 0) return fail(EKFSLAM_ERR_INVALID, "flaky_mod must be positive");
    CK(cudaStreamSynchronize(c->stream));
    if (c->world_points) { cudaFree(c->world_points); cudaFree(c->world_poses); c->world_points = nullptr; c->world_poses = nullptr; }
    const size_t np_ = (size_t)c->v.B * M * 3, nq = (size_t)(T + 1) * c->v.B * 7;
    CK(cudaMalloc((void**)&c->world_points, sizeof(double) * np_));
    CK(cudaMalloc((void**)&c->world_poses, sizeof(double) * nq));
    CK(cudaMemcpyAsync(c->world_points, points, sizeof(double) * np_, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->world_poses, poses, sizeof(double) * nq, cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    DevWorld& w = c->world;
    w.M = M; w.T = T; w.points = c->world_points; w.poses = c->world_poses;
    w.seed = wp->seed; w.b_offset = wp->b_offset; w.flaky_mod = wp->flaky_mod;
    w.noise_px = wp->noise_px; w.gross_px = wp->gross_px; w.p_outlier = wp->p_outlier; w.p_flaky = wp->p_flaky;
    w.band = wp->band_px;
    return EKFSLAM_OK;
}

int ekfslam_world_candidates(ekfslam_ctx* c, int t) {
    NEED_CTX(c);
    if (!c->world_points) return fail(EKFSLAM_ERR_STATE, "no world uploaded (ekfslam_world_upload)");
    if (t < 0 || t > c->world.T) return fail(EKFSLAM_ERR_INVALID, "frame index out of [0, T]");
    if (c->own_zc) return fail(EKFSLAM_ERR_STATE, "frame buffers are bound to caller memory (ekfslam_unbind_frame first)");
    launch_world_candidates(c, t);
    LAUNCHED();
    return EKFSLAM_OK;
}

int ekfslam_world_uniforms(ekfslam_ctx* c, int t, int n_u) {
    NEED_CTX(c);
    if (!c->world_points) return fail(EKFSLAM_ERR_STATE, "no world uploaded (ekfslam_world_upload)");
    if (n_u <= 0) return fail(EKFSLAM_ERR_INVALID, "n_u <= 0");
    if (c->own_zc) return fail(EKFSLAM_ERR_STATE, "frame buffers are bound to caller memory (ekfslam_unbind_frame first)");
    if (int r = ensure_u(c, n_u)) return r;
    c->v.n_u = n_u;
    launch_world_uniforms(c, t);
    LAUNCHED();
    return EKFSLAM_OK;
}

int ekfslam_download_uniforms(ekfslam_ctx* c, int b0, int nb, double* u, int n_u) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    if (!u || n_u != c->v.n_u || n_u <= 0) return fail(EKFSLAM_ERR_INVALID, "u is null or n_u differs from the resident stream");
    CK(cudaMemcpyAsync(u, c->v.u + (size_t)b0 * n_u, sizeof(double) * (size_t)nb * n_u, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

int ekfslam_world_detect(ekfslam_ctx* c, int t, int K) {
    NEED_CTX(c);
    if (!c->world_points) return fail(EKFSLAM_ERR_STATE, "no world uploaded (ekfslam_world_upload)");
    if (t < 0 || t > c->world.T) return fail(EKFSLAM_ERR_INVALID, "frame index out of [0, T]");
    if (int r = ensure_det(c, K)) return r;
    launch_world_detect(c, t);
    LAUNCHED();
    return EKFSLAM_OK;
}

// ---- scoring against the resident ground truth (k_eval.cu) -------------------------------------
// shared memory of the scoring launch: two doubles and one byte per feature slot
static int eval_fits(const ekfslam_ctx* c) {
    if ((size_t)c->v.N * 17 > 200 * 1024) return fail(EKFSLAM_ERR_INVALID, "evaluation supports N_max <= 12000");
    return EKFSLAM_OK;
}

int ekfslam_evaluate(ekfslam_ctx* c, int t) {
    NEED_CTX(c);
    if (!c->world_points) return fail(EKFSLAM_ERR_STATE, "evaluate: no world uploaded (ekfslam_world_upload)");
    if (t < 0 || t > c->world.T) return fail(EKFSLAM_ERR_INVALID, "frame index out of [0, T]");
    if (int r = eval_fits(c)) return r;
    DevEval& e = c->ev;
    if (!e.rec) {   // first evaluation: the buffers are allocated here, so a context that never evaluates holds none
        const size_t B = (size_t)c->v.B, BN = B * c->v.N;
        cudaError_t er = cudaMalloc((void**)&e.rec, sizeof(ekfslam_eval) * B);
        if (er == cudaSuccess) er = cudaMalloc((void**)&e.tot, sizeof(ekfslam_eval) * B);
        if (er == cudaSuccess) er = cudaMalloc((void**)&e.ferr, sizeof(double) * 3 * BN);
        if (er == cudaSuccess) er = cudaMalloc((void**)&e.fnees, sizeof(double) * BN);
        if (er != cudaSuccess) {   // all or nothing: e.rec != null means every scoring buffer exists
            for (void* q : {(void*)e.rec, (void*)e.tot, (void*)e.ferr, (void*)e.fnees}) if (q) cudaFree(q);
            e.rec = e.tot = nullptr; e.ferr = e.fnees = nullptr;
            cudaGetLastError();   // an allocation failure is reported here, not by the next launch check
            return fail(er == cudaErrorMemoryAllocation ? EKFSLAM_ERR_NOMEM : EKFSLAM_ERR_CUDA,
                        std::string("evaluation buffers: ") + cudaGetErrorString(er));
        }
        CK(cudaMemsetAsync(e.tot, 0, sizeof(ekfslam_eval) * B, c->stream));
        c->bytes += (int64_t)(2 * sizeof(ekfslam_eval) * B + sizeof(double) * 4 * BN);
    }
    launch_eval(c, 0, t, 0, c->v.B);
    LAUNCHED();
    return EKFSLAM_OK;
}

int ekfslam_download_eval(ekfslam_ctx* c, int b0, int nb, int totals, ekfslam_eval* rec, double* feat_err,
                          double* feat_nees) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    if (!rec) return fail(EKFSLAM_ERR_INVALID, "rec is null");
    if (totals && (feat_err || feat_nees))
        return fail(EKFSLAM_ERR_INVALID, "per-feature outputs exist for the last frame only (totals == 0)");
    const DevEval& e = c->ev;
    if (!e.rec) return fail(EKFSLAM_ERR_STATE, "nothing evaluated yet (ekfslam_evaluate)");
    const size_t o = (size_t)b0 * c->v.N, cnt = (size_t)nb * c->v.N;
    CK(cudaMemcpyAsync(rec, (totals ? e.tot : e.rec) + b0, sizeof(ekfslam_eval) * nb, cudaMemcpyDeviceToHost, c->stream));
    if (feat_err) CK(cudaMemcpyAsync(feat_err, e.ferr + 3 * o, sizeof(double) * 3 * cnt, cudaMemcpyDeviceToHost, c->stream));
    if (feat_nees) CK(cudaMemcpyAsync(feat_nees, e.fnees + o, sizeof(double) * cnt, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

int ekfslam_reset_eval(ekfslam_ctx* c) {
    NEED_CTX(c);
    if (c->ev.tot) CK(cudaMemsetAsync(c->ev.tot, 0, sizeof(ekfslam_eval) * c->v.B, c->stream));
    return EKFSLAM_OK;
}

int ekfslam_map_cartesian(ekfslam_ctx* c, int b0, int nb, double* p, double* cov) {
    NEED_CTX(c);
    if (check_range(c, b0, nb)) return EKFSLAM_ERR_INVALID;
    DevEval& e = c->ev;
    const size_t BN = (size_t)c->v.B * c->v.N;
    if (!e.mp) {
        cudaError_t er = cudaMalloc((void**)&e.mp, sizeof(double) * 3 * BN);
        if (er == cudaSuccess) er = cudaMalloc((void**)&e.mc, sizeof(double) * 6 * BN);
        if (er != cudaSuccess) {
            if (e.mp) cudaFree(e.mp);
            e.mp = nullptr;
            cudaGetLastError();
            return fail(er == cudaErrorMemoryAllocation ? EKFSLAM_ERR_NOMEM : EKFSLAM_ERR_CUDA,
                        std::string("map export buffers: ") + cudaGetErrorString(er));
        }
        c->bytes += (int64_t)(sizeof(double) * 9 * BN);
    }
    launch_eval(c, 1, 0, b0, nb);
    LAUNCHED();
    const size_t o = (size_t)b0 * c->v.N, cnt = (size_t)nb * c->v.N;
    if (p) CK(cudaMemcpyAsync(p, e.mp + 3 * o, sizeof(double) * 3 * cnt, cudaMemcpyDeviceToHost, c->stream));
    if (cov) CK(cudaMemcpyAsync(cov, e.mc + 6 * o, sizeof(double) * 6 * cnt, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return EKFSLAM_OK;
}

void* ekfslam_device_ptr(ekfslam_ctx* c, const char* name) {
    if (!c || !name) return nullptr;
    DevView& v = c->v;
    struct { const char* n; void* p; } tab[] = {
        {"x", v.x}, {"xp", v.xp}, {"P", v.P}, {"G", v.G}, {"W", v.W}, {"h", v.h}, {"Hc", v.Hc}, {"S", v.S},
        {"z", v.z}, {"zc", v.zc}, {"flags", v.flags}, {"mflags", v.mflags}, {"u", v.u}, {"stats", v.stats},
        {"Sb", v.Sb}, {"Li", v.Li}, {"yv", v.yv}};
    for (auto& e : tab)
        if (!strcmp(e.n, name)) return e.p;
    return nullptr;
}

}  // extern "C"
