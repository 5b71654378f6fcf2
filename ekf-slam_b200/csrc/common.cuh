// Internal definitions shared by the kernels and the C ABI (not installed).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <mutex>
#include "../../include/ekfslam.h"

#define EKF_XV 13        // camera state size, mc/fv.m:3-6
#define EKF_HC 13        // compact Jacobian columns: 7 (r,q) + 6 (feature block)
#define EKF_HSTRIDE 26   // doubles per feature in Hc: 2 rows x 13

struct DevCam {
    double k1, k2, Cx, Cy, f, dx, dy;
    double fku, fkv;  // f*(1/dx), f*(1/dy) in the reference's evaluation order
    double nRows, nCols;
};

// Everything a kernel needs; passed by value.
struct DevView {
    int B, N, nmax, ld;   // ld = leading dimension (doubles) of x rows, P rows, G/W rows
    int kmax;             // 2*N
    int n_u;              // uniforms per filter
    double* x;            // [B][ld]      x_k_k
    double* xp;           // [B][ld]      x_k_km1
    double* P;            // [B][nmax][ld] covariance (single buffer, updated in place)
    double* G;            // [B][kmax][ld] rows 2i,2i+1 = H_i * P
    double* W;            // [B][ncb][wrows][EKF_WPAD] W = inv(L) * G_sel, stored by 64-column panels (see w_at)
    long long wstride;    // doubles per filter in W = ncb * wrows * EKF_WPAD, ncb = ceil(ld / 64)
    int wrows;            // rows per panel of W (= kmax)
    double* Sb;           // [B][kmax][kmax] stacked innovation covariance / its Cholesky factor
    double* Li;           // [B][kmax][kmax] inverse of the Cholesky factor
    double* yv;           // [B][kmax]     inv(L)*(z-h)
    double* jn;           // [B][16]       normalisation Jacobian the covariance downdate applies
    double* jnt;          // [B][16]       normJac(q+) of the update being computed
    double* cv;           // [B][kmax]     inv(S)*(z-h) = inv(L)' * yv
    double* h;            // [B][N][2]
    double* Hc;           // [B][N][26]
    double* S;            // [B][N][4]
    double* z;            // [B][N][2]
    double* zc;           // [B][N][2]  candidates for the gate
    double* u;            // [B][n_u]
    uint8_t* ftype;       // [B][N]
    uint8_t* flags;       // [B][N]
    uint8_t* mflags;      // [B][N]  staged match / candidate flags of the current frame
    int32_t* foff;        // [B][N]
    int32_t* nstate;      // [B]
    int32_t* nfeat;       // [B]
    int32_t* counters;    // [B][N][2]
    int32_t* tag;         // [B][N]   feature identity (stand-in for features_info(i).feature_when_initialized)
    int32_t* sel;         // [B][N]   selected feature list of the running update
    int32_t* ksel;        // [B]      number of selected features
    int32_t* ktot;        // [B]      rows of W the covariance downdate has to apply
    int32_t* kmaxdev;     // [1]      max over the filters of the stacked rows of the running update (k_upd_S)
    int32_t* nhyp_tab;    // [(N+1)(N+2)/2] adaptive hypothesis count, host libm (see abi.cu)
    ekfslam_stats* stats; // [B]
};

// The synthetic world of the closed loop (k_map.cu): resident world points, camera trajectory, noise model.
struct DevWorld {
    int M, T;                    // world points per filter, frames (poses 0..T)
    const double* points;        // [B][M][3]
    const double* poses;         // [T+1][B][7]  r (3), q (4)
    unsigned long long seed;
    int b_offset;                // filter index offset of this context inside a larger batch (sharding)
    double noise_px, gross_px, p_outlier, p_flaky;
    int flaky_mod;
    double band;                 // excluded image band for new features
};

// per-kernel timing (ekfslam_enable_timing): every launch is bracketed by an event pair
enum {
    KT_BEGIN_FRAME = 0, KT_PREDICT, KT_FEATURES, KT_HP, KT_INNOV, KT_RANSAC, KT_UPD_S, KT_CHOL, KT_W, KT_DOWNDATE_HI,
    KT_DOWNDATE, KT_SYMMETRIZE, KT_ADD_FEATURES, KT_WFIX, KT_W_HI, KT_CHOL_HI, KT_UPD_S_HI, KT_HP_RESCUE, KT_WORLD, KT_EVAL, KT_COUNT
};
struct KTimer;

// scoring against the resident ground truth (k_eval.cu); allocated on the first ekfslam_evaluate /
// ekfslam_map_cartesian, so a context that never evaluates holds none of it
struct DevEval {
    ekfslam_eval* rec;    // [B]        record of the last evaluated frame
    ekfslam_eval* tot;    // [B]        running totals
    double* ferr;         // [B][N][3]  e_f of the last evaluated frame
    double* fnees;        // [B][N]     nees_f of the last evaluated frame
    double* mp;           // [B][N][3]  map export: p
    double* mc;           // [B][N][6]  map export: C_f packed (xx, yx, yy, zx, zy, zz)
};

struct ekfslam_ctx {
    int device;
    KTimer* timer;
    DevView v;
    DevCam cam;
    ekfslam_params prm;
    cudaStream_t own_stream;
    cudaStream_t stream;
    int64_t bytes;
    int64_t launches;
    int stage;  // call-order tracking
    // ekfslam_step_host overlaps its PCIe copies with the step: inputs go up on copy_stream while prediction and the
    // measurement model run (first needed by the matcher gate), x / flags / stats come down while the last covariance
    // downdate (which only touches P) is still running.
    cudaStream_t copy_stream;
    // side stream for launches that would otherwise run nearly alone on the GPU (the large resident-Cholesky variant:
    // a handful of filters, one CTA each, ~0.15 ms of latency) - forked / joined with ev_fork / ev_join
    cudaStream_t aux_stream, aux2_stream;
    cudaEvent_t ev_fork, ev_join, ev_join2;
    cudaEvent_t ev_in, ev_out, ev_main;
    int wait_inputs;     // ekfslam_step: make the stream wait for ev_in before the first kernel that reads zc / mflags / u
    int arm_out;         // launch_update(HI): record ev_out before the covariance downdate; cleared when recorded
    // pinned staging
    void* pin;
    size_t pin_bytes;
    int u_cap;
    void* step_graph;    // captured CUDA graph of the filter step (ekfslam_step_graph), opaque here
    int sm_count;        // multiprocessors of THIS context's device (persistent-kernel grid sizes)
    int32_t* kmax_host;  // pinned: host copy of *v.kmaxdev (lock-step Cholesky bounds its launch loops with it)
    // closed loop: synthetic world + detection list + map-management scratch (k_map.cu)
    DevWorld world;
    double* world_points; double* world_poses;
    double* det_uv; int32_t* det_tag; int32_t* det_n; int det_K;   // [B][K][2], [B][K], [B]
    uint8_t* mm_del; int32_t* mm_quota;                             // [B][N], [B]
    // the context's own frame buffers while caller-owned ones are bound (ekfslam_bind_frame)
    double* own_zc; uint8_t* own_mflags; double* own_u; int own_n_u;
    DevEval ev;
};

// W is stored panel-major: element (row t, column c) of a filter lives at ((c / 64) * wrows + t) * EKF_WPAD + c % 64.
// A K-chunk of a 64-column panel ([rows][68] doubles, the padded shared-memory layout of the tensor-core
// kernels) is then ONE contiguous range, i.e. one bulk copy per panel and stage instead of one per row.
#define EKF_WPAD 68
__host__ __device__ __forceinline__ size_t w_at(int wrows, int t, int c) {
    return ((size_t)(c >> 6) * wrows + t) * EKF_WPAD + (c & 63);
}

#define EKF_TRI(nic, s) (((nic) * ((nic) + 1)) / 2 + (s))

// The update's Cholesky runs lock-step over all filters (one launch per phase, k_chol_big.cu) for few filters with a
// large stacked innovation; otherwise one block per filter.  The lock-step path reads the batch's largest stacked size
// back to the host, so a step that takes it cannot be captured in a CUDA graph (ekfslam_step_graph).
inline bool chol_lockstep(const DevView& v) { return v.B < 128 && v.kmax >= 256; }

// one process-wide lock for the per-device function-attribute high-water marks (ENSURE_DYN_SMEM)
inline std::mutex& ekf_attr_mutex() { static std::mutex m; return m; }

// timing hooks (abi.cu): no-ops unless timing is enabled
void kt_begin(ekfslam_ctx* c, int slot);
void kt_end(ekfslam_ctx* c, int slot);
struct KScope {
    ekfslam_ctx* c; int slot;
    KScope(ekfslam_ctx* c_, int s_) : c(c_), slot(s_) { if (c->timer) kt_begin(c, slot); }
    ~KScope() { if (c->timer) kt_end(c, slot); c->launches++; }
};

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is a per-DEVICE setting: a process that drives several GPUs (one
// context per GPU) must raise it on each of them.  The high-water mark is kept per call site and device; NEED_CTX has
// made `dev` the current device.
#define ENSURE_DYN_SMEM(func, bytes, dev)                                                                    \
    do {                                                                                                     \
        static size_t _hw[64];                                                                               \
        const size_t _b = (size_t)(bytes);                                                                   \
        const int _d = (dev) & 63;                                                                           \
        if (_b > 48 * 1024) {                                                                                \
            std::lock_guard<std::mutex> _g(ekf_attr_mutex());   /* host threads driving different contexts */ \
            if (_b > _hw[_d]) {                                                                              \
                cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)_b);            \
                _hw[_d] = _b;                                                                                \
            }                                                                                                \
        }                                                                                                    \
    } while (0)

// launchers (defined in the kernel .cu files)
void launch_begin_frame(ekfslam_ctx* c);
void launch_predict(ekfslam_ctx* c);
void launch_features(ekfslam_ctx* c, int which, int parts);  // parts: 1 = h, 2 = H, 3 = both
void launch_hp(ekfslam_ctx* c, int need, int forbid, int slot = KT_HP);  // G rows for features with (flags&need)==need && !(flags&forbid)
void launch_innov_gather(ekfslam_ctx* c, int mode);          // S_i from 13x13 gathers of P (no G rows): 0 = S_i + R stored, 3 = rescue gate
void launch_innov(ekfslam_ctx* c, int mode);           // matcher gate (1) / explicit matches (2)
void launch_symmetrize(ekfslam_ctx* c, int b0, int nb);
void launch_ransac(ekfslam_ctx* c);
void launch_update(ekfslam_ctx* c, int mask, int which_prior, int flags = 0);
void launch_downdate(ekfslam_ctx* c, int slot);
void launch_chol_blocked64(ekfslam_ctx* c, int kact);   // k_chol_big.cu: S = L L', X = inv(L) for few filters with large k
void launch_reset_filters(ekfslam_ctx* c, int b0, int nb, const double* d_xv, const double* d_Pxv);
void launch_id2cart(ekfslam_ctx* c, double threshold, int force_index, int32_t* d_conv);
void launch_delete_features(ekfslam_ctx* c, int b0, int nb, const uint8_t* d_del);
// one feature per filter from uvd[lb * uvd_stride .. +1]; add (mask) / quota (add iff j < quota[b]) / tag_src may be null
void launch_add_features(ekfslam_ctx* c, int b0, int nb, const double* d_uvd, int uvd_stride, const uint8_t* d_add,
                         const int32_t* d_quota, int j, const int32_t* d_tag, int tag_stride,
                         double std_pxl, double rho0, double std_rho);
void launch_world_candidates(ekfslam_ctx* c, int t);
void launch_world_detect(ekfslam_ctx* c, int t);
void launch_world_uniforms(ekfslam_ctx* c, int t);
void launch_mm_plan(ekfslam_ctx* c, int min_features);
// mode 0: score filters [b0, b0+nb) against frame t of the world; mode 1: map export of filters [b0, b0+nb)
void launch_eval(ekfslam_ctx* c, int mode, int t, int b0, int nb);
