/*
 * ekfslam.h — C ABI of libekfslam.so: the B200-native (sm_100a, fp64) batched
 * implementation of the per-frame filter step of Civera-style monocular EKF-SLAM with
 * 1-point RANSAC (reference: diwakar-vsingh/EKF-SLAM, matlab_code/mono_slam.m:56-74).
 *
 * The reference has no FFI of its own (it is interpreted MATLAB); each entry point
 * below names the reference function(s) whose arithmetic it replaces ("mc/" =
 * matlab_code/).  A binding for this header is a ctypes stub (ekf-slam_b200/_lib.py)
 * or the Octave/MATLAB MEX gateway (mex/ekfslam_mex.c) — see INTEGRATION.md.
 *
 * Conventions
 *  - plain C types only; every call returns 0 or a negative ekfslam_status and
 *    records a message retrievable with ekfslam_last_error() (thread-local).
 *  - the caller owns host memory, the context owns device memory.  A context is
 *    bound to one CUDA device and one stream; it is not re-entrant.
 *  - B independent filters are stored structure-of-arrays.  Filter b has state
 *    dimension n[b] <= n_max and nfeat[b] <= N_max features.
 *  - state layout (mc/fv.m:3-6, mc/predict_camera_measurements.m:4-21):
 *    x = [r(3) q(4, scalar first) v(3) w(3) | feature blocks in features_info order];
 *    inverse-depth block [x y z theta phi rho], Cartesian block [X Y Z].
 *  - host matrices are column-major doubles (MATLAB/Octave layout) with leading
 *    dimension n_max; covariances are symmetric, so row-major callers need no transpose.
 *  - indices are 0-based.
 */
#ifndef EKFSLAM_H
#define EKFSLAM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ekfslam_ctx ekfslam_ctx;

typedef enum {
    EKFSLAM_OK = 0,
    EKFSLAM_ERR_INVALID = -1,  /* bad argument / shape                               */
    EKFSLAM_ERR_CUDA = -2,     /* CUDA runtime error (message has the cudaError name) */
    EKFSLAM_ERR_NOMEM = -3,    /* host or device allocation failed                    */
    EKFSLAM_ERR_STATE = -4,    /* call order violated (e.g. update before measure)    */
    EKFSLAM_ERR_NODEVICE = -5  /* no CUDA device: there is NO CPU fallback            */
} ekfslam_status;

/* feature types, mc/add_feature_to_info_vector.m:21 ('inversedepth') and
 * mc/inversedepth_2_cartesian.m:48 ('cartesian') */
enum { EKFSLAM_FEAT_NONE = 0, EKFSLAM_FEAT_INVERSEDEPTH = 1, EKFSLAM_FEAT_CARTESIAN = 2 };

/* per-feature flag bits (one byte per feature) — the boolean / "is empty" fields of
 * features_info, mc/add_feature_to_info_vector.m:23-29 */
enum {
    EKFSLAM_F_HAS_H = 1,  /* features_info(i).h non-empty (predicted this frame)          */
    EKFSLAM_F_HAS_Z = 2,  /* features_info(i).z non-empty (a match was found)             */
    EKFSLAM_F_IC = 4,     /* individually_compatible                                      */
    EKFSLAM_F_LI = 8,     /* low_innovation_inlier                                        */
    EKFSLAM_F_HI = 16,    /* high_innovation_inlier                                       */
    EKFSLAM_F_CAND = 32   /* a candidate pixel was supplied to the synthetic matcher gate */
};

/* camera, mc/initialize_cam.m:12-25 */
typedef struct {
    double k1, k2;   /* radial distortion                */
    double Cx, Cy;   /* principal point [px]             */
    double f;        /* focal length [mm]                */
    double dx, dy;   /* pixel size [mm]                  */
    int32_t nRows, nCols;
} ekfslam_camera;

/* filter tuning, mc/mono_slam.m:29-32 and mc/ransac_hypotheses.m:3,9 */
typedef struct {
    double std_a;        /* linear acceleration noise  (0.007)                      */
    double std_alpha;    /* angular acceleration noise (0.007)                      */
    double std_z;        /* image noise = RANSAC threshold (1.0)                    */
    double delta_t;      /* mc/predict_state_and_covariance.m:5 (1)                 */
    double chi2_gate;    /* mc/rescue_hi_inliers.m:3 (5.9915)                       */
    double p_spurious_free; /* mc/ransac_hypotheses.m:3 (0.99)                      */
    int32_t max_hyp;     /* mc/ransac_hypotheses.m:9 (1000)                         */
    int32_t fixed_hyp;   /* 0 = the reference's adaptive rule; >0 = run exactly this
                            many hypotheses per frame (BASELINE configs 2/5)        */
} ekfslam_params;

/* per-filter step statistics (the values NCCL gathers in the multi-GPU driver) */
typedef struct {
    int32_t n_ic;          /* individually compatible matches                         */
    int32_t ransac_iters;  /* hypotheses drawn  (loop iterations of ransac_hypotheses) */
    int32_t ransac_scored; /* distinct hypotheses actually scored                      */
    int32_t max_support;   /* support of the winning hypothesis                        */
    int32_t n_li;          /* low-innovation inliers used in the first update          */
    int32_t n_hi;          /* high-innovation inliers used in the second update        */
    int32_t status;        /* bit0: uniform stream exhausted; bit1: S not SPD;
                              bit2: add_features found no room (n_max / N_max)         */
    int32_t reserved;
} ekfslam_stats;

const char* ekfslam_last_error(void);
int ekfslam_version(void);
/* number of usable CUDA devices (0 => every other call fails with ERR_NODEVICE) */
int ekfslam_device_count(void);

void ekfslam_default_camera(ekfslam_camera* cam);  /* mc/initialize_cam.m:3-10 */
void ekfslam_default_params(ekfslam_params* p);    /* the constants listed above */

/* ---- context ------------------------------------------------------------- */
int ekfslam_create(ekfslam_ctx** out, int device, int B, int N_max, int n_max);
int ekfslam_destroy(ekfslam_ctx* ctx);
/* use the caller's cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream);
 * NULL restores the context's own stream */
int ekfslam_set_stream(ekfslam_ctx* ctx, void* cuda_stream);
int ekfslam_set_camera(ekfslam_ctx* ctx, const ekfslam_camera* cam);
int ekfslam_set_params(ekfslam_ctx* ctx, const ekfslam_params* p);
int ekfslam_synchronize(ekfslam_ctx* ctx);
int ekfslam_dims(const ekfslam_ctx* ctx, int* B, int* N_max, int* n_max, int* ld);
/* bytes of device memory the context holds */
int64_t ekfslam_device_bytes(const ekfslam_ctx* ctx);
/* kernels launched by this context since creation (bench.py's gpu_launches) */
int64_t ekfslam_launch_count(const ekfslam_ctx* ctx);

/* ---- filter struct  <->  device (mc/ekf_filter.m:37-46) -------------------- */
/* which: 0 = (x_k_k, p_k_k), 1 = (x_k_km1, p_k_km1).  x: [nb][n_max]; P: [nb][n_max*n_max]
 * column-major, ld n_max; nstate: [nb].  P or x may be NULL to skip.  The device keeps P exactly
 * symmetric: on upload its lower triangle is mirrored into the upper one (a host P that is
 * symmetric only to rounding, e.g. J*P*J', changes by <= 1 ulp).  Upload nstate (or the feature
 * types) before or together with P. */
int ekfslam_upload_state(ekfslam_ctx* ctx, int b0, int nb, int which, const double* x,
                         const double* P, const int32_t* nstate);
int ekfslam_download_state(ekfslam_ctx* ctx, int b0, int nb, int which, double* x, double* P,
                           int32_t* nstate);

/* ---- features_info <-> device (mc/add_feature_to_info_vector.m:7-32) ------- */
/* type: [nb][N_max] EKFSLAM_FEAT_*; nfeat: [nb].  Resets all per-frame fields. */
int ekfslam_upload_feature_types(ekfslam_ctx* ctx, int b0, int nb, const uint8_t* type,
                                 const int32_t* nfeat);
/* explicit matches (what mc/matching.m:52-53 writes): z [nb][N_max][2]; flags [nb][N_max]
 * with bits HAS_Z / IC honoured (other bits ignored). */
int ekfslam_upload_matches(ekfslam_ctx* ctx, int b0, int nb, const double* z, const uint8_t* flags);
/* candidate pixels for the synthetic matcher gate: zc [nb][N_max][2], has [nb][N_max] */
int ekfslam_upload_candidates(ekfslam_ctx* ctx, int b0, int nb, const double* zc, const uint8_t* has);
/* uniform stream replacing rand(1) of mc/select_random_match.m:12: u [nb][n_u] */
int ekfslam_upload_uniforms(ekfslam_ctx* ctx, int b0, int nb, const double* u, int n_u);
/* any pointer may be NULL.  h [nb][N_max][2]; Hc [nb][N_max][2][13] compact Jacobian
 * (columns 0-6 = d/d(r,q); 7-12 = d/d(feature block), 3 valid for Cartesian);
 * S [nb][N_max][4]; z [nb][N_max][2]; flags [nb][N_max]; offs [nb][N_max] 0-based state
 * offset of each feature; counters [nb][N_max][2] = times_predicted, times_measured */
int ekfslam_download_features(ekfslam_ctx* ctx, int b0, int nb, double* h, double* Hc, double* S,
                              double* z, uint8_t* flags, int32_t* offs, int32_t* counters);
/* the inverse of ekfslam_download_features for the fields a stage reads (NULL = keep) */
int ekfslam_upload_features(ekfslam_ctx* ctx, int b0, int nb, const double* h, const double* Hc,
                            const double* S, const double* z, const uint8_t* flags);
/* the map layout: type [nb][N_max] EKFSLAM_FEAT_*, nfeat [nb] (either may be NULL) */
int ekfslam_download_feature_types(ekfslam_ctx* ctx, int b0, int nb, uint8_t* type, int32_t* nfeat);
int ekfslam_download_stats(ekfslam_ctx* ctx, int b0, int nb, ekfslam_stats* stats);

/* ---- the filter step, stage by stage (all B filters, stream-ordered) ------- */
/* mc/update_features_info.m:4-18: bump counters, clear per-frame flags/h/z/H/S */
int ekfslam_begin_frame(ekfslam_ctx* ctx);
/* mc/ekf_prediction.m:3 -> mc/predict_state_and_covariance.m:3-27 (fv, dfv_by_dxv, func_Q).
 * (x_k_k,p_k_k) -> (x_k_km1,p_k_km1).  The covariance is updated IN PLACE: only its first
 * 13 rows/columns change, so after this call p_k_k is no longer available on the device. */
int ekfslam_predict(ekfslam_ctx* ctx);
/* mc/search_IC_matches.m:4-10 = mc/predict_camera_measurements.m:4-28 (hi_inverse_depth,
 * hi_cartesian, hu, distort_fm) + mc/calculate_derivatives.m:3-28 (calculate_Hi_*) +
 * S_i = H_i P H_i' + R_i.  which: 1 = at (x_k_km1,p_k_km1), 0 = at (x_k_k,p_k_k).
 * S_i only needs the 13x13 block of P that H_i touches; the full rows P H_i' (2 x n per feature) are
 * built where they are consumed: per scored hypothesis inside ekfslam_ransac, per update by ekfslam_hp. */
int ekfslam_measure(ekfslam_ctx* ctx, int which);
/* the kernels of ekfslam_measure, separately callable, and the row product of the updates:
 * ekfslam_features: parts&1 = mc/predict_camera_measurements.m (h), parts&2 =
 *                   mc/calculate_derivatives.m (H, linearised at the stored h);
 * ekfslam_innovation: S_i = H_i P H_i' + R_i (mc/search_IC_matches.m:6-10) from 13x13 gathers of P;
 * ekfslam_hp:       rows 2i,2i+1 of G = H_i * P (= (P H_i')', mc/update.m:8-9) for every feature whose
 *                   flag byte f has (f & need) == need && (f & forbid) == 0.  ekfslam_update_masked /
 *                   ekfslam_update_iterated read these rows for the features they stack;
 *                   ekfslam_update_li, ekfslam_rescue (+ ekfslam_update_hi) and ekfslam_step call it
 *                   themselves for exactly the rows they need. */
int ekfslam_features(ekfslam_ctx* ctx, int which, int parts);
int ekfslam_hp(ekfslam_ctx* ctx, int need, int forbid);
int ekfslam_innovation(ekfslam_ctx* ctx);
/* gating rule of mc/matching.m:16,38 applied to the uploaded candidates:
 * all(eig(S)<100) && nu'inv(S)nu < chi2 -> z, individually_compatible */
int ekfslam_gate(ekfslam_ctx* ctx);
/* copy the explicit matches staged by ekfslam_upload_matches into features_info
 * (what mc/matching.m:52-53 writes: z and individually_compatible) */
int ekfslam_apply_matches(ekfslam_ctx* ctx);
/* mc/ransac_hypotheses.m:3-47 (select_random_match, generate_state_vector_pattern,
 * compute_hypothesis_support_fast, set_as_most_supported_hypothesis).  Needs S_i (ekfslam_measure /
 * ekfslam_innovation) and the matches; the gain P H_p' inv(S_p) of a hypothesis (:24-25) is formed on demand. */
int ekfslam_ransac(ekfslam_ctx* ctx);
/* mc/ekf_update_li_inliers.m:4-21 -> mc/update.m:3-32 (+normJac) from (x_k_km1,p_k_km1) */
int ekfslam_update_li(ekfslam_ctx* ctx);
/* mc/rescue_hi_inliers.m:3-22: h, H of every feature at x_k_k, chi2 gate of the candidates (IC && !LI) from
 * 13x13 gathers of p_k_k, then the rows H p_k_k of the rescued features (for ekfslam_update_hi) */
int ekfslam_rescue(ekfslam_ctx* ctx);
/* mc/ekf_update_hi_inliers.m:4-21 -> mc/update.m from (x_k_k,p_k_k) */
int ekfslam_update_hi(ekfslam_ctx* ctx);
/* mc/update.m:3-32 on explicit rows: for filter b the update uses the features whose flag
 * byte has any bit of `mask`; which_prior 1 = from x_k_km1, 0 = from x_k_k */
int ekfslam_update_masked(ekfslam_ctx* ctx, int mask, int which_prior);

/* EXTENSION (mc/ekf_update_iterated.m:3 calls update_iterated, which does not exist in the reference):
 * standard iterated EKF over the features whose flag byte has a bit of `mask`,
 *   x_{j+1} = x^- + K_j (z - h(x_j) - H_j (x^- - x_j)),  j = 0..n_iter-1,  x_0 = x^-,
 * h/H re-evaluated at every iterate, P from the last linearisation, then the quaternion fix-up of
 * mc/update.m:18-24.  which_prior 1: prior (x_k_km1, P), 0: prior (x_k_k, P) (x_k_km1 is overwritten). */
int ekfslam_update_iterated(ekfslam_ctx* ctx, int mask, int which_prior, int n_iter);

/* one whole filter step on resident state = mc/mono_slam.m:56-74 without takeImage:
 * begin_frame (if reset!=0), predict, measure(1), matcher (match_mode 1 = gate the staged
 * candidates, 2 = apply the staged explicit matches, 0 = flags already on the device),
 * ransac, update_li, rescue, update_hi */
int ekfslam_step(ekfslam_ctx* ctx, int reset, int match_mode);

/* ekfslam_step replayed from a captured CUDA graph (latency path: a single filter's step is ~25 small launches).
 * The graph is captured on first use and re-captured whenever anything the kernels see changes (buffers, parameters,
 * camera, reset / match_mode).  Falls back to ekfslam_step where capture is not possible (per-kernel timing enabled,
 * few filters with N_max >= 128: the lock-step Cholesky reads a size back to the host).  Stage frames with
 * ekfslam_upload_candidates / ekfslam_upload_uniforms or ekfslam_stage_frame (NOT ekfslam_bind_frame, which changes
 * the buffer addresses and forces a re-capture). */
int ekfslam_step_graph(ekfslam_ctx* ctx, int reset, int match_mode);
/* copy a device-resident frame (zc [B][N_max][2], staged flag bytes [B][N_max], uniforms [B][n_u]) into the
 * context's own frame buffers, stream-ordered */
int ekfslam_stage_frame(ekfslam_ctx* ctx, const void* d_zc, const void* d_fl, const void* d_u, int n_u);

/* the same step fed from HOST buffers (the drop-in call a per-frame driver makes):
 * copies this frame's pixels zc [B][N_max][2] and flag bytes fl [B][N_max] (match_mode 1:
 * candidates, EKFSLAM_F_CAND bit; match_mode 2: explicit matches, HAS_Z|IC bits) and the
 * uniforms u [B][n_u] to the device, runs ekfslam_step(reset=1), copies back x_k_k
 * [B][n_max], the flag bytes [B][N_max] and the stats [B] (each may be NULL), and
 * synchronises.  Copies are asynchronous when the host buffers are pinned. */
int ekfslam_step_host(ekfslam_ctx* ctx, int match_mode, const double* zc, const uint8_t* fl,
                      const double* u, int n_u, double* x_out, uint8_t* flags_out,
                      ekfslam_stats* stats_out);

/* ---- "next" rows (SURVEY §8f): map management on the device ---------------- */
/* mc/initialize_x_and_p.m:3-24 broadcast: filters [b0,b0+nb) become the camera-only filter with state
 * xv [13] and covariance Pxv [13*13] and an EMPTY map (nstate = 13, nfeat = 0). */
int ekfslam_reset_filters(ekfslam_ctx* ctx, int b0, int nb, const double* xv, const double* Pxv);
/* mc/add_features_inverse_depth.m:18-22 -> mc/hinv.m:3-26 +
 * mc/add_a_feature_covariance_inverse_depth.m:3-64: append one inverse-depth feature per
 * filter from its distorted pixel uvd [nb][2] (add may be NULL = all; add[b]==0 skips filter b).
 * Operates on (x_k_k,p_k_k); grows nstate by 6 and nfeat by 1. */
int ekfslam_add_features(ekfslam_ctx* ctx, int b0, int nb, const double* uvd, const uint8_t* add,
                         double std_pxl, double initial_rho, double std_rho);

/* mc/inversedepth_2_cartesian.m:3-52 on (x_k_k,p_k_k) of every filter: the FIRST inverse-depth feature whose
 * linearity index 4*std_d*cos(alpha)/d is below `threshold` (reference: 0.1) becomes Cartesian (at most one
 * per call, :49): x block [x y z theta phi rho] -> [X Y Z], P <- J P J'.  force_index >= 0 instead converts
 * that feature of every filter unconditionally.  converted [B] (may be NULL) receives the index or -1. */
int ekfslam_inversedepth_2_cartesian(ekfslam_ctx* ctx, double threshold, int force_index, int32_t* converted);
/* mc/delete_a_feature.m:4-25 for every feature with del[b][i] != 0 (del: [nb][N_max]); the state, the
 * covariance and the features_info arrays are compacted. */
int ekfslam_delete_features(ekfslam_ctx* ctx, int b0, int nb, const uint8_t* del);

/* mc/map_management.m:1-35 for every filter, on the device, in the reference's order:
 *   1. delete_features (:7; NOT shipped by the reference - rule of the published toolbox it derives from:
 *      times_predicted > 5 and times_measured < 0.5*times_predicted) via mc/delete_a_feature.m:4-25
 *   2. measured = #{low_innovation_inlier || high_innovation_inlier} over the survivors (:11-14)
 *   3. mc/update_features_info.m:4-18 (:17)
 *   4. mc/inversedepth_2_cartesian.m:3-52, at most one conversion (:22)
 *   5. initialize_features (:27-35): min_n features if measured == 0, else min_n - measured if that is
 *      positive; the corner search of mc/initialize_a_feature.m:22-57 (CV Toolbox) is replaced by the
 *      context's DETECTION LIST (ekfslam_upload_detections or ekfslam_world_detect), one attempt per
 *      detection, attempt cap 50 (mc/initialize_features.m:5); each accepted corner goes through
 *      mc/add_features_inverse_depth.m (initial_rho = 1, std_rho = 1, std_pxl = std_z,
 *      mc/initialize_a_feature.m:10-12).
 * Operates on (x_k_k, p_k_k).  Follow it with ekfslam_step(reset = 0): step 3 already reset the frame. */
int ekfslam_map_management(ekfslam_ctx* ctx, int min_number_of_features_in_image);
/* detection list: uv [nb][K][2] distorted corner pixels, tag [nb][K] (may be NULL -> -1), n [nb] valid entries */
int ekfslam_upload_detections(ekfslam_ctx* ctx, int b0, int nb, int K, const double* uv, const int32_t* tag,
                              const int32_t* n);
int ekfslam_download_detections(ekfslam_ctx* ctx, int b0, int nb, int K, double* uv, int32_t* tag, int32_t* n);
/* features_info bookkeeping fields: counters [nb][N_max][2] = times_predicted, times_measured
 * (mc/add_feature_to_info_vector.m:16-17) and tag [nb][N_max] = the feature's identity, the stand-in for
 * feature_when_initialized (:10).  Either may be NULL. */
int ekfslam_upload_feature_meta(ekfslam_ctx* ctx, int b0, int nb, const int32_t* counters, const int32_t* tag);
int ekfslam_download_feature_tags(ekfslam_ctx* ctx, int b0, int nb, int32_t* tag);
/* the staged candidates of the current frame: zc [nb][N_max][2], fl [nb][N_max] (EKFSLAM_F_CAND bit) */
int ekfslam_download_candidates(ekfslam_ctx* ctx, int b0, int nb, double* zc, uint8_t* fl);

/* ---- synthetic world on the device (stand-in for the image front-end, SURVEY §8f rank 3) ---- */
/* The reference's matcher (mc/matching.m:16-53: FAST corners in the search ellipse, FREAK match) and its feature
 * detector (mc/initialize_a_feature.m:22-57) need MATLAB's CV Toolbox and an image sequence that is not in the
 * repository.  Their stand-in keeps resident: M world points per filter and the true camera trajectory; per
 * frame it produces (i) for every feature in every map the candidate pixel z = distort(project(point(tag))) +
 * noise (or a gross outlier), staged exactly like ekfslam_upload_candidates, and (ii) the detection list for
 * ekfslam_map_management.  Noise is counter-based (seed, filter, frame, point), so a frame can be regenerated. */
typedef struct {
    uint64_t seed;
    int32_t b_offset;     /* index of this context's filter 0 inside a larger sharded batch       */
    int32_t flaky_mod;    /* point w is flaky when w % flaky_mod == flaky_mod - 1                  */
    double noise_px;      /* std of the pixel noise                                                */
    double gross_px;      /* gross outliers are uniform in +-gross_px                              */
    double p_outlier;     /* outlier probability of an ordinary point                              */
    double p_flaky;       /* outlier probability of a flaky point                                  */
    double band_px;       /* excluded image band for new features (reference: 21)                  */
} ekfslam_world_params;
/* points [B][M][3], poses [T+1][B][7] = r (3), q (4, scalar first); M <= 2048 */
int ekfslam_world_upload(ekfslam_ctx* ctx, int M, int T, const double* points, const double* poses,
                         const ekfslam_world_params* wp);
int ekfslam_world_candidates(ekfslam_ctx* ctx, int t);      /* stage the candidates of frame t        */
int ekfslam_world_detect(ekfslam_ctx* ctx, int t, int K);   /* fill the detection list from frame t   */
/* RANSAC uniform stream of frame t, n_u per filter (stands in for the rand(1) of mc/select_random_match.m:12) */
int ekfslam_world_uniforms(ekfslam_ctx* ctx, int t, int n_u);
/* the resident uniform stream, u [nb][n_u] (n_u must equal the resident stream's length) */
int ekfslam_download_uniforms(ekfslam_ctx* ctx, int b0, int nb, double* u, int n_u);

/* ---- scoring against the resident ground truth (B independent Monte-Carlo runs) ---- */
/* Evaluation reads the resident estimate (x_k_k, P): called between ekfslam_predict and the li update it scores the
 * predicted covariance.  It touches nothing else of the filter (x, xp, P, flags, counters, tags and stats are
 * read-only to it).  Definitions, with (r_t, q_t) the true pose of frame t (q scalar first):
 *   camera:  e_r = x[0:3] - r_t;  d = conj(q_t) * x[3:7] (not renormalised), s = sign(d_w) (+1 at 0),
 *            e_theta = 2 s d_xyz, angle = 2 atan2(|d_xyz|, |d_w|);  J = blockdiag(I3, 2 s E Q_L(conj(q_t))) on the 7
 *            (r, q) columns (Q_L = left-multiplication matrix, E keeps rows 1..3), C_pose = J P[0:7,0:7] J' (6x6);
 *            nees_pos = e_r' inv(P_rr) e_r (3 dof), nees_pose = e' inv(C_pose) e with e = [e_r; e_theta] (6 dof),
 *            both through a Cholesky factorisation.
 *   feature: slot i of filter b is valid when i < nfeat[b]; its tag names its world point.  Inverse-depth
 *            [x y z theta phi rho] -> p = [x y z] + m(theta, phi) / rho, m = [cos(phi) sin(theta), -sin(phi),
 *            cos(phi) cos(theta)] (mc/inversedepth_2_cartesian.m:37-45), a Cartesian block is p itself;
 *            C_f = J_f P_ff J_f' (3x3), e_f = p - points[b][tag], nees_f = e_f' inv(C_f) e_f (Cholesky).
 *            rho <= 0 or a Cholesky pivot of C_f <= 0: not evaluable (NaN per-feature outputs, n_skip, status bit 2);
 *            a tag outside [0, M): no truth (NaN, n_skip, status bit 1).
 * Sums run over the evaluable features in feature order; the reduction has a fixed order (no floating-point
 * atomics), so a record is bit-identical from run to run.  When a camera Cholesky pivot is <= 0 the affected NEES
 * (nees_pose, and nees_pos when P_rr itself fails) is NaN and status bit 0 is set; a NaN carries into the totals. */
typedef struct {
    double pos_sq_err;  /* |e_r|^2                                   */
    double rot_sq_err;  /* angle^2 [rad^2]                           */
    double nees_pos;    /* 3 dof                                     */
    double nees_pose;   /* 6 dof                                     */
    double map_sq_err;  /* sum of |e_f|^2 over the evaluable features */
    double map_nees;    /* sum of nees_f over the evaluable features  */
    int32_t n_map;      /* evaluable features                        */
    int32_t n_skip;     /* valid slots without truth or not evaluable */
    int32_t frames;     /* 1 per evaluation (totals: frames summed)  */
    int32_t status;     /* bit0: camera covariance not SPD; bit1: a feature without truth; bit2: a feature not evaluable */
} ekfslam_eval;
/* score every filter against frame t of the world (ekfslam_world_upload); stream-ordered, no host copies.  The
 * per-frame record replaces the previous one and is added field by field (status OR-ed) into the running totals.
 * ERR_STATE without a world, ERR_INVALID for t outside [0, T]. */
int ekfslam_evaluate(ekfslam_ctx* ctx, int t);
/* rec [nb]: the last frame's records (totals == 0) or the running totals (totals != 0).  feat_err [nb][N_max][3] and
 * feat_nees [nb][N_max] (either may be NULL) are the last frame's e_f and nees_f, NaN where a slot is empty, has no
 * truth or is not evaluable; they exist only for the last frame, so they must be NULL when totals != 0.
 * ERR_STATE before the first ekfslam_evaluate. */
int ekfslam_download_eval(ekfslam_ctx* ctx, int b0, int nb, int totals, ekfslam_eval* rec, double* feat_err,
                          double* feat_nees);
/* zero the running totals (stream-ordered) */
int ekfslam_reset_eval(ekfslam_ctx* ctx);
/* the map in Cartesian coordinates, no world needed: p [nb][N_max][3] = p of every slot, cov [nb][N_max][6] = C_f
 * packed (xx, yx, yy, zx, zy, zz); NaN for empty and not evaluable slots.  Either pointer may be NULL. */
int ekfslam_map_cartesian(ekfslam_ctx* ctx, int b0, int nb, double* p, double* cov);

/* ---- measurement hooks ------------------------------------------------------ */
/* bracket every kernel launch with a CUDA event pair on the context's stream and accumulate the
 * elapsed time per kernel; enabling again resets the accumulators, on=0 removes the events */
int ekfslam_enable_timing(ekfslam_ctx* ctx, int on);
int ekfslam_kernel_count(void);
/* synchronises, then returns the accumulated milliseconds and launch count of kernel `slot` */
int ekfslam_kernel_time(ekfslam_ctx* ctx, int slot, char* name, int name_cap, double* ms,
                        int64_t* launches);
/* point the per-frame inputs (candidates / matches zc [B][N_max][2], flag bytes [B][N_max],
 * uniforms [B][n_u]) at caller-owned DEVICE buffers instead of the context's own staging
 * buffers — no copy; lets a driver keep many frames resident in HBM.  unbind restores. */
int ekfslam_bind_frame(ekfslam_ctx* ctx, const void* d_zc, const void* d_fl, const void* d_u, int n_u);
int ekfslam_unbind_frame(ekfslam_ctx* ctx);

/* ---- raw device pointers (for callers that own the stream, e.g. torch) ----- */
/* name: "x","xp","P","G","W","h","Hc","S","z","zc","flags","mflags","u","stats","Sb","Li","yv" */
void* ekfslam_device_ptr(ekfslam_ctx* ctx, const char* name);

#ifdef __cplusplus
}
#endif
#endif /* EKFSLAM_H */
