/* cubemap_b200.h — C ABI of libcubemap_b200.so (B200 / sm_100a hot path of CubemapSLAM).
 *
 * The reference has no FFI layer: its "operator API" for this path is four C++ entry points compiled into
 * libCubemapSLAM.so. Each function below names the reference interface it replaces (file:line in the reference
 * tree); the facade classes in include/ORBExtractor.h, ORBMatcher.h, Optimizer.h, CubemapWarp.h keep the
 * reference signatures and forward to these. INTEGRATION.md shows the maintainer-side binding.
 *
 * Conventions: every function returns 0 on success or a negative CSLAM_E_* code (cslam_last_error() gives the
 * text, thread-local); no exceptions cross the ABI; the caller owns every buffer it passes; the library owns
 * device memory and streams; "_dev" entry points take DEVICE pointers and run asynchronously on the handle's
 * stream (cslam_*_sync to wait), all others take HOST pointers and are synchronous. There is no CPU fallback:
 * without a CUDA device creation fails with CSLAM_E_NODEVICE.
 */
#ifndef CUBEMAP_B200_H
#define CUBEMAP_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define CSLAM_OK 0
#define CSLAM_E_NODEVICE -1
#define CSLAM_E_BADARG -2
#define CSLAM_E_CUDA -3
#define CSLAM_E_CAPACITY -4   /* an internal fixed-capacity buffer overflowed (reported, never silently truncated) */
#define CSLAM_E_NCCL -5

const char* cslam_last_error(void);
int cslam_version(void);
int cslam_device_count(void);

/* ---------------------------------------------------------------------------------------------- camera / warp
 * CamModelGeneral::SetCamParams (src/CamModelGeneral.cpp:75-93) as configured by System::System (src/System.cpp:63-89). */
typedef struct cslam_cam_params {
    double c, d, e, u0, v0;
    double poly[5];      /* Camera.a0..a4, zero padded (src/System.cpp:67-69) */
    double invpoly[12];  /* Camera.pol0..pol11, zero padded (src/System.cpp:70-72) */
    int32_t Iw, Ih;      /* fisheye image size */
    int32_t face_w, face_h; /* CubeFace.w/h; fx=fy=cx=cy=w/2 (src/System.cpp:83-84). Must be square. */
    double fov_deg;
} cslam_cam_params;

/* cv::KeyPoint field order (28 bytes) — element type of ORBextractor's output vector. */
typedef struct cslam_keypoint {
    float x, y, size, angle, response;
    int32_t octave, class_id;
} cslam_keypoint;

typedef struct cslam_orb_params {  /* ORBextractor::ORBextractor arguments (src/ORBExtractor.cpp:381-383) */
    int32_t nfeatures;
    float scale_factor;
    int32_t nlevels, ini_th_fast, min_th_fast;
} cslam_orb_params;

/* Front end = System::CreateUndistortRectifyMap (src/System.cpp:301-324, run once here on the host exactly like the
 * reference does at start-up) + CvtFisheyeToCubeMap_reverseQuery_withInterpolation (src/System.cpp:327-355)
 * + ORBextractor::operator() (src/ORBExtractor.cpp:838-926), batched over `max_batch` frames per launch group.
 * `mask` is the (3*face_h x 3*face_w) CV_8U cubemap mask the reference passes to every Frame (host pointer, copied). */
typedef struct cslam_frontend cslam_frontend;
int cslam_frontend_create(cslam_frontend** out, int device, const cslam_cam_params* cam, const cslam_orb_params* orb,
                          const uint8_t* mask, int mask_pitch, int max_batch);
void cslam_frontend_destroy(cslam_frontend* fe);
int cslam_frontend_kp_capacity(const cslam_frontend* fe);   /* per-frame keypoint slots = nfeatures + 3*nlevels */
void* cslam_frontend_stream(const cslam_frontend* fe);      /* cudaStream_t the _dev calls are enqueued on */
int cslam_frontend_sync(cslam_frontend* fe);                /* waits, then reports sticky capacity/CUDA errors */

/* System::CvtFisheyeToCubeMap_reverseQuery_withInterpolation(cubemapImg, fisheyeImg, INTER_LINEAR) for `batch`
 * frames. fisheye: batch x Ih x Iw (pitch Iw); canvas: batch x 3H x canvas_pitch, corner tiles are left untouched. */
int cslam_warp(cslam_frontend* fe, const uint8_t* fisheye, int batch, uint8_t* canvas, int canvas_pitch);
/* ORBextractor::operator()(image, mask, keypoints, descriptors) on host cubemap canvases (3H x 3W, given pitch).
 * kps: batch x kp_capacity; desc: batch x kp_capacity x 32; n_out: batch. */
int cslam_orb_extract(cslam_frontend* fe, const uint8_t* canvas, int canvas_pitch, int batch, cslam_keypoint* kps,
                      uint8_t* desc, int32_t* n_out);
/* warp + extract, host fisheye frames in, host keypoints/descriptors out (copies inside). */
int cslam_frontend_run(cslam_frontend* fe, const uint8_t* fisheye, int batch, cslam_keypoint* kps, uint8_t* desc,
                       int32_t* n_out);
/* Same with device-resident input and output (asynchronous on the front end's stream). */
int cslam_frontend_run_dev(cslam_frontend* fe, const uint8_t* fisheye_dev, int batch, cslam_keypoint* kps_dev,
                           uint8_t* desc_dev, int32_t* n_out_dev);
/* Debug / stage-parity access (host copies of the last batch's intermediates). level image is apron-less. */
int cslam_frontend_level_size(const cslam_frontend* fe, int level, int* w, int* h);
int cslam_frontend_get_level(cslam_frontend* fe, int frame, int level, uint8_t* out /* h*w */);
int cslam_frontend_get_candidates(cslam_frontend* fe, int frame, int level, int32_t* xyr /* cap*3 */, int cap, int* n);
int cslam_frontend_get_maps(const cslam_frontend* fe, float* map1, float* map2);   /* 3H x 3W float32 each */
int cslam_frontend_tables(const cslam_frontend* fe, float* scale, float* inv_scale, float* sigma2, float* inv_sigma2,
                          int32_t* features_per_level, int32_t* umax16);
/* Per-kernel device timing for bench.py's roofline block: when enabled, CUDA events are recorded on the front end's
 * stream between launches and accumulated per kernel kind at the next cslam_frontend_sync. kind 0..4 =
 * k_warp, k_pyramid, k_fast, k_distribute, k_describe. */
int cslam_frontend_set_timing(cslam_frontend* fe, int enable);
int cslam_frontend_get_timing(const cslam_frontend* fe, int kind, const char** name, double* ms, int64_t* count);
/* Number of kernel launches issued by this front end so far (bench.py's gpu_launches). */
int64_t cslam_frontend_launches(const cslam_frontend* fe);

/* ---------------------------------------------------------------------------------------------- matcher
 * ORBMatcher (include/ORBMatcher.h:42-104). Thresholds TH_LOW=50, TH_HIGH=100, HISTO_LENGTH=12 (src/ORBMatcher.cpp:42-45). */
typedef struct cslam_matcher cslam_matcher;
int cslam_matcher_create(cslam_matcher** out, int device, int max_pairs, int max_features);
void cslam_matcher_destroy(cslam_matcher* m);
void* cslam_matcher_stream(const cslam_matcher* m);
int cslam_matcher_sync(cslam_matcher* m);
int64_t cslam_matcher_launches(const cslam_matcher* m);

/* ORBMatcher::DescriptorDistance (src/ORBMatcher.cpp:951-967), host-side convenience for n descriptor pairs. */
int cslam_hamming(cslam_matcher* m, const uint8_t* a, const uint8_t* b, int n, int32_t* dist);
/* All-pairs matcher (BASELINE config 3; semantics defined in DESIGN.md §matcher — SearchByBoW's acceptance rule and
 * rotation histogram over all columns, per row of A): descA npairs x nA x 32, angA npairs x nA, same for B.
 * match12: npairs x nA (column of B or -1); dist12/second12 may be NULL; nmatches: npairs. */
int cslam_match_bruteforce(cslam_matcher* m, const uint8_t* descA, const float* angA, int nA, const uint8_t* descB,
                           const float* angB, int nB, int npairs, float nnratio, int th_low, int check_ori,
                           int32_t* match12, int32_t* dist12, int32_t* second12, int32_t* nmatches);
int cslam_match_bruteforce_dev(cslam_matcher* m, const uint8_t* descA, const float* angA, int nA, const uint8_t* descB,
                               const float* angB, int nB, int npairs, float nnratio, int th_low, int check_ori,
                               int32_t* match12, int32_t* dist12, int32_t* second12, int32_t* nmatches);
/* The same matcher between consecutive frames of a front-end batch, reading cslam_frontend_run_dev's output layout directly (device pointers,
 * asynchronous): frame f is matched against frame f+1, f = 0 .. nframes-2; kp_stride = cslam_frontend_kp_capacity; n = the front end's n_out. */
int cslam_match_frames_dev(cslam_matcher* m, const cslam_keypoint* kps, const uint8_t* desc, const int32_t* n, int kp_stride, int nframes, float nnratio, int th_low,
                           int check_ori, int32_t* match12, int32_t* nmatches);
int cslam_match_frames(cslam_matcher* m, const cslam_keypoint* kps, const uint8_t* desc, const int32_t* n, int kp_stride, int nframes, float nnratio, int th_low, int check_ori,
                       int32_t* match12, int32_t* nmatches);   /* host buffers, synchronous */
/* Measured POPC issue rate of this GPU (32-bit population counts per second with the XOR+POPC+ADD mix of the Hamming kernels, no memory traffic):
 * the ceiling the matcher's roofline fraction is quoted against (bench.py). */
int cslam_ubench_popc(cslam_matcher* m, double* popc32_per_s);
/* Same for 3-input u16x2 min/max (VIMNMX3.U16x2), the instruction k_fast is bound by; out: thread-level operations per second. */
int cslam_ubench_minmax3(cslam_matcher* m, double* ops_per_s);
/* ORBMatcher::SearchByBoW(KeyFrame*, Frame&, vector<MapPoint*>&) (src/ORBMatcher.cpp:409-539) for npairs (KF,F) pairs.
 * kf_valid: 1 where the KF feature has a good MapPoint; node_kf/node_f: DBoW2 FeatureVector node id per feature.
 * match_f: npairs x nF (index of the KF feature whose MapPoint is assigned, or -1); nmatches: npairs. */
int cslam_search_by_bow(cslam_matcher* m, const uint8_t* descKF, const float* angKF, const uint8_t* kf_valid,
                        const int32_t* node_kf, int nKF, const uint8_t* descF, const float* angF, const int32_t* node_f,
                        int nF, int npairs, float nnratio, int check_ori, int32_t* match_f, int32_t* nmatches);
int cslam_search_by_bow_dev(cslam_matcher* m, const uint8_t* descKF, const float* angKF, const uint8_t* kf_valid,
                            const int32_t* node_kf, int nKF, const uint8_t* descF, const float* angF, const int32_t* node_f,
                            int nF, int npairs, float nnratio, int check_ori, int32_t* match_f, int32_t* nmatches);

/* ORBMatcher::SearchByBoW(KeyFrame*, KeyFrame*, vector<MapPoint*>&) (src/ORBMatcher.cpp:541-674, loop closing): both sides need a good
 * MapPoint (valid1/valid2), features of the second key frame are consumed, acceptance is the strict best < TH_LOW.
 * match12: npairs x n1 (index of the matched feature of key frame 2, or -1). */
int cslam_search_by_bow_kf(cslam_matcher* m, const uint8_t* desc1, const float* ang1, const uint8_t* valid1, const int32_t* node1, int n1,
                           const uint8_t* desc2, const float* ang2, const uint8_t* valid2, const int32_t* node2, int n2, int npairs,
                           float nnratio, int check_ori, int32_t* match12, int32_t* nmatches);

/* ---------------------------------------------------------------------------------------------- vocabulary (DBoW2 transform)
 * ORBVocabulary::transform(features, BowVector&, FeatureVector&, levelsup) as Frame::ComputeBoW / KeyFrame::ComputeBoW call it (src/Frame.cpp:719-726;
 * ThirdParty/DBoW2/DBoW2/TemplatedVocabulary.h:1127-1262). The tree is given as flat arrays for nodes 1..n_nodes in ORBvoc.txt's line order (what
 * TemplatedVocabulary::loadFromTextFile :1337-1415 reads): parent id, leaf flag, 32 descriptor bytes, weight; scoring L1_NORM, weighting TF_IDF.
 * Outputs per frame (stride slots): node = FeatureVector node id of the feature at level L - levelsup (-1: stopped word) - exactly the per-feature node
 * array cslam_search_by_bow takes -; bow_word / bow_val = the BowVector in map order (bow_count entries, L1-normalised doubles, bit-identical to DBoW2). */
typedef struct cslam_vocabulary cslam_vocabulary;
int cslam_vocabulary_create(cslam_vocabulary** out, int device, int k, int L, int n_nodes, const int32_t* parent, const uint8_t* is_leaf, const uint8_t* desc, const double* weight,
                            int max_frames, int max_features);
void cslam_vocabulary_destroy(cslam_vocabulary* v);
void* cslam_vocabulary_stream(const cslam_vocabulary* v);
int cslam_vocabulary_sync(cslam_vocabulary* v);
int cslam_bow_transform(cslam_vocabulary* v, const uint8_t* desc, const int32_t* n, int stride, int nframes, int levelsup, int32_t* word /* may be NULL */, int32_t* node,
                        int32_t* bow_word, double* bow_val, int32_t* bow_count);
int cslam_bow_transform_dev(cslam_vocabulary* v, const uint8_t* desc, const int32_t* n, int stride, int nframes, int levelsup, int32_t* word, int32_t* leaf, int32_t* node,
                            int32_t* bow_word, double* bow_val, int32_t* bow_count);

/* ---------------------------------------------------------------------------------------------- tracker
 * The matcher on the steady-state frame path and the per-frame indexing it needs (SURVEY.md 8(f) rows 1 and 3):
 *   Frame::ComputeKeyPointRays (src/Frame.cpp:746-760) + Frame::AssignFeaturesToGrid (:158-176)      -> cslam_frame_index
 *   Frame::GetFeaturesInArea (:251-716)                                                               -> inside the search kernels; cslam_area_rects on the host
 *   ORBMatcher::SearchByProjection(Frame&, const Frame&, th, mono)  (src/ORBMatcher.cpp:130-251)      -> cslam_search_by_projection_last
 *   ORBMatcher::SearchByProjection(Frame&, const vector<MapPoint*>&, th)  (src/ORBMatcher.cpp:51-128) -> cslam_search_by_projection_local
 * All calls are batched over independent frames; "stride" = slots per frame in the batched arrays (<= 4096), n[] = used slots.
 * Grid layout: cell_start = (5*50*50 + 1) uint16 per frame, CSR over cells in mGrid[face][col][row] order; cell_idx = feature indices,
 * ascending inside a cell (the order AssignFeaturesToGrid produces). */
typedef struct cslam_tracker cslam_tracker;
int cslam_tracker_create(cslam_tracker** out, int device, int max_frames, int max_features);
void cslam_tracker_destroy(cslam_tracker* t);
void* cslam_tracker_stream(const cslam_tracker* t);
int cslam_tracker_sync(cslam_tracker* t);
int64_t cslam_tracker_launches(const cslam_tracker* t);
#define CSLAM_GRID_CELLS 12500
int cslam_frame_index(cslam_tracker* t, const cslam_keypoint* kps, const int32_t* n, int nframes, int kp_stride, int face_w, int face_h, float* rays /* may be NULL */,
                      uint16_t* cell_start, uint16_t* cell_idx);
int cslam_frame_index_dev(cslam_tracker* t, const cslam_keypoint* kps, const int32_t* n, int nframes, int kp_stride, int face_w, int face_h, float* rays, uint16_t* cell_start,
                          uint16_t* cell_idx);
/* Host utility, no device needed: the (up to 3) cell rectangles Frame::GetFeaturesInArea visits for a window, in visiting order;
 * rects: 3 x {face, col0, col1, row0, row1}, not yet clamped to [0, 49] (AddCells clamps). Returns their number. */
int cslam_area_rects(float x, float y, float r, int face_w, int face_h, int32_t* rects);
/* has_mp: LastFrame.mvpMapPoints[i] != NULL && !mvbOutlier[i]; Xw / d_mp: that MapPoint's GetWorldPos() / GetDescriptor(); mp_obs: Observations() > 0;
 * cur_taken: CurrentFrame.mvpMapPoints[i2] holds a MapPoint with Observations() > 0 before the call; cos_fov_th: CamModelGeneral::GetCosFovTh().
 * match_cur: npairs x cur_stride, index of the LastFrame feature whose MapPoint is assigned to the slot; -1 = slot untouched; -2 = assigned and then cleared by
 * the rotation-consistency filter (the reference sets the slot to NULL). nmatches: the function's return value. */
int cslam_search_by_projection_last(cslam_tracker* t, int npairs, const cslam_keypoint* k_cur, const uint8_t* d_cur, const int32_t* n_cur, int cur_stride,
                                    const uint8_t* cur_taken, const float* Tcw_cur, const cslam_keypoint* k_last, const int32_t* n_last, int last_stride,
                                    const uint8_t* has_mp, const float* Xw, const uint8_t* d_mp, const uint8_t* mp_obs, int face_w, int face_h, float cos_fov_th, float th,
                                    int check_ori, float scale_factor, int nlevels, int32_t* match_cur, int32_t* nmatches);
int cslam_search_by_projection_last_dev(cslam_tracker* t, int npairs, const cslam_keypoint* k_cur, const uint8_t* d_cur, const int32_t* n_cur, int cur_stride,
                                        const uint16_t* cell_start, const uint16_t* cell_idx, const uint8_t* cur_taken, const float* Tcw_cur,
                                        const cslam_keypoint* k_last, const int32_t* n_last, int last_stride, const uint8_t* has_mp, const float* Xw, const uint8_t* d_mp,
                                        const uint8_t* mp_obs, int face_w, int face_h, float cos_fov_th, float th, int check_ori, float scale_factor, int nlevels,
                                        int32_t* match_cur, int32_t* nmatches);
/* in_view: mbTrackInView && !isBad(); proj_xy / level / view_cos: mTrackProjX/Y, mnTrackScaleLevel, mTrackViewCos left by Frame::isInFrustum. */
int cslam_search_by_projection_local(cslam_tracker* t, int nframes, const cslam_keypoint* k_f, const uint8_t* d_f, const int32_t* n_f, int f_stride, const uint8_t* f_taken,
                                     const int32_t* n_mp, int mp_stride, const uint8_t* in_view, const float* proj_xy, const int32_t* level, const float* view_cos,
                                     const uint8_t* d_mp, const uint8_t* mp_obs, int face_w, int face_h, float th, float nnratio, float scale_factor, int nlevels,
                                     int32_t* match_f, int32_t* nmatches);
int cslam_search_by_projection_local_dev(cslam_tracker* t, int nframes, const cslam_keypoint* k_f, const uint8_t* d_f, const int32_t* n_f, int f_stride,
                                         const uint16_t* cell_start, const uint16_t* cell_idx, const uint8_t* f_taken, const int32_t* n_mp, int mp_stride,
                                         const uint8_t* in_view, const float* proj_xy, const int32_t* level, const float* view_cos, const uint8_t* d_mp,
                                         const uint8_t* mp_obs, int face_w, int face_h, float th, float nnratio, float scale_factor, int nlevels, int32_t* match_f,
                                         int32_t* nmatches);

/* What Tracking does between SearchByProjection and PoseOptimization (src/Optimizer.cpp:80-131): the matched slots of each frame, in slot order and
 * with the ray.z >= cos_fov_th test when rays are given, become (world point, key point, 1/sigma^2) correspondences at stride cur_stride; count_out[p] of them.
 * inv_sigma2_levels_dev: mvInvLevelSigma2 (one float per pyramid level) on the device. Device pointers, asynchronous on the tracker's stream. */
int cslam_tracker_gather_pose_inputs_dev(cslam_tracker* t, int npairs, const int32_t* match_cur, const cslam_keypoint* k_cur, const int32_t* n_cur, int cur_stride,
                                         const float* rays_cur, float cos_fov_th, const float* Xw_last, int last_stride, const float* inv_sigma2_levels_dev,
                                         float* Xw_out, float* kp_xy_out, float* inv_sigma2_out, int32_t* count_out);

/* ---------------------------------------------------------------------------------------------- optimizer
 * Optimizer::LocalBundleAdjustment (src/Optimizer.cpp:192-451) on the already collected local window.
 * Vertices must be ordered like g2o orders them: KFs by mnId, points by mnId. */
typedef struct cslam_ba_problem {
    int32_t n_kf, n_mp, n_edges;
    float* Tcw;              /* n_kf x 16 row-major float32 (KeyFrame::GetPose), in/out */
    const uint8_t* kf_fixed; /* n_kf: mnId==0 or member of lFixedCameras */
    float* points;           /* n_mp x 3 float32 (MapPoint::GetWorldPos), in/out */
    const int32_t* edge_mp;  /* n_edges */
    const int32_t* edge_kf;  /* n_edges */
    const float* kp_xy;      /* n_edges x 2, keypoint on the cubemap canvas (mvKeys[].pt) */
    const float* inv_sigma2; /* n_edges, mvInvLevelSigma2[kp.octave] */
    int32_t face_w, face_h;
} cslam_ba_problem;

typedef struct cslam_ba_result {
    uint8_t* outlier;        /* n_edges: observations the reference would erase (src/Optimizer.cpp:403-416); may be NULL */
    double* pose_fp64;       /* n_kf x 7 (t, qx qy qz qw) before the float32 cast; may be NULL */
    double* points_fp64;     /* n_mp x 3; may be NULL */
    double* lm_log;          /* log_cap x 4: chi2, lambda, trials, accepted per LM iteration; may be NULL */
    int32_t log_cap;
    int32_t iterations;      /* out: LM iterations run (both optimize() calls) */
    int32_t trials;          /* out: total LM trials (linear solves) */
} cslam_ba_result;

typedef struct cslam_optimizer cslam_optimizer;
int cslam_optimizer_create(cslam_optimizer** out, int device);
void cslam_optimizer_destroy(cslam_optimizer* o);
int64_t cslam_optimizer_launches(const cslam_optimizer* o);
/* Per-kernel device timing of cslam_local_ba for bench.py's roofline block (CUDA events between launches; disables the CUDA-graph replay while on).
 * kind 0..9 = k_ba_errors, k_ba_lin_points, k_ba_lin_poses, k_ba_dinv, k_ba_schur, exchange, k_ba_solve, k_ba_backsub, k_ba_update, k_ba_scale. */
int cslam_optimizer_set_timing(cslam_optimizer* o, int enable);
int cslam_optimizer_get_timing(const cslam_optimizer* o, int kind, const char** name, double* ms, int64_t* count);
/* Test / measurement hook (like cslam_ubench_*): the reduced-camera-system solve of cslam_local_ba alone, with the same launch, on a dense n x n
 * symmetric system. Sg: host, (n+1) x n row-major, rows 0..n-1 = S (only the lower triangle is read), row n = the right-hand side g.
 * stage: -1 = the production rule, 0 = trailing update reads the panels from L2, 1 = panels staged in shared memory (CSLAM_E_BADARG if they do
 * not fit). cluster: CTAs of the solver cluster, 0 = the optimizer's own (CSLAM_SOLVE_CLUSTER, default 8), else 1..16 (> 8 is non-portable;
 * CSLAM_E_BADARG if the device cannot schedule it). x: n doubles out, undefined when *failed. failed: 1 on a zero / non-finite pivot.
 * n > 26112 (4352 free key frames) is CSLAM_E_CAPACITY, reported before Sg is read. */
int cslam_ba_solve_dense(cslam_optimizer* o, int n, const double* Sg, int stage, int cluster, double* x, int32_t* failed);
/* Landmark-sharded multi-GPU BA: every rank calls with the SAME problem; rank r owns landmarks l % nranks == r and
 * all-reduces the reduced camera system over NCCL. id128: ncclUniqueId bytes from cslam_nccl_unique_id on rank 0. */
int cslam_nccl_unique_id(uint8_t id128[128]);
int cslam_optimizer_init_nccl(cslam_optimizer* o, const uint8_t id128[128], int rank, int nranks);
/* its1/its2: iterations of the two optimize() calls (reference: 5 and 10). stop_flag: the reference's pbStopFlag. */
int cslam_local_ba(cslam_optimizer* o, cslam_ba_problem* p, const volatile uint8_t* stop_flag, int its1, int its2,
                   cslam_ba_result* r);
/* Optimizer::PoseOptimization (src/Optimizer.cpp:48-190), batched: `nframes` independent frames, frame f owns
 * correspondences [offset[f], offset[f+1]). Tcw: nframes x 16 in/out; outlier: per correspondence (mvbOutlier);
 * inliers: nframes (return value of the reference function). */
int cslam_pose_optimization(cslam_optimizer* o, int nframes, const int32_t* offset, float* Tcw, const float* Xw,
                            const float* kp_xy, const float* inv_sigma2, int face_w, int face_h, uint8_t* outlier,
                            int32_t* inliers, double* pose_fp64);

/* Device-resident PoseOptimization for pipelines: frame f owns correspondences [f*stride, f*stride + count[f]); all pointers on the device;
 * asynchronous on the optimizer's stream (cslam_optimizer_stream / cslam_optimizer_sync). */
int cslam_pose_optimization_dev(cslam_optimizer* o, int nframes, int stride, const int32_t* count, float* Tcw, const float* Xw, const float* kp_xy, const float* inv_sigma2,
                                int face_w, int face_h, uint8_t* outlier, int32_t* inliers);
void* cslam_optimizer_stream(const cslam_optimizer* o);
int cslam_optimizer_sync(cslam_optimizer* o);

/* ---------------------------------------------------------------------------------------------------------------------------------
 * LocalMapping feature operations (SURVEY §8(f) rank 4): the Hamming / projection work either side of LocalBA on the mapping thread.
 * Host buffers in, host results out (one call per batch); no CPU fallback.
 * --------------------------------------------------------------------------------------------------------------------------------- */
typedef struct cslam_mapper cslam_mapper;
int cslam_mapper_create(cslam_mapper** out, int device);
void cslam_mapper_destroy(cslam_mapper* m);
int64_t cslam_mapper_launches(const cslam_mapper* m);

/* MapPoint::ComputeDistinctiveDescriptors (reference src/MapPoint.cpp:243-303) for a batch of MapPoints: `desc` = the observation descriptors of
 * all points back to back (32 bytes each, in the order the reference iterates mObservations), offset[p] .. offset[p+1] = the rows of point p.
 * best[p] = row (relative to offset[p]) with the least median Hamming distance to the others, first such row; -1 for a point without rows. */
int cslam_distinctive_descriptors(cslam_mapper* m, const uint8_t* desc, const int32_t* offset, int n_points, int32_t* best);

/* The search of ORBMatcher::Fuse(KeyFrame* pKF, const vector<MapPoint*>&, th) (reference src/ORBMatcher.cpp:1126-1240): for every MapPoint the key
 * point of pKF it would be fused with. Per MapPoint the caller evaluates on its own objects what Fuse tests before the search - mp_valid = !isBad &&
 * !IsInKeyFrame(pKF) && depth inside [min, max]DistanceInvariance && PO.Pn >= 0.5 dist - and mp_level = pMP->PredictScale(dist3D, pKF); the
 * library projects (Rcw p + tcw, TransformRaysToCubemap, IsInImage), walks KeyFrame::GetFeaturesInArea(u, v, th * mvScaleFactors[level]) in the
 * reference's order with the level / 5.99-chi2 gates and returns best_idx (-1: none) / best_dist (256: none). The caller then applies
 * `bestDist <= TH_LOW` and the Replace / AddObservation bookkeeping in MapPoint order. scale_factors / inv_level_sigma2: pKF->mvScaleFactors /
 * mvInvLevelSigma2 (nlevels <= 16); n_kf <= 4096. */
int cslam_fuse_search(cslam_mapper* m, const cslam_keypoint* k_kf, const uint8_t* d_kf, int n_kf, const float* Tcw /* 4x4 row-major */, int n_mp, const uint8_t* mp_valid,
                      const float* mp_xw /* n_mp x 3 */, const int32_t* mp_level, const uint8_t* mp_desc /* n_mp x 32 */, float th, const float* scale_factors,
                      const float* inv_level_sigma2, int nlevels, int face_w, int face_h, int32_t* best_idx, int32_t* best_dist);

/* ORBMatcher::SearchForTriangulation(pKF1, pKF2, E12, vMatchedPairs) (reference src/ORBMatcher.cpp:971-1124) for `npairs` key-frame pairs in one
 * launch (LocalMapping::CreateNewMapPoints matches the new key frame against ~20 neighbours). Pair p reads rows [p*stride, p*stride + n[p]) of
 * the per-feature arrays: key points, descriptors, bearing vectors (mvKeyRays), has_mp (GetMapPoint(idx) != NULL), node = the vocabulary node of
 * the feature in mFeatVec (levelsup 4; in [0, 2^20 - 1)). Ow1 = pKF1->GetCameraCenter() (3), Tcw2 = pKF2's pose (16), E12 (9, row-major).
 * scale_factors / level_sigma2 = pKF2->mvScaleFactors / mvLevelSigma2. match12[p*stride1 + i1] = matched feature of KF2 or -1; nmatches[p].
 * (As in the reference, vbMatched2 is never set: two features of KF1 may choose the same feature of KF2.) */
int cslam_search_for_triangulation(cslam_mapper* m, int npairs, const cslam_keypoint* k1, const uint8_t* d1, const float* rays1, const uint8_t* has_mp1, const int32_t* node1,
                                   const int32_t* n1, int stride1, const cslam_keypoint* k2, const uint8_t* d2, const float* rays2, const uint8_t* has_mp2, const int32_t* node2,
                                   const int32_t* n2, int stride2, const float* Ow1, const float* Tcw2, const float* E12, const float* scale_factors,
                                   const float* level_sigma2, int nlevels, int face_w, int face_h, int check_orientation, int32_t* match12, int32_t* nmatches);

#ifdef __cplusplus
}
#endif
#endif
