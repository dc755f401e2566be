/*
 * epivo_b200.h -- C ABI of the B200-native (sm_100a) per-frame-pair geometric core of
 * Ronnypetson/epivo: descriptor matching -> essential matrix (RANSAC / LMedS, 5-point) ->
 * cheirality pose recovery -> SE(3)-chain Levenberg-Marquardt refinement.
 *
 * The reference has no FFI: the path sits behind ordinary C++ call sites into OpenCV and
 * its own jac_Rt_gen_.cpp.  Each entry point below names the reference call it replaces
 * (file:line into the reference tree).  Plain pointers and sizes only; all buffers are
 * caller-owned HOST memory unless a function says "device"; no pointer is retained after
 * return.  Every function returns 0 (EPIVO_OK) or a negative error code and never aborts
 * or throws; epivo_last_error() gives the message.  A context owns one CUDA stream and its
 * workspaces: one context per host thread; distinct contexts are fully concurrent (the
 * reference's LM keeps a mutable global T0_mem, jac_Rt_gen_.cpp:20 -- this ABI has no
 * globals).  There is no CPU fallback: without a CUDA device epivo_create fails.
 */
#ifndef EPIVO_B200_H
#define EPIVO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EPIVO_OK 0
#define EPIVO_ERR_INVALID -1      /* bad argument */
#define EPIVO_ERR_CUDA -2         /* CUDA runtime error (message has the cudaError string) */
#define EPIVO_ERR_UNSUPPORTED -3  /* size / mode outside what the kernels are built for */
#define EPIVO_ERR_NOMODEL -4      /* estimator found no model (cv::findEssentialMat returns empty Mat) */

/* cv::NormTypes / cv:: robust method ids, so callers can pass the OpenCV constants through */
#define EPIVO_NORM_HAMMING 6
#define EPIVO_NORM_HAMMING2 7
#define EPIVO_LMEDS 4
#define EPIVO_RANSAC 8

#define EPIVO_MATCH_NN 0          /* BFMatcher(norm, false).match : 1-NN, first minimum        */
#define EPIVO_MATCH_CROSSCHECK 1  /* BFMatcher(norm, true).match  : mutual NN (reference mode) */
#define EPIVO_MATCH_RATIO 2       /* knnMatch(k=2) + Lowe ratio test d1 < ratio*d2             */

typedef struct epivo_ctx epivo_ctx;

int epivo_create(epivo_ctx** out, int device);
void epivo_destroy(epivo_ctx* ctx);
const char* epivo_last_error(const epivo_ctx* ctx);
const char* epivo_version(void);
/* the context's cudaStream_t (as void*), so callers can record their own CUDA events on it */
void* epivo_stream(epivo_ctx* ctx);
/* number of this library's kernels launched on the context so far */
int64_t epivo_launch_count(const epivo_ctx* ctx);
int epivo_sync(epivo_ctx* ctx);
/* device time (CUDA events on the context stream) of the kernels of the last epivo_lm_rt / epivo_lm_rt_batch call,
 * without its host<->device copies: what the benchmark reports next to the end-to-end time */
int epivo_last_kernel_ms(epivo_ctx* ctx, float* ms);

/* ---- M1: cv::BFMatcher(normType, crossCheck).match(desc0, desc1, matches) ------------
 * replaces kitti_ba.cpp:602,641.  q: nq x desc_bytes, t: nt x desc_bytes, row-major u8
 * (desc_bytes in {16, 32, 64}; ORB = 32).  Outputs (capacity nq each) sorted by query_idx;
 * dist = integer distance (DMatch::distance is its float); dist2 = second-best distance
 * (written in EPIVO_MATCH_RATIO mode only, may be NULL otherwise). */
int epivo_match_hamming(epivo_ctx* ctx, const uint8_t* q, int nq, const uint8_t* t, int nt,
                        int desc_bytes, int norm, int mode, float ratio,
                        int32_t* query_idx, int32_t* train_idx, int32_t* dist, int32_t* dist2,
                        int* n_out);
/* cv::BFMatcher(normType).knnMatch(q, t, 2): per query the two nearest by (distance, index);
 * train_idx2/dist2 are nq x 2.  Entries beyond nt are -1. */
int epivo_knn2_hamming(epivo_ctx* ctx, const uint8_t* q, int nq, const uint8_t* t, int nt,
                       int desc_bytes, int norm, int32_t* train_idx2, int32_t* dist2);

/* ---- E1/E2: cv::findEssentialMat(p0, p1, cam, method, prob, threshold, mask) ----------
 * replaces kitti.cpp:98-104, kitti_E.cpp:98-104, euroc_E.cpp:202-208, kitti_ba.cpp:232,308,702.
 * p0/p1: n x 2 float32 pixels; K: 3x3 row-major float64 (the shim widens the float cv::Mat).
 * samples: optional fixed hypothesis set, m x 5 int32 indices; NULL => OpenCV's own sample
 * stream (cv::RNG(-1), ptsetreg.cpp), which makes the whole call reproduce cv2.
 * E: 3x3 row-major; mask: n bytes in {0,1}.  n < 5 or no model => EPIVO_ERR_NOMODEL.
 * n == 5 returns only the first solution in E (use epivo_five_point for all of them). */
int epivo_find_essential(epivo_ctx* ctx, const float* p0, const float* p1, int n, const double K[9],
                         int method, double prob, double threshold, int max_iters,
                         const int32_t* samples, int m,
                         double E[9], uint8_t* mask, int* n_inliers, int* iters_run);

/* K2 alone: the 5-point minimal solver on m samples of 5 K-normalised correspondences
 * (x1, x2: m x 5 x 2 float64).  E_out: m x 10 x 9, n_models: m. */
int epivo_five_point(epivo_ctx* ctx, const double* x1, const double* x2, int m,
                     double* E_out, int32_t* n_models);

/* K2b: 8-point hypotheses (north_star names them; the reference has no call site -- every findEssentialMat call runs
 * OpenCV's 5-point estimator).  m samples of 8 K-normalised correspondences (x1, x2: m x 8 x 2) -> one essential matrix
 * each (m x 9, row-major, unit Frobenius norm: null vector of the 8 x 9 epipolar system projected onto the essential
 * manifold, U diag(1,1,0) V'); ok[i] = 0 when the eight points are degenerate.  Score them with epivo_score_sampson. */
int epivo_eight_point(epivo_ctx* ctx, const double* x1, const double* x2, int m, double* E_out, int32_t* ok);

/* N4 front end, detector: cv::FastFeatureDetector (FAST-9/16) for a batch of n_images 8-bit images of rows x cols
 * (dense, row-major, one after another) -- replaces FastFeatureDetector::create(40)->detect(src, kp0, Mat()) at
 * kitti_E.cpp:71-74 and kitti_ba.cpp:49,62 (threshold 40) and create() at kitti_ba.cpp:98,117-118 (threshold 10).
 * nonmax != 0: OpenCV's 3x3 non-maximum suppression on cornerScore.  kps: n_images x max_kp x 2 floats (x, y) in
 * OpenCV's order (row by row, left to right); response: n_images x max_kp floats (the score; 0 without suppression)
 * or NULL; counts[i] = corners FOUND in image i -- when it exceeds max_kp only the first max_kp are stored.
 * Coordinates, order and response are bit-exact with OpenCV.  threshold must lie in [0, 255] (beyond that OpenCV's
 * vector and scalar code paths give different answers). */
int epivo_fast_detect(epivo_ctx* ctx, const uint8_t* images, int n_images, int rows, int cols, int threshold,
                      int nonmax, int max_kp, float* kps, float* response, int32_t* counts);

/* N4 front end, tracker: cv::calcOpticalFlowPyrLK with a 21 x 21 window (the default the reference uses) over a
 * sequence of n_frames 8-bit images of rows x cols: pair i (0 <= i < n_frames - 1) tracks its counts[i] points
 * pts[i][0..counts[i]) (n_frames-1 x max_pts x 2 floats, x y) from frame i into frame i + 1 -- replaces
 * calcOpticalFlowPyrLK(src, tgt, pt0, pt1_, status, err) at kitti_E.cpp:79-84 and kitti_ba.cpp:203-208,281-286.
 * The reference's defaults are max_level 3, max_count 30, epsilon 0.01, min_eig_threshold 1e-4 (flags 0, no initial
 * flow).  next_pts: n_frames-1 x max_pts x 2; status: n_frames-1 x max_pts bytes {0,1}; err: n_frames-1 x max_pts floats
 * (OpenCV's `err`: mean absolute window difference at the final position, 0 where the track is lost) or NULL -- as in
 * OpenCV, passing `err` also clears the status of a point whose final position left the image; every reference call
 * site passes it.  Entries beyond counts[i] are not written.  Pyramid, derivatives and the fixed-point windows are
 * exact; positions agree with OpenCV to 1e-3 px except where a stopping test of the iteration falls on the other side
 * (see DESIGN.md). */
int epivo_lk_track(epivo_ctx* ctx, const uint8_t* images, int n_frames, int rows, int cols, const float* pts,
                   const int32_t* counts, int max_pts, int max_level, int max_count, double epsilon,
                   double min_eig_threshold, float* next_pts, uint8_t* status, float* err);

/* N4 front end, undistortion: cv::remap(src, dst, map1, map2, INTER_LINEAR) (BORDER_CONSTANT) for a batch of n_images
 * 8-bit images of rows x cols with the FIXED-POINT maps of initUndistortRectifyMap / convertMaps -- map_xy: drows x
 * dcols x 2 int16 (CV_16SC2: integer source x, y), map_frac: drows x dcols uint16 (CV_16UC1: (fy << 5) | fx, fractions
 * in 1/32 pixel) -- as the EuRoC driver builds them once (euroc_E.cpp:105-113) and applies them to every frame
 * (:169-174).  out: n_images x drows x dcols.  Bit-exact with OpenCV. */
int epivo_remap(epivo_ctx* ctx, const uint8_t* images, int n_images, int rows, int cols, const int16_t* map_xy,
                const uint16_t* map_frac, int drows, int dcols, int border_value, uint8_t* out);

/* N4 front end, descriptor extractor: cv::ORB::detectAndCompute for a batch of n_images 8-bit images of rows x cols --
 * replaces `ORB::create(10000, 1.2f, 8, 15, 0, 2, ORB::FAST_SCORE)` + `orb->detect(src, kp)` + `orb->compute(src, kp, desc)`
 * at kitti_ba.cpp:128-152.  Built for that configuration's family: firstLevel 0, WTA_K 2, FAST score, patchSize 31;
 * nfeatures, scale_factor (1 < s <= 2), nlevels (<= 16), edge_threshold (>= 15) and fast_threshold are free.
 * kps: n_images x max_kp epivo_keypoint (cv::KeyPoint's layout: x, y in image coordinates, size = 31 * level scale,
 * angle in degrees, response = FAST score, octave = level, class_id -1) in OpenCV's order (level by level, inside a
 * level the order KeyPointsFilter::retainBest leaves); desc: n_images x max_kp x 32 bytes; counts[i] = keypoints FOUND
 * in image i (ties at a level's budget are all kept, as in OpenCV, so it may exceed nfeatures) -- when it exceeds
 * max_kp only the first max_kp are stored.  Every field and every descriptor bit is identical to OpenCV 4.13's. */
typedef struct epivo_keypoint {
    float x, y, size, angle, response;
    int32_t octave, class_id;
} epivo_keypoint;
int epivo_orb_detect_and_compute(epivo_ctx* ctx, const uint8_t* images, int n_images, int rows, int cols, int nfeatures,
                                 float scale_factor, int nlevels, int edge_threshold, int fast_threshold, int max_kp,
                                 epivo_keypoint* kps, uint8_t* desc, int32_t* counts);

/* The pyramid epivo_orb_detect_and_compute builds for these arguments, without touching a GPU (no context needed):
 * level_rows / level_cols / level_features: nlevels entries each -- size of every level and its retainBest budget, as
 * OpenCV's ORB computes them.  Returns EPIVO_ERR_UNSUPPORTED for the configurations the extractor refuses (a level that
 * rounds to an empty image -- OpenCV asserts there --, nlevels outside [1, 16], scale_factor outside (1, 2]). */
int epivo_orb_level_geometry(int rows, int cols, int nfeatures, float scale_factor, int nlevels, int32_t* level_rows,
                             int32_t* level_cols, int32_t* level_features);

/* K3 alone: Sampson scoring of a fixed hypothesis set of m models (m x 9) against n
 * correspondences with OpenCV's exact inlier rule.  threshold in pixels (RANSAC rule);
 * counts: m inlier counts; medians: m LMedS medians (float32, may be NULL); best: index of
 * the first model with the largest count; best_mask: n bytes {0,1} of that model. */
int epivo_score_sampson(epivo_ctx* ctx, const double* E, int m, const float* p0, const float* p1,
                        int n, const double K[9], double threshold,
                        int32_t* counts, float* medians, int* best, uint8_t* best_mask);

/* ---- P1: cv::recoverPose(E, p0, p1, cam, R, t, mask) ----------------------------------
 * replaces kitti_E.cpp:120, euroc_E.cpp:251, kitti_ba.cpp:245,322,715.  mask: {0,255}. */
int epivo_recover_pose(epivo_ctx* ctx, const double E[9], const float* p0, const float* p1, int n,
                       const double K[9], double dist_thresh, const uint8_t* in_mask,
                       double R[9], double t[3], uint8_t* mask, int* n_good);

/* ---- L4: Levenberg_Marquardt(n_zeta, epsilon, reps, wreps, lambda0, T0s, pr, p_r, lm_res)
 * replaces jac_Rt_gen_.cpp:287-478 (called at kitti_E.cpp:196, kitti_ba.cpp:881,1044).
 * reps: n_rep x 2 int32 (first zeta, last zeta); wreps: n_rep; T0s: n_zeta x 16 row-major,
 * updated in place; pr / p_r: n_rep x N x 3.  epivo_lm_res is the reference's LM_res
 * (used at jac_Rt_gen_.cpp:473-475 but defined nowhere in the reference). */
typedef struct { double H_norm, r_norm, lambda; } epivo_lm_res;
int epivo_lm_rt(epivo_ctx* ctx, int n_zeta, double epsilon, const int32_t* reps, const double* wreps,
                int n_rep, double lambda0, int max_iters, double huber_delta,
                double* T0s, const double* pr, const double* p_r, int N,
                epivo_lm_res* out, int* iters_run);
/* B independent problems of identical shape in one launch (kitti_ba windows sharded per GPU):
 * T0s: B x n_zeta x 16, pr/p_r: B x n_rep x N x 3, wreps: B x n_rep, out: B, iters_run: B. */
int epivo_lm_rt_batch(epivo_ctx* ctx, int B, int n_zeta, double epsilon, const int32_t* reps,
                      const double* wreps, int n_rep, double lambda0, int max_iters,
                      double huber_delta, double* T0s, const double* pr, const double* p_r, int N,
                      epivo_lm_res* out, int32_t* iters_run);

/* ---- fused per-pair pipeline over a frame sequence (the benchmark's hot path) --------
 * frame f = kp_per_frame keypoints (float32 x,y) + descriptors (32 B); pair i = (f_i, f_i+1):
 * match -> gather -> findEssentialMat -> compact -> recoverPose -> fallbacks -> LM -> revert,
 * i.e. the body of the loop kitti_E.cpp:54-201 with the BFMatcher association of
 * kitti_ba.cpp:641-693 in place of the optical-flow front end. */
typedef struct {
    int norm;               /* EPIVO_NORM_HAMMING2            kitti_ba.cpp:602 */
    int match_mode;         /* EPIVO_MATCH_CROSSCHECK         kitti_ba.cpp:602 */
    float ratio;            /* 0.8 (ratio mode only) */
    double K[9];            /* kitti_E.cpp:38-40 */
    int method;             /* EPIVO_RANSAC (kitti.cpp:101) or EPIVO_LMEDS (kitti_E.cpp:101) */
    double prob;            /* 0.99 */
    double threshold;       /* 1.0  (kitti.cpp:103) */
    int max_iters;          /* 1000 (OpenCV default) */
    double dist_thresh;     /* 50   (recoverPose default) */
    double min_trace;       /* 2.7: trace(R) < 3*0.9 -> R = I, t = fallback_t   kitti_E.cpp:128-131 */
    double fallback_t[3];   /* (0.1, 0.1, -0.9)                                  kitti_E.cpp:130 */
    double min_t_norm;      /* 1e-5                                              kitti_E.cpp:133 */
    int lm_points;          /* 48                                                kitti_E.cpp:170 */
    double lm_lambda0;      /* 1e-2                                              kitti_E.cpp:196 */
    double lm_epsilon;      /* 1e-8 */
    int lm_max_iters;       /* 30                                                jac_Rt_gen_.cpp:323 */
    double huber_delta;     /* 1e-5                                              jac_Rt_gen_.cpp:17 */
    double lm_revert;       /* revert T to the recoverPose init if r_norm > this (1e-9, kitti_E.cpp:198) */
} epivo_pipeline_params;
void epivo_pipeline_params_default(epivo_pipeline_params* p);   /* the KITTI values above */

typedef struct {
    double E[9];
    double R[9];            /* recoverPose */
    double t[3];
    double T0[16];          /* LM initial pose after the kitti_E.cpp:128-135 fallbacks */
    double T[16];           /* final pose (LM result, or T0 if reverted / LM not run) */
    epivo_lm_res lm;
    int32_t n_matches, n_inliers, n_good, ransac_iters, n_models, lm_iters;
    int32_t lm_ran;         /* 1 if >= lm_points cheirality-good points existed (kitti_E.cpp:194) */
    int32_t lm_reverted;
} epivo_pair_result;

typedef struct epivo_seq epivo_seq;
int epivo_seq_create(epivo_ctx* ctx, epivo_seq** out, int max_frames, int kp_per_frame);
void epivo_seq_destroy(epivo_seq* seq);
/* host -> device copy of n_frames frames starting at frame slot first_frame (async on the
 * context stream; kps n_frames x kp x 2 f32, descs n_frames x kp x 32 u8) */
int epivo_seq_upload(epivo_seq* seq, int first_frame, int n_frames, const float* kps, const uint8_t* descs);
/* kitti_ba.cpp:114-156 (extract_good_kp) straight into the sequence: ORB (epivo_orb_detect_and_compute's configuration
 * arguments) on n_frames 8-bit images of rows x cols; keypoint positions, descriptors and the per-frame counts go into
 * frame slots first_frame .. first_frame + n_frames - 1 without leaving the device -- the same bytes as
 * epivo_orb_detect_and_compute + KeyPoint::convert + epivo_seq_upload + epivo_seq_set_counts.  A frame with more than
 * kp_per_frame keypoints keeps the first kp_per_frame (OpenCV's order).  counts_out (nullable): keypoints FOUND per frame. */
int epivo_seq_extract_orb(epivo_seq* seq, int first_frame, int n_frames, const uint8_t* images, int rows, int cols,
                          int nfeatures, float scale_factor, int nlevels, int edge_threshold, int fast_threshold,
                          int32_t* counts_out);
/* Real detectors return a different number of keypoints per frame: counts[i] (<= kp_per_frame) keypoints of
 * frame slot first_frame + i are valid (the rest of the slot is ignored).  Default: every slot is full. */
int epivo_seq_set_counts(epivo_seq* seq, int first_frame, int n_frames, const int32_t* counts);
/* Explicit pair list.  kitti_ba.cpp:603-607 does not walk consecutive frames only: it matches
 * (i + window[j].first, i + window[j].second) for every window offset j (e.g. (0,1), (0,2), (1,2), or the
 * left/right frames of a stereo rig).  After this call pair p matches frame fq[p] (query, desc0 of
 * kitti_ba.cpp:630) against frame ft[p] (train, desc1), and run / process / download / get_matches address
 * pairs [0, n_pairs).  epivo_seq_create_pairs gives room for more pairs than max_frames - 1.
 * n_pairs = 0 or NULL lists restore the default (p, p + 1).  epivo_seq_cloud's pose chain assumes consecutive pairs. */
int epivo_seq_create_pairs(epivo_ctx* ctx, epivo_seq** out, int max_frames, int kp_per_frame, int max_pairs);
int epivo_seq_set_pairs(epivo_seq* seq, int n_pairs, const int32_t* fq, const int32_t* ft);
/* enqueue the pipeline for pairs [first_pair, first_pair + n_pairs) (async) */
int epivo_seq_run(epivo_seq* seq, const epivo_pipeline_params* p, int first_pair, int n_pairs);
/* The reference-facing call with HOST buffers: upload n_frames frames (kps n_frames x kp x 2 f32,
 * descs n_frames x kp x 32 u8, ideally pinned), run all n_frames-1 pairs, copy the results back
 * and synchronise.  The upload is pipelined under the matcher on a second (copy) stream. */
int epivo_seq_process(epivo_seq* seq, const epivo_pipeline_params* p, int n_frames, const float* kps,
                      const uint8_t* descs, epivo_pair_result* out);
/* The same geometry for correspondences the caller already has -- the LK tracks with status 1 of kitti_E.cpp:86-95,
 * euroc_E.cpp:190-196 -- instead of descriptor matches: pair i has counts[i] point pairs p0[i][k] -> p1[i][k]
 * (n_pairs x max_pts x 2 floats each, pixels; max_pts <= kp_per_frame of the sequence object).  Runs
 * findEssentialMat -> recoverPose -> fallbacks -> LM for pairs [0, n_pairs) and returns the results (n_matches =
 * counts[i]); epivo_seq_get_masks / epivo_seq_cloud work on them as after epivo_seq_process. */
int epivo_seq_process_points(epivo_seq* seq, const epivo_pipeline_params* p, int n_pairs, const float* p0, const float* p1,
                             const int32_t* counts, int max_pts, epivo_pair_result* out);
/* The loop body of kitti_E.cpp:54-201 / kitti.cpp / euroc_E.cpp:169-208 from 8-bit frames, on the device:
 * [remap] -> FastFeatureDetector(fast_threshold, nonmax) on the first frame of every pair -> calcOpticalFlowPyrLK
 * (21x21, maxLevel 3, 30 iterations, eps 0.01, minEig 1e-4, err passed: the reference's defaults) into the second
 * frame -> keep the tracks with status 1, in corner order -> findEssentialMat -> recoverPose -> fallbacks -> LM.
 * Pairs: consecutive (p, p+1) or the list of epivo_seq_set_pairs.  map_xy/map_frac: NULL, or the fixed-point maps
 * of epivo_remap (drows x dcols; BORDER_CONSTANT 0), applied to every frame first.  A frame with more than
 * kp_per_frame corners tracks the first kp_per_frame (OpenCV's order).  corners_out (nullable, n_frames entries):
 * corners FAST found per frame.  out: one epivo_pair_result per pair, n_matches = tracks kept.
 * images: n_frames x rows x cols, dense.  The front end runs in windows of at most 256 frames that overlap by the
 * largest |ft - fq| of the pair list; a list whose span does not fit a window returns EPIVO_ERR_UNSUPPORTED.
 * Afterwards epivo_seq_get_masks and epivo_seq_cloud work as after epivo_seq_process_points, and
 * epivo_seq_get_matches reports for every kept track the index of its corner in the query frame's FAST list
 * (query_idx == train_idx, dist 0). */
int epivo_seq_process_frames(epivo_seq* seq, const epivo_pipeline_params* p, int n_frames, const uint8_t* images,
                             int rows, int cols, const int16_t* map_xy, const uint16_t* map_frac, int drows, int dcols,
                             int fast_threshold, int32_t* corners_out, epivo_pair_result* out);
/* after epivo_seq_process_frames: the kept tracks of one pair in pixels (the reference's _cpt0 / _cpt1_), n_out x 2
 * floats each (capacity kp_per_frame); EPIVO_ERR_INVALID unless the last run was epivo_seq_process_frames */
int epivo_seq_get_points(epivo_seq* seq, int pair, float* p0, float* p1, int* n_out);
/* device -> host copy of the results of the last run and stream sync */
int epivo_seq_download(epivo_seq* seq, epivo_pair_result* out, int first_pair, int n_pairs);
/* per-stage device time of the last run (CUDA events on the context stream), ms:
 * [0] total [1] match [2] presolve (part of 3) [3] essential [4] pose [5] lm [6] finish [7] matcher tile kernel alone
 * [8] number of pair groups; the geometry runs after the matcher, but epivo_seq_process's matcher pieces alternate
 * between two streams, so there [1] and [7] count the time two pieces overlap twice. */
int epivo_seq_stage_ms(epivo_seq* seq, float* ms, int n);
/* debug/parity views of the last run, host copies: matches of one pair */
int epivo_seq_get_matches(epivo_seq* seq, int pair, int32_t* query_idx, int32_t* train_idx,
                          int32_t* dist, int* n_out);
int epivo_seq_get_masks(epivo_seq* seq, int pair, uint8_t* e_mask, int* n_e, uint8_t* pose_mask, int* n_pose);

/* ---- N3: windowed bundle adjustment over the pairs of the last run (mono) ----------------
 * kitti_ba.cpp:757-905 (bundle_adjustment, mono) over the pairs of the last epivo_seq_run / epivo_seq_process /
 * epivo_seq_process_frames, without leaving the device: the reprojections of match_kp (kitti_ba.cpp:583-755) are
 * gathered from the pair data that run left, and every window's LM runs in one batched launch.
 * window: n_rep offsets (first[j], second[j]) (kitti_ba.cpp:1131-1144, e.g. (0,1),(0,2),(1,2)); windows start at
 * i = 0, stride, 2*stride, ... while i + max offset < num_frames (:780-801).  For window i, rep j uses the pair
 * (i + first[j], i + second[j]) and the chain uses (i + lo + k, i + lo + k + 1), k < n_zeta = hi - lo (lo / hi: the
 * smallest / largest offset).  All of these must be in the pair list -- a key listed twice means its first entry --
 * and in the last run.  Per pair: fewer than 8 matches or no E-inlier -> R = I, t = (0.1, 0.1, -0.9) and no points
 * (:741-744), else recoverPose's R, t and the matches (kept tracks) that are E-inliers with rec_mask == 255, in order;
 * a rep gets its pair's first 32 such points, K-normalised as cam_ * (u, v, 1), or weight 0 with fewer (:819-824).
 * LM: epsilon 1e-8, lambda0 1e-2, 30 iterations, N = 32 (:881).  Then the reference's sequential tail on the host:
 * a window with r_norm > 1e-2 keeps its initial chain (:889-891), translations are divided by the norm of the
 * translation of the window's first frame when an earlier window optimized it (:853-856, 898-901), later windows
 * overwrite the overlap.  The result equals ba.match_kp followed by ba.bundle_adjustment(stereo=False).
 * Kinv: the 3x3 inverse intrinsics, row-major (the driver's cam_).  opt_T: num_frames x 16 (identity where no window
 * reaches).  win_T (n_zeta x 16 per window, the LM's chains before the revert rule) / lm / iters / reverted (nullable):
 * per window, at most (num_frames + stride - 1) / stride entries; *n_windows: the number of windows.
 * Refused before any launch: EPIVO_ERR_INVALID for a missing pair (named in the message), a pair outside the last run,
 * first[j] == second[j], a negative offset, stride < 1, num_frames outside [2, max_frames], a last run of
 * epivo_seq_process_points or no run over the current pair list; EPIVO_ERR_UNSUPPORTED for a window whose LM does not
 * fit in shared memory (n_zeta > 18 or so).  No window fits: identity opt_T, *n_windows = 0, nothing launched. */
int epivo_seq_bundle_adjust(epivo_seq* seq, int n_rep, const int32_t* first, const int32_t* second, int stride,
                            int num_frames, const double Kinv[9], double huber_delta, double* opt_T, double* win_T,
                            epivo_lm_res* lm, int32_t* iters, uint8_t* reverted, int32_t* n_windows);

/* ---- N3: windowed bundle adjustment over the pairs of the last run (stereo) --------------
 * kitti_ba.cpp:908-1068 (bundle_adjustment_stereo): epivo_seq_bundle_adjust with the stereo node layout.  Frame f of
 * the rig is node 2f (left) and node 2f + 1 (right); the frame slots of the sequence are the nodes, so the last run
 * covered 2 * num_frames slots.  window: the driver's n_rep frame offsets (first[j], second[j]), e.g. (0,1),(0,2),(1,2);
 * each entry (a, b) becomes the three node reps (2a, 2b), (2a+1, 2b), (2a, 2a+1) (:934-941), so ws = 3 has 9 reps over
 * n_zeta = 4 nodes.  stride is in frames: windows start at frame i = 0, stride, ... while 2i + the largest node offset
 * < 2 * num_frames (:943-963), and use the node pairs (2i + a', 2i + b') of the expanded reps and the chain
 * (2i + lo + k, 2i + lo + k + 1).  The pair list that holds every key the windows read, chain pairs (2f+1, 2f+2)
 * included, is ba.window_pairs(ba.expand_stereo_window(window), 2 * stride, 2 * num_frames).
 * pair_w (nullable): one weight per entry of the current pair list, indexed as epivo_seq_set_pairs -- the reproj.w of
 * that pair; NULL is 1.0 everywhere.  The driver sets 0 on the left -> right pairs (2f, 2f+1) to freeze the rig
 * extrinsics (:171-172, :1000-1008).  A rep with 32 points weighs its pair's pair_w and carries its real K-normalised
 * rows even when that weight is 0; a rep with fewer weighs 0 with all-ones rows.  A key listed twice uses its first
 * entry, for the points and the weight alike.  The selection, fallbacks, LM and revert rule are the mono call's; there is
 * no scale carry (:1054-1066): later windows overwrite the overlap with their chains unscaled.  The result equals
 * ba.match_kp with each reproj.w set from pair_w, followed by ba.bundle_adjustment(stereo=True).
 * opt_T: 2 * num_frames x 16 (identity where no window reaches).  win_T / lm / iters / reverted / *n_windows as in the
 * mono call.  Refused before any launch: everything the mono call refuses, with num_frames outside [2, max_frames / 2]
 * and a window offset of max_frames / 2 or more; a non-finite pair_w entry (EPIVO_ERR_INVALID).  EPIVO_ERR_UNSUPPORTED
 * when the expanded window's LM does not fit (n_zeta = 2 * the largest frame offset, in nodes).  No window fits:
 * identity opt_T for the 2 * num_frames nodes, *n_windows = 0, nothing launched. */
int epivo_seq_bundle_adjust_stereo(epivo_seq* seq, int n_rep, const int32_t* first, const int32_t* second, int stride,
                                   int num_frames, const double* pair_w, const double Kinv[9], double huber_delta,
                                   double* opt_T, double* win_T, epivo_lm_res* lm, int32_t* iters, uint8_t* reverted,
                                   int32_t* n_windows);

/* ---- N2: pose chain + depth / point cloud of the last run (kitti_E.cpp:203-254, euroc_E.cpp:303-349) ----
 * For the pairs [first_pair, +n_pairs) of the last epivo_seq_run / epivo_seq_process:
 *   dT_i     = [R_i | t_i/|t_i| * scales[i]]   (refined pose, GT-scaled translation; scales NULL = 1)
 *   poses[i] = the chained camera pose BEFORE pair i (all_T, kitti_E.cpp:227), poses[n_pairs] the last
 *              one: (n_pairs + 1) x 16 doubles, starting from identity, cT <- cT * dT^-1
 *   points   = for every E-inlier of every pair, in order, the reference's depth-from-parallax point
 *              X = poses[i] * (d * K^-1 x0) with d = |P t| / |P R K^-1 x0|, kept iff |P R K^-1 x0| > 1e-2
 *   limits[i]= number of cloud points before pair i (the reference's `limits`), n_pairs entries
 * points may be NULL (or cap 0) to get only poses / limits / *n_points; at most cap points are written. */
int epivo_seq_cloud(epivo_seq* seq, const double* scales, int first_pair, int n_pairs, double* poses,
                    double* points, int64_t cap, int64_t* limits, int64_t* n_points);

/* D1 alone, for a sequence sharded over several GPUs (SURVEY 8e): T_pairs = the refined 4x4 of every pair in sequence
 * order (n x 16, host; what the ranks all-gather), scales = GT step lengths or NULL; poses = (n + 1) x 16 chained camera
 * poses starting from identity, cT <- cT * dT^-1 with dT = [R | t/|t| * scale] (kitti_E.cpp:218-228), computed by the
 * same device block scan as epivo_seq_cloud. */
int epivo_chain_poses(epivo_ctx* ctx, const double* T_pairs, const double* scales, int n, double* poses);

/* ---- pipe micro-benchmarks (roofline denominators MEASURED_PEAKS.json lacks) ----------
 * which: 0 POPC.32, 1 LOP3, 2 FP64 FMA, 3 FP32 FMA, 4 IADD3, 5 FP64 MMA m8n8k4 (in FMA);
 * result = thread-ops / s on the whole GPU */
int epivo_microbench(epivo_ctx* ctx, int which, double* ops_per_sec);

#ifdef __cplusplus
}
#endif
#endif /* EPIVO_B200_H */
