// Declarations of the per-stage launchers shared by api.cu and seq.cu.  All pointers are
// DEVICE pointers; launches go to ctx->stream.
#pragma once
#include "common.cuh"

// ---- essential.cu --------------------------------------------------------------------
struct EssentialPlan {
    int n_pairs, stride;
    const double* xn;        // [pair][4][stride]
    const int32_t* n;        // [pair]
    int method;
    double prob, thresh;     // thresh = pixel threshold / ((fx+fy)/2)
    int max_iters;
    const int32_t* samples;  // optional [m][5]
    int m;
    float* errbuf;           // epv_essential_errbuf_floats() floats (LMedS scratch)
    double* E;               // [pair][9]
    uint8_t* mask;           // [pair][stride]
    int32_t *n_inliers, *iters, *n_models, *status;   // [pair]
    double* xin;             // optional [pair][4][stride]
    void* work;              // device scratch of epv_essential_work_bytes(n_pairs) bytes
    size_t work_bytes;
    cudaEvent_t ev_presolved = nullptr;   // optional: recorded after the first round's sample + solve kernels
};
size_t epv_essential_work_bytes(int n_pairs);
int epv_essential_launch(epivo_ctx* ctx, const EssentialPlan& p);
size_t epv_essential_errbuf_floats(int n_pairs, int stride);
int epv_normalize_launch(epivo_ctx* ctx, const float* d_p0, const float* d_p1, int n, int stride, const double K[9],
                         double* d_xn);
int epv_five_point_launch(epivo_ctx* ctx, const double* d_x1, const double* d_x2, int m, double* d_rec /* m x 96 */,
                          uint32_t* d_items /* m x 10 */, double* d_item_z /* m x 10 */, int32_t* d_count /* 1 */,
                          double* d_E /* m x 10 x 9 */, uint32_t* d_flags /* m */);
int epv_score_launch(epivo_ctx* ctx, const double* d_E, int m, const double* d_xn, int stride, int n, double thresh,
                     int32_t* d_counts, float* d_medians, float* d_errbuf, int* d_best, uint8_t* d_mask);

// ---- pose.cu -------------------------------------------------------------------------
struct PosePlan {
    int n_pairs, stride;
    const double* E;         // [pair][9]
    const double* xn;        // [pair][4][stride] K-normalised points (the E inliers)
    const int32_t* n;        // [pair]
    const uint8_t* in_mask;  // optional [pair][stride]
    double dist_thresh;
    double* R;               // [pair][9]
    double* t;               // [pair][3]
    uint8_t* mask;           // [pair][stride] {0,255}
    int32_t* n_good;         // [pair]
    const int32_t* skip;     // optional [pair]: nonzero status => pair skipped (outputs zeroed)
};
int epv_pose_launch(epivo_ctx* ctx, const PosePlan& p);
int epv_eight_point_launch(epivo_ctx* ctx, const double* d_x1, const double* d_x2, int m, double* d_E, int32_t* d_ok);

// ---- lm.cu ---------------------------------------------------------------------------
struct LmPlan {
    int B;                   // independent problems
    int n_zeta, n_rep, N;
    const int32_t* reps;     // [n_rep][2] (shared by all problems)
    const double* wreps;     // [B][n_rep]
    double epsilon, lambda0, huber_delta;
    int max_iters;
    double* T0s;             // [B][n_zeta][16] in/out
    const double* pr;        // [B][n_rep][N][3]
    const double* p_r;       // [B][n_rep][N][3]
    epivo_lm_res* out;       // [B]
    int32_t* iters;          // [B]
    const int32_t* active;   // optional [B]: 0 => problem skipped, T0s untouched
    int single_pair;         // caller asserts reps == {(0,0)}: warp-per-problem kernel when n_zeta == 1, N <= 64
};
int epv_lm_launch(epivo_ctx* ctx, const LmPlan& p);
// epv_lm_launch's refusals for a problem with N <= 32 points per rep (the shape it then picks, 64 x 32, unless
// EPIVO_LM_SHAPE overrides it), without launching: for callers that check everything before their first launch
int epv_lm_check_n32(epivo_ctx* ctx, int n_zeta, int n_rep);

// ---- cloud.cu (N2: pose chain + per-inlier depth / point cloud, kitti_E.cpp:203-254) ------
int epv_chain_launch(epivo_ctx* ctx, const epivo_pair_result* d_res, const double* d_scales, int n, double* d_poses);
int epv_cloud_launch(epivo_ctx* ctx, int n_pairs, int stride, const epivo_pair_result* d_res, const double* d_scales,
                     const double* d_poses, const double* d_xin, const int32_t* d_ninl, int32_t* d_counts,
                     int64_t* d_limits, double* d_points, int64_t cap, int pass);

// ---- frontend.cu (N4: FAST-9/16 detector, kitti_E.cpp:71-74) ---------------------------------
size_t epv_fast_work_bytes(int n_images, int rows, int cols);
int epv_fast_launch(epivo_ctx* ctx, const uint8_t* d_img, int n_images, int rows, int cols, int threshold, int nonmax,
                    int max_kp, float* d_kps, float* d_resp, int32_t* d_counts, void* work);
size_t epv_lk_work_bytes(int n_frames, int rows, int cols, int max_level);
int epv_lk_launch(epivo_ctx* ctx, const uint8_t* d_images, int n_frames, int rows, int cols, const float* d_pts,
                  const int32_t* d_counts, int max_pts, int max_level, int max_count, double epsilon, double min_eig,
                  float* d_next, uint8_t* d_status, float* d_err /* nullable */, void* work);
// the two halves of epv_lk_launch, for callers that track a pair list over a batch of frames
int epv_lk_pyramids(epivo_ctx* ctx, const uint8_t* d_images, int n_frames, int rows, int cols, int max_level, int n_deriv,
                    void* work);
int epv_lk_track_launch(epivo_ctx* ctx, const void* work, int n_frames, int rows, int cols, int max_level, int n_pairs,
                        const int32_t* d_pair_frames /* nullable */, const float* d_pts, const int32_t* d_counts, int max_pts,
                        int max_count, double epsilon, double min_eig, float* d_next, uint8_t* d_status, float* d_err);
int epv_remap_launch(epivo_ctx* ctx, const uint8_t* d_img, int n_images, int rows, int cols, const int16_t* d_map_xy,
                     const uint16_t* d_map_frac, int drows, int dcols, int border, uint8_t* d_out);

// ---- orb.cu (N4: cv::ORB::detectAndCompute, kitti_ba.cpp:128-152) ------------------------------
struct EpvOrbPlan {
    alignas(8) char geom[704];          // OrbGeom (orb.cu): level sizes, scales, budgets, buffer offsets
    size_t pyr_bytes;                   // pyramid bytes for the whole batch (level 0 block first)
    size_t cand_total;                  // candidate slots over all levels and images
    size_t tab_entries;                 // words of the resize weight tables
};
int epv_orb_plan(epivo_ctx* ctx, int n_images, int rows, int cols, int nfeatures, float scale_factor, int nlevels,
                 int edge_threshold, int max_kp, EpvOrbPlan* plan);
size_t epv_orb_work_bytes(const EpvOrbPlan& plan);
int epv_orb_launch(epivo_ctx* ctx, const EpvOrbPlan& plan, int fast_threshold, uint8_t* d_pyr, void* d_kps,
                   uint8_t* d_desc, int32_t* d_counts, uint32_t* h_tab);
