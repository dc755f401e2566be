// Fused per-pair pipeline over a device-resident frame sequence (the benchmark's hot path):
//   match (K1) -> gather + K-normalise -> findEssentialMat (K2+K3) -> inlier compaction ->
//   recoverPose (K4) -> kitti_E.cpp:128-135 fallbacks -> Levenberg_Marquardt (K5) -> revert rule.
// This is the body of the reference loop kitti_E.cpp:54-201 with the BFMatcher association
// of kitti_ba.cpp:641-693 as the correspondence source.  Pairs are processed in chunks so
// that a chunk's intermediates (keys, matches, normalised points, masks) stay L2-resident;
// everything is enqueued on the context stream with no host synchronisation in between.
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <unordered_map>
#include <vector>

#include "common.cuh"
#include "stages.cuh"

namespace {
constexpr int SEQ_CHUNK = 8192;          // pairs per launch group (single stream: large groups, fewer tails)
constexpr int SEQ_CHUNK_OVERLAP = 1024;  // group size when the two-stream pipelining is switched on
constexpr int SEQ_STAGES = 7;      // prep, match, finalize, essential, pose, lm, (total)
constexpr int SEQ_MAX_CHUNKS = 256;
}  // namespace

struct epivo_seq {
    epivo_ctx* ctx = nullptr;
    int max_frames = 0, kp = 0, stride = 0, chunk = SEQ_CHUNK;
    // frames
    float* d_kps = nullptr;
    uint32_t* d_desc = nullptr;
    uint32_t* d_planes = nullptr;
    int32_t* d_counts = nullptr;     // keypoints actually present in every frame slot (<= kp)
    bool counts_set = false;
    // pair list: pair p matches frame fq[p] (query) against frame ft[p] (train); the default is (p, p + 1).
    // kitti_ba.cpp:603-607 walks (i + window[j].first, i + window[j].second) -- an arbitrary list of this kind
    int32_t *d_fq = nullptr, *d_ft = nullptr;
    bool pairs_set = false;
    int max_pairs = 0, n_list = 0;   // capacity / pairs currently addressable
    int frames_hi = 0;               // frames [0, frames_hi) have been uploaded (plane pre-pass range in list mode)
    int list_max = 0;                // largest frame index the pair list references
    std::vector<int32_t> h_fq, h_ft; // host copy of the pair list (epivo_seq_process_frames plans its windows from it)
    // per pair, whole sequence
    int32_t *d_mq = nullptr, *d_mt = nullptr, *d_md = nullptr, *d_nmatch = nullptr;
    uint8_t *d_emask = nullptr, *d_pmask = nullptr;
    double *d_E = nullptr, *d_R = nullptr, *d_t = nullptr, *d_T = nullptr, *d_T0 = nullptr;
    int32_t *d_ninl = nullptr, *d_iters = nullptr, *d_nmodels = nullptr, *d_status = nullptr, *d_ngood = nullptr;
    int32_t *d_lmactive = nullptr, *d_lmiters = nullptr;
    epivo_lm_res* d_lmres = nullptr;
    epivo_pair_result* d_results = nullptr;
    // per chunk
    uint32_t *d_rowkey = nullptr, *d_rowkey2 = nullptr, *d_colkey = nullptr;
    double *d_xn = nullptr, *d_xin = nullptr, *d_lmp = nullptr, *d_lmq = nullptr, *d_w = nullptr;
    float* d_err = nullptr;
    int32_t* d_reps = nullptr;
    char* d_esswork = nullptr;      // essential-stage scratch for one pair group
    size_t esswork_bytes = 0;
    // host staging for results
    epivo_pair_result* h_results = nullptr;
    // timing
    cudaEvent_t ev[SEQ_MAX_CHUNKS][SEQ_STAGES] = {};
    cudaEvent_t evk[SEQ_MAX_CHUNKS][2] = {};     // around the matcher tile kernel alone
    cudaEvent_t evp[SEQ_MAX_CHUNKS] = {};        // after sample + presolve
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
    cudaStream_t stream2 = nullptr;          // geometry stream (FP64 kernels) -- overlaps the integer-bound matcher
    cudaStream_t stream3 = nullptr;          // host-buffer path: every other matcher piece (see seq_execute)
    cudaStream_t stream4 = nullptr;          // host-buffer path, copy-bound regime: geometry of the groups already matched
    cudaEvent_t ev_piece[SEQ_MAX_CHUNKS] = {};   // matcher piece c (tiles + finalize) complete
    int geo_mode = 0;                        // 2: geometry between the matcher pieces of the host-buffer path (epivo_seq_set_overlap)
    cudaEvent_t ev_matched[SEQ_MAX_CHUNKS] = {};
    cudaEvent_t ev_geo_done = nullptr;
    int overlap = 0;   // measured on B200: co-running the matcher and the FP64 kernels gains nothing (see DESIGN.md)
    int match_pad = 0;
    int last_mgroups = 0, last_ggroups = 0;
    int last_n_pairs = 0, last_first = 0;
    // epivo_seq_process_frames: the kept tracks of every pair in pixels, [pair][p0 | p1][stride][2] floats (allocated by
    // the first call); last_frames: the last run was process_frames, so epivo_seq_get_points may read them
    float* d_trk = nullptr;
    bool last_frames = false;
    // what the last run left on the device for the pairs [last_first, +last_n_pairs) of the current pair list:
    // matches into the frame slots' keypoints (run / process), kept tracks in d_trk (process_frames), or caller points
    // that were not kept (process_points).  epivo_seq_bundle_adjust reads pixels from the first two, through the frames
    // of the pair list, so unlike last_frames this is reset by epivo_seq_set_pairs.
    enum { RUN_NONE, RUN_DESC, RUN_POINTS, RUN_FRAMES } last_run = RUN_NONE;
    std::vector<void*> allocs;
};

namespace {

template <typename T>
int seq_alloc(epivo_seq* s, T** p, size_t count) {
    epivo_ctx* ctx = s->ctx;
    void* q = nullptr;
    EPV_CUDA(ctx, cudaMalloc(&q, std::max<size_t>(count, 1) * sizeof(T)));
    s->allocs.push_back(q);
    *p = reinterpret_cast<T*>(q);
    return EPIVO_OK;
}

// After recoverPose: the reference's sanity fallbacks, LM input assembly (first lm_points
// compacted E-inliers, gated on >= lm_points cheirality-good points; kitti_E.cpp:170-194).
__global__ void lm_prep_kernel(int n_pairs, int stride, epivo_pipeline_params prm, const double* __restrict__ R,
                               const double* __restrict__ t, const int32_t* __restrict__ status,
                               const int32_t* __restrict__ n_inl, const int32_t* __restrict__ n_good,
                               const double* __restrict__ xin, double* __restrict__ T0, double* __restrict__ T,
                               double* __restrict__ lmp, double* __restrict__ lmq, double* __restrict__ w,
                               int32_t* __restrict__ active) {
    const int pair = blockIdx.x;
    if (pair >= n_pairs) return;
    const int tid = threadIdx.x;
    const int N = prm.lm_points;
    __shared__ double sT[16];
    if (tid == 0) {
        double Rm[9], tv[3];
        for (int i = 0; i < 9; ++i) Rm[i] = R[(int64_t)pair * 9 + i];
        for (int i = 0; i < 3; ++i) tv[i] = t[(int64_t)pair * 3 + i];
        const bool ok = status[pair] == 0;
        if (!ok || (Rm[0] + Rm[4] + Rm[8]) < prm.min_trace) {            // kitti_E.cpp:128-131
            for (int i = 0; i < 9; ++i) Rm[i] = (i % 4 == 0) ? 1.0 : 0.0;
            for (int i = 0; i < 3; ++i) tv[i] = prm.fallback_t[i];
        }
        if (sqrt(tv[0] * tv[0] + tv[1] * tv[1] + tv[2] * tv[2]) < prm.min_t_norm)   // kitti_E.cpp:133-135
            for (int i = 0; i < 3; ++i) tv[i] = prm.fallback_t[i];
        for (int i = 0; i < 3; ++i) {
            for (int j = 0; j < 3; ++j) sT[i * 4 + j] = Rm[i * 3 + j];
            sT[i * 4 + 3] = tv[i];
        }
        sT[12] = sT[13] = sT[14] = 0.0;
        sT[15] = 1.0;
        // kitti_E.cpp:170-194: N = min(48, #E-inliers) (asserted >= 48), LM runs iff 48 of the
        // recoverPose mask entries are 255
        active[pair] = (ok && n_inl[pair] >= N && n_good[pair] >= N) ? 1 : 0;
        w[pair] = 1.0;
    }
    __syncthreads();
    if (tid < 16) {
        T0[(int64_t)pair * 16 + tid] = sT[tid];
        T[(int64_t)pair * 16 + tid] = sT[tid];
    }
    // rows j_ = 0..N-1 of the compacted inlier list (kitti_E.cpp:176-182 indexes cpt0[N_mask])
    const double* x = xin + (int64_t)pair * 4 * stride;
    for (int i = tid; i < N; i += blockDim.x) {
        const bool have = i < n_inl[pair];
        double* p = lmp + ((int64_t)pair * N + i) * 3;
        double* q = lmq + ((int64_t)pair * N + i) * 3;
        p[0] = have ? x[i] : 1.0;
        p[1] = have ? x[stride + i] : 1.0;
        p[2] = 1.0;
        q[0] = have ? x[2 * stride + i] : 1.0;
        q[1] = have ? x[3 * stride + i] : 1.0;
        q[2] = 1.0;
    }
}

// pixel -> K-normalised float64 coordinate, x = u / fx - cx / fx as the one fused scale-and-shift OpenCV's convertTo
// computes (a = 1 / fx, b = -cx * a); every kernel that feeds the geometry with tracks calls this one function
__device__ __forceinline__ double knorm(float u, double a, double b) { return __fma_rn((double)u, a, b); }

// correspondences supplied by the caller (LK tracks, kitti_E.cpp:86-95) instead of descriptor matches: the same
// pixel -> K-normalised float64 step the matcher's finalize kernel ends with, for a batch of pairs
__global__ void __launch_bounds__(256) points_in_kernel(const float* __restrict__ p0, const float* __restrict__ p1,
                                                        const int32_t* __restrict__ counts, int max_pts, int stride,
                                                        double ax, double bx, double ay, double by,
                                                        double* __restrict__ xn, int32_t* __restrict__ nmatch,
                                                        int32_t* __restrict__ mq, int32_t* __restrict__ mt) {
    const int pair = blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
    const int n = min(max(counts[pair], 0), max_pts);
    if (i == 0) nmatch[pair] = n;
    if (i >= n) return;
    const float2 a = reinterpret_cast<const float2*>(p0)[(size_t)pair * max_pts + i];
    const float2 b = reinterpret_cast<const float2*>(p1)[(size_t)pair * max_pts + i];
    double* x = xn + (size_t)pair * 4 * stride;
    x[i] = knorm(a.x, ax, bx);
    x[stride + i] = knorm(a.y, ay, by);
    x[2 * stride + i] = knorm(b.x, ax, bx);
    x[3 * stride + i] = knorm(b.y, ay, by);
    mq[(size_t)pair * stride + i] = i;           // epivo_seq_get_matches then reports the identity association
    mt[(size_t)pair * stride + i] = i;
}

// kitti_E.cpp:86-95 on the device: one CTA per pair of a frame window keeps the LK tracks with status 1, in corner
// order (ballot / popc offsets per warp, a running carry over the CTA), and writes them where the geometry reads
// correspondences -- the same outputs as points_in_kernel on the filtered point lists.  meta: the window's pairs as
// [previous frame][n], [next frame][n], [sequence pair index][n]; kps / found: the window's FAST corners and counts.
__global__ void __launch_bounds__(256) track_compact_kernel(const int32_t* __restrict__ meta, int n, const float* __restrict__ kps,
                                                            const int32_t* __restrict__ found, int kp,
                                                            const float* __restrict__ next, const uint8_t* __restrict__ status,
                                                            int stride, double ax, double bx, double ay, double by,
                                                            float* __restrict__ trk, double* __restrict__ xn,
                                                            int32_t* __restrict__ nmatch, int32_t* __restrict__ mq,
                                                            int32_t* __restrict__ mt, int32_t* __restrict__ md) {
    __shared__ int s_warp[8];
    __shared__ int s_carry;
    const int j = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int fq = meta[j], pair = meta[2 * n + j];
    const int cnt = min(found[fq], kp);
    const float2* c = reinterpret_cast<const float2*>(kps) + (size_t)fq * kp;
    const float2* nx = reinterpret_cast<const float2*>(next) + (size_t)j * kp;
    const uint8_t* st = status + (size_t)j * kp;
    float2* t0 = reinterpret_cast<float2*>(trk) + (size_t)pair * 2 * stride;
    float2* t1 = t0 + stride;
    double* x = xn + (size_t)pair * 4 * stride;
    const size_t mo = (size_t)pair * stride;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < cnt; base += 256) {
        const int i = base + tid;
        const bool keep = i < cnt && st[i] == 1;
        const unsigned bal = __ballot_sync(0xFFFFFFFFu, keep);
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        int off = s_carry, total = 0;
        for (int w = 0; w < 8; ++w) {
            off += w < warp ? s_warp[w] : 0;
            total += s_warp[w];
        }
        if (keep) {
            const int k = off + __popc(bal & ((1u << lane) - 1));
            const float2 a = c[i], b = nx[i];
            t0[k] = a;
            t1[k] = b;
            x[k] = knorm(a.x, ax, bx);
            x[stride + k] = knorm(a.y, ay, by);
            x[2 * stride + k] = knorm(b.x, ax, bx);
            x[3 * stride + k] = knorm(b.y, ay, by);
            mq[mo + k] = i;                   // the track's corner in the query frame's FAST list
            mt[mo + k] = i;
            md[mo + k] = 0;
        }
        __syncthreads();
        if (tid == 0) s_carry += total;
        __syncthreads();
    }
    if (tid == 0) nmatch[pair] = s_carry;
}

// ---- windowed bundle adjustment (epivo_seq_bundle_adjust) -------------------------------------------------------------
constexpr int BA_MIN_PT = 32;     // kitti_ba.cpp:777: points per reprojection

struct BaKinv { double k[9]; };   // cam_, the inverse intrinsics, row-major

// one row of cam_ * Vector3d(u, v, 1) as Eigen evaluates it (and ba.normalize's h @ Kinv.T): two products, two sums
__device__ __forceinline__ double ba_knorm_row(const double* k, double u, double v) {
    return __dadd_rn(__dadd_rn(__dmul_rn(k[0], u), __dmul_rn(k[1], v)), k[2]);
}

// the pair has a recoverPose estimate and points (ba.match_kp; kitti_ba.cpp:741-744 otherwise)
__device__ __forceinline__ bool ba_pair_used(const int32_t* nmatch, const int32_t* ninl, int p) {
    return nmatch[p] >= 8 && ninl[p] > 0;
}

// ba.match_kp + ba.assemble on the device: one CTA per (rep j, window b) reads pair p = tab[b][j] of the last run.
// Its reprojection points are the matches (kept tracks) that are E-inliers AND whose recoverPose mask entry -- indexed by
// the inlier's ordinal -- is 255, in match order; the first 32 are K-normalised into pr / p_r[b][j].  A scan of 256 entries
// at a time takes two ballot / popc prefixes (inlier ordinal, kept ordinal) with running carries, and stops once 32 are
// kept.  Fewer than 32 kept (or a pair without points): weight 0 and all-ones rows (kitti_ba.cpp:819-824), decided after
// the scan, so no row is ever half written.  32 kept: the rows, and the weight pw[p] (stereo: the pair's reproj.w, which
// is 0 on the left -> right pairs, kitti_ba.cpp:1000-1008), or 1 when pw is NULL (mono).  The rep-0 CTA of a window also
// writes the window's initial chain from the (j, j+1) pairs tab[B * n_rep + b * n_zeta + k] into T0 (kept for the revert
// rule) and T (the LM's in/out chain).
// Pixels: trk != NULL -> the kept tracks of process_frames, else the keypoints of the matched frame slots.
__global__ void __launch_bounds__(256) ba_assemble_kernel(const int32_t* __restrict__ tab, int n_rep, int n_zeta, int stride,
                                                          int kp, BaKinv ki, const int32_t* __restrict__ nmatch,
                                                          const int32_t* __restrict__ ninl, const uint8_t* __restrict__ emask,
                                                          const uint8_t* __restrict__ pmask, const double* __restrict__ R,
                                                          const double* __restrict__ t, const int32_t* __restrict__ fq,
                                                          const int32_t* __restrict__ ft, const int32_t* __restrict__ mq,
                                                          const int32_t* __restrict__ mt, const float* __restrict__ kps,
                                                          const float* __restrict__ trk, const double* __restrict__ pw,
                                                          double* __restrict__ T0,
                                                          double* __restrict__ T, double* __restrict__ pr,
                                                          double* __restrict__ p_r, double* __restrict__ w) {
    __shared__ int s_warp[2][8];
    __shared__ int s_inl, s_keep;
    __shared__ double s_rows[BA_MIN_PT][6];
    const int j = blockIdx.x, b = blockIdx.y, B = gridDim.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned below = (1u << lane) - 1u;
    const int p = tab[(size_t)b * n_rep + j];
    const bool used = ba_pair_used(nmatch, ninl, p);
    const int nm = used ? nmatch[p] : 0, ni = used ? ninl[p] : 0;
    const size_t o = (size_t)p * stride;
    const float2* kq = reinterpret_cast<const float2*>(kps) + (size_t)fq[p] * kp;
    const float2* kt = reinterpret_cast<const float2*>(kps) + (size_t)ft[p] * kp;
    const float2* t0 = trk ? reinterpret_cast<const float2*>(trk) + (size_t)p * 2 * stride : nullptr;
    if (tid == 0) { s_inl = 0; s_keep = 0; }
    __syncthreads();
    for (int base = 0; base < nm; base += 256) {
        const int i = base + tid;
        const bool inl = i < nm && emask[o + i] == 1;
        const unsigned bi = __ballot_sync(0xFFFFFFFFu, inl);
        if (lane == 0) s_warp[0][warp] = __popc(bi);
        __syncthreads();
        int oi = s_inl, ti = 0;
        for (int v = 0; v < 8; ++v) {
            oi += v < warp ? s_warp[0][v] : 0;
            ti += s_warp[0][v];
        }
        const int ji = oi + __popc(bi & below);                 // the inlier's ordinal: its recoverPose mask entry
        const bool keep = inl && ji < ni && pmask[o + ji] == 255;
        const unsigned bk = __ballot_sync(0xFFFFFFFFu, keep);
        if (lane == 0) s_warp[1][warp] = __popc(bk);
        __syncthreads();
        int ok = s_keep, tk = 0;
        for (int v = 0; v < 8; ++v) {
            ok += v < warp ? s_warp[1][v] : 0;
            tk += s_warp[1][v];
        }
        const int k = ok + __popc(bk & below);
        if (keep && k < BA_MIN_PT) {
            const float2 a = t0 ? t0[i] : kq[mq[o + i]];
            const float2 c = t0 ? t0[stride + i] : kt[mt[o + i]];
            for (int r = 0; r < 3; ++r) {
                s_rows[k][r] = ba_knorm_row(ki.k + 3 * r, (double)a.x, (double)a.y);
                s_rows[k][3 + r] = ba_knorm_row(ki.k + 3 * r, (double)c.x, (double)c.y);
            }
        }
        __syncthreads();
        if (tid == 0) {
            s_inl += ti;
            s_keep += tk;
        }
        __syncthreads();
        if (s_keep >= BA_MIN_PT) break;
    }
    const bool full = s_keep >= BA_MIN_PT;
    const size_t ro = ((size_t)b * n_rep + j) * BA_MIN_PT * 3;
    for (int e = tid; e < BA_MIN_PT * 3; e += 256) {
        pr[ro + e] = full ? s_rows[e / 3][e % 3] : 1.0;
        p_r[ro + e] = full ? s_rows[e / 3][3 + e % 3] : 1.0;
    }
    if (tid == 0) w[(size_t)b * n_rep + j] = full ? (pw ? pw[p] : 1.0) : 0.0;
    if (j != 0) return;
    for (int e = tid; e < n_zeta * 16; e += 256) {
        const int k = e >> 4, r = (e >> 2) & 3, c = e & 3;
        const int q = tab[(size_t)B * n_rep + (size_t)b * n_zeta + k];
        const bool uq = ba_pair_used(nmatch, ninl, q);
        const double fb = r == 2 ? -0.9 : 0.1;                  // kitti_ba.cpp:741-744: R = I, t = (0.1, 0.1, -0.9)
        double v;
        if (r == 3) v = c == 3 ? 1.0 : 0.0;
        else if (c == 3) v = uq ? t[(size_t)q * 3 + r] : fb;
        else v = uq ? R[(size_t)q * 9 + r * 3 + c] : (r == c ? 1.0 : 0.0);
        const size_t to = ((size_t)b * n_zeta + k) * 16 + (r * 4 + c);
        T0[to] = v;
        T[to] = v;
    }
}

__global__ void finish_kernel(int n_pairs, epivo_pipeline_params prm, const double* __restrict__ E,
                              const double* __restrict__ R, const double* __restrict__ t,
                              const double* __restrict__ T0, double* __restrict__ T,
                              const epivo_lm_res* __restrict__ lmres, const int32_t* __restrict__ lmiters,
                              const int32_t* __restrict__ active, const int32_t* __restrict__ nmatch,
                              const int32_t* __restrict__ ninl, const int32_t* __restrict__ ngood,
                              const int32_t* __restrict__ iters, const int32_t* __restrict__ nmodels,
                              epivo_pair_result* __restrict__ out) {
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair >= n_pairs) return;
    epivo_pair_result r;
    for (int i = 0; i < 9; ++i) { r.E[i] = E[(int64_t)pair * 9 + i]; r.R[i] = R[(int64_t)pair * 9 + i]; }
    for (int i = 0; i < 3; ++i) r.t[i] = t[(int64_t)pair * 3 + i];
    const bool ran = active[pair] != 0;
    r.lm.H_norm = ran ? lmres[pair].H_norm : 0.0;
    r.lm.r_norm = ran ? lmres[pair].r_norm : 0.0;
    r.lm.lambda = ran ? lmres[pair].lambda : prm.lm_lambda0;
    const bool revert = ran && !(r.lm.r_norm <= prm.lm_revert);        // kitti_E.cpp:198-200 (NaN reverts too)
    for (int i = 0; i < 16; ++i) {
        r.T0[i] = T0[(int64_t)pair * 16 + i];
        r.T[i] = (ran && !revert) ? T[(int64_t)pair * 16 + i] : r.T0[i];
    }
    r.n_matches = nmatch[pair];
    r.n_inliers = ninl[pair];
    r.n_good = ngood[pair];
    r.ransac_iters = iters[pair];
    r.n_models = nmodels[pair];
    r.lm_iters = ran ? lmiters[pair] : 0;
    r.lm_ran = ran ? 1 : 0;
    r.lm_reverted = revert ? 1 : 0;
    out[pair] = r;
}

}  // namespace

extern "C" {

void epivo_pipeline_params_default(epivo_pipeline_params* p) {
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->norm = EPIVO_NORM_HAMMING2;
    p->match_mode = EPIVO_MATCH_CROSSCHECK;
    p->ratio = 0.8f;
    // kitti_E.cpp:38-40: cam is a float Mat, which findEssentialMat widens to double
    const double K[9] = {(double)718.8560f, 0.0, (double)607.1928f, 0.0, (double)718.8560f, (double)185.2157f,
                         0.0, 0.0, 1.0};
    memcpy(p->K, K, sizeof(K));
    p->method = EPIVO_RANSAC;
    p->prob = 0.99;
    p->threshold = 1.0;
    p->max_iters = 1000;
    p->dist_thresh = 50.0;
    p->min_trace = 3.0 * 0.9;
    p->fallback_t[0] = 0.1;
    p->fallback_t[1] = 0.1;
    p->fallback_t[2] = -0.9;
    p->min_t_norm = 1e-5;
    p->lm_points = 48;
    p->lm_lambda0 = 1e-2;
    p->lm_epsilon = 1e-8;
    p->lm_max_iters = 30;
    p->huber_delta = 1e-5;
    p->lm_revert = 1e-9;
}

int epivo_seq_create(epivo_ctx* ctx, epivo_seq** out, int max_frames, int kp_per_frame) {
    return epivo_seq_create_pairs(ctx, out, max_frames, kp_per_frame, max_frames - 1);
}

int epivo_seq_create_pairs(epivo_ctx* ctx, epivo_seq** out, int max_frames, int kp_per_frame, int max_pairs) {
    if (!ctx || !out) return EPIVO_ERR_INVALID;
    *out = nullptr;
    if (max_frames < 2 || kp_per_frame < 1) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "need >= 2 frames and >= 1 keypoint");
    if (max_pairs < max_frames - 1) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "max_pairs %d < max_frames - 1", max_pairs);
    if (kp_per_frame > (int)EPV_IDX_MASK) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "too many keypoints per frame");
    EPV_CUDA(ctx, cudaSetDevice(ctx->device));
    epivo_seq* s = new epivo_seq();
    s->ctx = ctx;
    s->max_frames = max_frames;
    s->kp = kp_per_frame;
    s->stride = (kp_per_frame + 31) / 32 * 32;
    s->max_pairs = max_pairs;
    s->n_list = max_frames - 1;
    const size_t F = max_frames, P = max_pairs, st = s->stride, kp = kp_per_frame;
    s->chunk = (int)std::min<size_t>(SEQ_CHUNK, P);
    const size_t C = P;        // group-scoped buffers are allocated for every pair, so groups never alias
    int rc = 0;
#define A(ptr, count) if (!rc) rc = seq_alloc(s, &s->ptr, (count))
    A(d_kps, F * kp * 2);
    A(d_desc, F * kp * 8);
    A(d_planes, F * kp * 8);
    A(d_counts, F);
    A(d_fq, P); A(d_ft, P);
    A(d_mq, P * st); A(d_mt, P * st); A(d_md, P * st); A(d_nmatch, P);
    A(d_emask, P * st); A(d_pmask, P * st);
    A(d_E, P * 9); A(d_R, P * 9); A(d_t, P * 3); A(d_T, P * 16); A(d_T0, P * 16);
    A(d_ninl, P); A(d_iters, P); A(d_nmodels, P); A(d_status, P); A(d_ngood, P);
    A(d_lmactive, P); A(d_lmiters, P); A(d_lmres, P); A(d_results, P);
    A(d_rowkey, C * st); A(d_rowkey2, C * st); A(d_colkey, C * st);
    A(d_xn, C * 4 * st); A(d_xin, C * 4 * st);
    A(d_lmp, C * 64 * 3); A(d_lmq, C * 64 * 3); A(d_w, C);
    A(d_err, epv_essential_errbuf_floats((int)C, (int)st));
    A(d_reps, 2);
    s->esswork_bytes = epv_essential_work_bytes((int)std::min<size_t>(P, SEQ_CHUNK));
    A(d_esswork, s->esswork_bytes);
#undef A
    if (!rc && cudaMallocHost(&s->h_results, P * sizeof(epivo_pair_result)) != cudaSuccess) rc = EPIVO_ERR_CUDA;
    bool ev_ok = true;
    for (int c = 0; c < SEQ_MAX_CHUNKS && ev_ok; ++c)
    {
        for (int k = 0; k < SEQ_STAGES; ++k) ev_ok &= cudaEventCreate(&s->ev[c][k]) == cudaSuccess;
        for (int k = 0; k < 2; ++k) ev_ok &= cudaEventCreate(&s->evk[c][k]) == cudaSuccess;
        ev_ok &= cudaEventCreate(&s->evp[c]) == cudaSuccess;
    }
    for (int c = 0; c < SEQ_MAX_CHUNKS && ev_ok; ++c)
        ev_ok &= cudaEventCreateWithFlags(&s->ev_matched[c], cudaEventDisableTiming) == cudaSuccess;
    ev_ok = ev_ok && cudaEventCreate(&s->ev_begin) == cudaSuccess && cudaEventCreate(&s->ev_end) == cudaSuccess;
    ev_ok = ev_ok && cudaEventCreateWithFlags(&s->ev_geo_done, cudaEventDisableTiming) == cudaSuccess;
    {
        // the second stream carries the H2D pieces of the host-buffer path and, in overlap mode, the geometry
        // kernels: highest priority, so that their short CTAs take the SM slots the long matcher CTAs free up
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);       // hi = numerically lowest = highest priority
        ev_ok = ev_ok && cudaStreamCreateWithPriority(&s->stream2, cudaStreamNonBlocking, hi) == cudaSuccess;
        ev_ok = ev_ok && cudaStreamCreateWithFlags(&s->stream3, cudaStreamNonBlocking) == cudaSuccess;
        // highest priority: a geometry kernel is a chain of ~70 short dependent launches; behind a resident wave of
        // 0.9 ms matcher CTAs each of them would wait for a free slot at normal priority
        ev_ok = ev_ok && cudaStreamCreateWithPriority(&s->stream4, cudaStreamNonBlocking, hi) == cudaSuccess;
        for (int c = 0; c < SEQ_MAX_CHUNKS && ev_ok; ++c)
            ev_ok &= cudaEventCreateWithFlags(&s->ev_piece[c], cudaEventDisableTiming) == cudaSuccess;
    }
    if (rc || !ev_ok) {
        epivo_seq_destroy(s);
        if (!rc) EPV_FAIL(ctx, EPIVO_ERR_CUDA, "event creation failed");
        return rc;
    }
    const int32_t reps[2] = {0, 0};
    EPV_CUDA(ctx, cudaMemcpyAsync(s->d_reps, reps, 8, cudaMemcpyHostToDevice, ctx->stream));
    {
        std::vector<int32_t> full((size_t)max_frames, kp_per_frame);
        EPV_CUDA(ctx, cudaMemcpyAsync(s->d_counts, full.data(), full.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
        EPV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    rc = epivo_seq_set_pairs(s, 0, nullptr, nullptr);      // consecutive pairs (p, p + 1)
    if (rc) { epivo_seq_destroy(s); return rc; }
    s->pairs_set = false;
    EPV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *out = s;
    return EPIVO_OK;
}

void epivo_seq_destroy(epivo_seq* s) {
    if (!s) return;
    cudaSetDevice(s->ctx->device);
    cudaStreamSynchronize(s->ctx->stream);
    for (void* p : s->allocs) cudaFree(p);
    if (s->h_results) cudaFreeHost(s->h_results);
    for (int c = 0; c < SEQ_MAX_CHUNKS; ++c)
        for (int k = 0; k < SEQ_STAGES; ++k)
            if (s->ev[c][k]) cudaEventDestroy(s->ev[c][k]);
    for (int c = 0; c < SEQ_MAX_CHUNKS; ++c)
        for (int k = 0; k < 2; ++k)
            if (s->evk[c][k]) cudaEventDestroy(s->evk[c][k]);
    for (int c = 0; c < SEQ_MAX_CHUNKS; ++c)
        if (s->evp[c]) cudaEventDestroy(s->evp[c]);
    for (int c = 0; c < SEQ_MAX_CHUNKS; ++c)
        if (s->ev_matched[c]) cudaEventDestroy(s->ev_matched[c]);
    if (s->ev_geo_done) cudaEventDestroy(s->ev_geo_done);
    if (s->stream2) { cudaStreamSynchronize(s->stream2); cudaStreamDestroy(s->stream2); }
    if (s->stream3) { cudaStreamSynchronize(s->stream3); cudaStreamDestroy(s->stream3); }
    if (s->stream4) { cudaStreamSynchronize(s->stream4); cudaStreamDestroy(s->stream4); }
    for (int c = 0; c < SEQ_MAX_CHUNKS; ++c)
        if (s->ev_piece[c]) cudaEventDestroy(s->ev_piece[c]);
    if (s->ev_begin) cudaEventDestroy(s->ev_begin);
    if (s->ev_end) cudaEventDestroy(s->ev_end);
    delete s;
}

int epivo_seq_upload(epivo_seq* s, int first_frame, int n_frames, const float* kps, const uint8_t* descs) {
    if (!s) return EPIVO_ERR_INVALID;
    epivo_ctx* ctx = s->ctx;
    if (first_frame < 0 || n_frames < 0 || first_frame + n_frames > s->max_frames || !kps || !descs)
        EPV_FAIL(ctx, EPIVO_ERR_INVALID, "frame range [%d,+%d) outside [0,%d)", first_frame, n_frames, s->max_frames);
    EPV_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t kp = s->kp;
    EPV_CUDA(ctx, cudaMemcpyAsync(s->d_kps + (size_t)first_frame * kp * 2, kps, (size_t)n_frames * kp * 8,
                                  cudaMemcpyHostToDevice, ctx->stream));
    EPV_CUDA(ctx, cudaMemcpyAsync(s->d_desc + (size_t)first_frame * kp * 8, descs, (size_t)n_frames * kp * 32,
                                  cudaMemcpyHostToDevice, ctx->stream));
    s->frames_hi = std::max(s->frames_hi, first_frame + n_frames);
    return EPIVO_OK;
}

int epivo_seq_set_pairs(epivo_seq* s, int n_pairs, const int32_t* fq, const int32_t* ft) {
    if (!s) return EPIVO_ERR_INVALID;
    epivo_ctx* ctx = s->ctx;
    std::vector<int32_t> h;
    if (n_pairs <= 0 || !fq || !ft) {                      // back to the consecutive pairs (p, p + 1)
        n_pairs = s->max_frames - 1;
        h.resize((size_t)n_pairs * 2);
        for (int p = 0; p < n_pairs; ++p) { h[p] = p; h[(size_t)n_pairs + p] = p + 1; }
        s->pairs_set = false;
    } else {
        if (n_pairs > s->max_pairs) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "%d pairs > capacity %d (epivo_seq_create_pairs)", n_pairs, s->max_pairs);
        h.resize((size_t)n_pairs * 2);
        int lmax = 0;
        for (int p = 0; p < n_pairs; ++p) {
            if (fq[p] < 0 || fq[p] >= s->max_frames || ft[p] < 0 || ft[p] >= s->max_frames)
                EPV_FAIL(ctx, EPIVO_ERR_INVALID, "pair %d = (%d,%d) outside [0,%d)", p, fq[p], ft[p], s->max_frames);
            h[p] = fq[p];
            h[(size_t)n_pairs + p] = ft[p];
            lmax = std::max(lmax, std::max(fq[p], ft[p]));
        }
        s->list_max = lmax;                              // only once the whole list has been accepted
        s->pairs_set = true;
    }
    s->h_fq.assign(h.begin(), h.begin() + n_pairs);
    s->h_ft.assign(h.begin() + n_pairs, h.end());
    s->last_run = epivo_seq::RUN_NONE;                   // pair p of the last run is no longer pair p of the list
    EPV_CUDA(ctx, cudaSetDevice(ctx->device));
    EPV_CUDA(ctx, cudaMemcpyAsync(s->d_fq, h.data(), (size_t)n_pairs * 4, cudaMemcpyHostToDevice, ctx->stream));
    EPV_CUDA(ctx, cudaMemcpyAsync(s->d_ft, h.data() + n_pairs, (size_t)n_pairs * 4, cudaMemcpyHostToDevice, ctx->stream));
    EPV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    s->n_list = n_pairs;
    return EPIVO_OK;
}

int epivo_seq_set_counts(epivo_seq* s, int first_frame, int n_frames, const int32_t* counts) {
    if (!s) return EPIVO_ERR_INVALID;
    epivo_ctx* ctx = s->ctx;
    if (first_frame < 0 || n_frames < 0 || first_frame + n_frames > s->max_frames || (n_frames > 0 && !counts))
        EPV_FAIL(ctx, EPIVO_ERR_INVALID, "frame range [%d,+%d) outside [0,%d)", first_frame, n_frames, s->max_frames);
    for (int i = 0; i < n_frames; ++i)
        if (counts[i] < 0 || counts[i] > s->kp) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "counts[%d] = %d outside [0,%d]", i, counts[i], s->kp);
    EPV_CUDA(ctx, cudaSetDevice(ctx->device));
    // pageable source: the copy is staged before the call returns, so the caller's array may go away
    EPV_CUDA(ctx, cudaMemcpyAsync(s->d_counts + first_frame, counts, (size_t)n_frames * 4, cudaMemcpyHostToDevice, ctx->stream));
    EPV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    s->counts_set = true;
    return EPIVO_OK;
}

// keypoints (epivo_keypoint) and descriptors of a batch of frames -> the frame slots of the sequence; one thread per
// (frame, keypoint) word: 2 position floats + 8 descriptor words
__global__ void __launch_bounds__(256) seq_orb_to_slots_kernel(const epivo_keypoint* __restrict__ kps, const uint32_t* __restrict__ desc,
                                                               const int32_t* __restrict__ found, int n_frames, int kp,
                                                               float* __restrict__ slot_kps, uint32_t* __restrict__ slot_desc,
                                                               int32_t* __restrict__ slot_counts) {
    const int f = blockIdx.y;
    const int n = min(found[f], kp);
    if (blockIdx.x == 0 && threadIdx.x == 0) slot_counts[f] = n;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n * 8; i += gridDim.x * 256) {
        const int k = i >> 3, w = i & 7;
        slot_desc[((size_t)f * kp + k) * 8 + w] = desc[((size_t)f * kp + k) * 8 + w];
        if (w < 2) slot_kps[((size_t)f * kp + k) * 2 + w] = w == 0 ? kps[(size_t)f * kp + k].x : kps[(size_t)f * kp + k].y;
    }
}

int epivo_seq_extract_orb(epivo_seq* s, int first_frame, int n_frames, const uint8_t* images, int rows, int cols,
                          int nfeatures, float scale_factor, int nlevels, int edge_threshold, int fast_threshold,
                          int32_t* counts_out) {
    if (!s) return EPIVO_ERR_INVALID;
    epivo_ctx* ctx = s->ctx;
    if (first_frame < 0 || n_frames < 0 || first_frame + n_frames > s->max_frames)
        EPV_FAIL(ctx, EPIVO_ERR_INVALID, "frame range [%d,+%d) outside [0,%d)", first_frame, n_frames, s->max_frames);
    if (n_frames == 0) return EPIVO_OK;
    if (!images || rows <= 0 || cols <= 0) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "null or empty images");
    if (fast_threshold < 0 || fast_threshold > 255) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "fast_threshold %d outside [0, 255]", fast_threshold);
    const int kp = s->kp;
    EpvOrbPlan plan;
    int rc = epv_orb_plan(ctx, n_frames, rows, cols, nfeatures, scale_factor, nlevels, edge_threshold, kp, &plan);
    if (rc) return rc;
    EPV_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t nk = (size_t)n_frames * kp;
    rc = epv_ws_reserve(ctx, epv_orb_work_bytes(plan) + nk * (sizeof(epivo_keypoint) + 32) + (size_t)n_frames * 4 + 4096);
    if (rc) return rc;
    rc = epv_pin_reserve(ctx, (plan.tab_entries + 1) * 4 + 512);
    if (rc) return rc;
    uint8_t* d_pyr = epv_ws_take<uint8_t>(ctx, plan.pyr_bytes);
    epivo_keypoint* d_kps = epv_ws_take<epivo_keypoint>(ctx, nk + 1);
    uint8_t* d_desc = epv_ws_take<uint8_t>(ctx, nk * 32 + 32);
    int32_t* d_found = epv_ws_take<int32_t>(ctx, n_frames);
    uint32_t* h_tab = epv_pin_take<uint32_t>(ctx, plan.tab_entries + 1);
    EPV_CUDA(ctx, cudaMemcpyAsync(d_pyr, images, (size_t)n_frames * rows * cols, cudaMemcpyHostToDevice, ctx->stream));
    rc = epv_orb_launch(ctx, plan, fast_threshold, d_pyr, d_kps, d_desc, d_found, h_tab);
    if (rc) return rc;
    seq_orb_to_slots_kernel<<<dim3(std::max(1, std::min((kp * 8 + 255) / 256, 64)), n_frames), 256, 0, ctx->stream>>>(
        d_kps, (const uint32_t*)d_desc, d_found, n_frames, kp, s->d_kps + (size_t)first_frame * kp * 2,
        s->d_desc + (size_t)first_frame * kp * 8, s->d_counts + first_frame);
    EPV_LAUNCHED(ctx);
    if (counts_out) EPV_CUDA(ctx, cudaMemcpyAsync(counts_out, d_found, (size_t)n_frames * 4, cudaMemcpyDeviceToHost, ctx->stream));
    EPV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));       // the workspace and the resize tables are free for the next call
    s->counts_set = true;
    s->frames_hi = std::max(s->frames_hi, first_frame + n_frames);
    return EPIVO_OK;
}

int epivo_seq_set_overlap(epivo_seq* s, int overlap) {
    if (!s) return EPIVO_ERR_INVALID;
    s->overlap = overlap == 1 ? 1 : 0;
    s->geo_mode = overlap == 2 ? 2 : 0;
    return EPIVO_OK;
}

// geometry of one group on the context's CURRENT stream (the caller selects the stream)
static int seq_run_geometry(epivo_seq* s, const epivo_pipeline_params* prm, int c, int p0, int np) {
    epivo_ctx* ctx = s->ctx;
    const int st = s->stride;
    const size_t o = (size_t)p0;                 // group-scoped buffers are indexed by absolute pair
    int rc;
    EPV_CUDA(ctx, cudaEventRecord(s->ev[c][2], ctx->stream));
    EpvRange r_geo(ctx, "epivo: geometry (findEssentialMat + recoverPose + LM)");
    EssentialPlan ep{};
    ep.n_pairs = np;
    ep.stride = st;
    ep.xn = s->d_xn + o * 4 * st;
    ep.n = s->d_nmatch + p0;
    ep.method = prm->method;
    ep.prob = prm->prob;
    ep.thresh = prm->threshold / ((prm->K[0] + prm->K[4]) / 2.0);
    ep.max_iters = prm->max_iters;
    ep.samples = nullptr;
    ep.m = 0;
    ep.errbuf = s->d_err + epv_essential_errbuf_floats(p0, st);
    ep.E = s->d_E + o * 9;
    ep.mask = s->d_emask + o * st;
    ep.n_inliers = s->d_ninl + p0;
    ep.iters = s->d_iters + p0;
    ep.n_models = s->d_nmodels + p0;
    ep.status = s->d_status + p0;
    ep.xin = s->d_xin + o * 4 * st;
    ep.work = s->d_esswork;          // one group at a time uses it: groups are stream-ordered
    ep.work_bytes = s->esswork_bytes;
    ep.ev_presolved = s->evp[c];
    {
        EpvRange r(ctx, "epivo: findEssentialMat");
        rc = epv_essential_launch(ctx, ep);
    }
    if (rc) return rc;
    EPV_CUDA(ctx, cudaEventRecord(s->ev[c][3], ctx->stream));
    PosePlan pp{};
    pp.n_pairs = np;
    pp.stride = st;
    pp.E = s->d_E + o * 9;
    pp.xn = s->d_xin + o * 4 * st;
    pp.n = s->d_ninl + p0;
    pp.in_mask = nullptr;
    pp.dist_thresh = prm->dist_thresh;
    pp.R = s->d_R + o * 9;
    pp.t = s->d_t + o * 3;
    pp.mask = s->d_pmask + o * st;
    pp.n_good = s->d_ngood + p0;
    pp.skip = s->d_status + p0;
    {
        EpvRange r(ctx, "epivo: recoverPose");
        rc = epv_pose_launch(ctx, pp);
    }
    if (rc) return rc;
    EPV_CUDA(ctx, cudaEventRecord(s->ev[c][4], ctx->stream));
    lm_prep_kernel<<<np, 64, 0, ctx->stream>>>(np, st, *prm, s->d_R + o * 9, s->d_t + o * 3, s->d_status + p0,
                                               s->d_ninl + p0, s->d_ngood + p0, s->d_xin + o * 4 * st,
                                               s->d_T0 + o * 16, s->d_T + o * 16, s->d_lmp + o * 64 * 3,
                                               s->d_lmq + o * 64 * 3, s->d_w + p0, s->d_lmactive + p0);
    EPV_LAUNCHED(ctx);
    LmPlan lp{};
    lp.B = np;
    lp.n_zeta = 1;
    lp.n_rep = 1;
    lp.N = prm->lm_points;
    lp.reps = s->d_reps;
    lp.wreps = s->d_w + p0;
    lp.epsilon = prm->lm_epsilon;
    lp.lambda0 = prm->lm_lambda0;
    lp.huber_delta = prm->huber_delta;
    lp.max_iters = prm->lm_max_iters;
    lp.T0s = s->d_T + o * 16;
    lp.pr = s->d_lmp + o * 64 * 3;
    lp.p_r = s->d_lmq + o * 64 * 3;
    lp.out = s->d_lmres + p0;
    lp.iters = s->d_lmiters + p0;
    lp.active = s->d_lmactive + p0;
    lp.single_pair = 1;
    {
        EpvRange r(ctx, "epivo: Levenberg_Marquardt");
        rc = epv_lm_launch(ctx, lp);
    }
    if (rc) return rc;
    EPV_CUDA(ctx, cudaEventRecord(s->ev[c][5], ctx->stream));
    finish_kernel<<<(np + 127) / 128, 128, 0, ctx->stream>>>(
        np, *prm, s->d_E + o * 9, s->d_R + o * 9, s->d_t + o * 3, s->d_T0 + o * 16, s->d_T + o * 16, s->d_lmres + p0,
        s->d_lmiters + p0, s->d_lmactive + p0, s->d_nmatch + p0, s->d_ninl + p0, s->d_ngood + p0, s->d_iters + p0,
        s->d_nmodels + p0, s->d_results + p0);
    EPV_LAUNCHED(ctx);
    EPV_CUDA(ctx, cudaEventRecord(s->ev[c][6], ctx->stream));
    return EPIVO_OK;
}

// matcher + finalize of one group on the context stream
static int seq_run_match(epivo_seq* s, const epivo_pipeline_params* prm, int c, int p0, int np, bool planes_ready = false) {
    epivo_ctx* ctx = s->ctx;
    const int kp = s->kp, st = s->stride;
    const size_t o = (size_t)p0;
    int rc;
    EPV_CUDA(ctx, cudaEventRecord(s->ev[c][0], ctx->stream));
    EpvRange r_match(ctx, "epivo: BFMatcher::match");
    MatchPlan mp{};
    mp.desc = s->d_desc + o * kp * 8;                     // group-local view: frames p0 .. p0+np
    mp.planes = s->d_planes + o * kp * 8;
    // bit planes of the group's frames; the first frame of a later group was already converted as
    // the last frame of the previous one, converting it again writes the same values
    mp.total_rows = (int64_t)(np + 1) * kp;
    mp.words = 8;
    mp.norm = prm->norm;
    mp.top2 = prm->match_mode == EPIVO_MATCH_RATIO;
    mp.n_pairs = np;
    mp.q0 = 0;
    mp.qs = kp;
    mp.t0 = kp;
    mp.ts = kp;
    mp.nq = kp;
    mp.nt = kp;
    mp.tsplits = 1;
    mp.rowkey = s->d_rowkey + o * st;
    mp.rowkey2 = s->d_rowkey2 + o * st;
    mp.colkey = s->d_colkey + o * st;
    mp.stride = st;
    mp.ev0 = s->evk[c][0];
    mp.ev1 = s->evk[c][1];
    mp.pad_smem = s->match_pad;
    const bool general = s->counts_set || s->pairs_set;     // per-frame counts and / or an explicit pair list
    bool prepass = true;
    if (general) {
        mp.desc = s->d_desc;                                // frames are addressed through fq / ft from the array base
        mp.planes = s->d_planes;
        mp.fq = s->d_fq + p0;
        mp.ft = s->d_ft + p0;
        mp.counts = s->d_counts;
        if (s->pairs_set) {                                 // any frame may be referenced: convert every uploaded
            prepass = (c == 0);                             // frame once per run, with the first group
            mp.prepass_row0 = 0;
            mp.total_rows = (int64_t)s->frames_hi * kp;
        } else {
            mp.prepass_row0 = (int64_t)p0 * kp;
        }
    }
    if (planes_ready) prepass = false;                      // converted on the copy stream, piece by piece
    rc = epv_match_launch(ctx, mp, prepass);
    if (rc) return rc;
    EPV_CUDA(ctx, cudaEventRecord(s->ev[c][1], ctx->stream));
    FinalizePlan fp{};
    fp.n_pairs = np;
    fp.nq = kp;
    fp.nt = kp;
    fp.stride = st;
    fp.mode = prm->match_mode;
    fp.tsplits = 1;
    fp.ratio = prm->ratio;
    fp.rowkey = s->d_rowkey + o * st;
    fp.rowkey2 = s->d_rowkey2 + o * st;
    fp.colkey = s->d_colkey + o * st;
    fp.mq = s->d_mq + o * st;
    fp.mt = s->d_mt + o * st;
    fp.md = s->d_md + o * st;
    fp.md2 = nullptr;
    fp.n_matches = s->d_nmatch + p0;
    fp.kps = s->d_kps + o * kp * 2;
    fp.q0 = 0;
    fp.qs = kp;
    fp.t0 = kp;
    fp.ts = kp;
    fp.p0 = nullptr;
    fp.p1 = nullptr;
    fp.xn = s->d_xn + o * 4 * st;
    const double ax = 1.0 / prm->K[0], ay = 1.0 / prm->K[4];
    fp.ax = ax;
    fp.bx = -prm->K[2] * ax;
    fp.ay = ay;
    fp.by = -prm->K[5] * ay;
    if (general) {
        fp.kps = s->d_kps;
        fp.fq = s->d_fq + p0;
        fp.ft = s->d_ft + p0;
        fp.counts = s->d_counts;
    }
    rc = epv_finalize_launch(ctx, fp);
    if (rc) return rc;
    return EPIVO_OK;
}

// Tuning aid (EPIVO_UPLOAD_DELAY_US): a sleeping kernel on the copy stream behind every upload piece, to reproduce on
// one GPU the input rate a rank sees when eight ranks share the host's copy path.
__device__ __forceinline__ unsigned long long epv_globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__global__ void upload_delay_kernel(unsigned us) {
    const unsigned long long t0 = epv_globaltimer_ns();
    while (epv_globaltimer_ns() - t0 < (unsigned long long)us * 1000ull) __nanosleep(2000);
}

// Common executor.  With host buffers (h_kps/h_desc != NULL) the frames are uploaded in pieces on
// the copy stream and every matcher group starts as soon as its frames have landed, so the
// host->device transfer hides under the matcher; the geometry then runs once over all pairs.
static int seq_execute(epivo_seq* s, const epivo_pipeline_params* prm, int first_pair, int n_pairs,
                       const float* h_kps, const uint8_t* h_desc, int n_frames_up) {
    epivo_ctx* ctx = s->ctx;
    if (first_pair < 0 || n_pairs < 0 || first_pair + n_pairs > s->n_list)
        EPV_FAIL(ctx, EPIVO_ERR_INVALID, "pair range [%d,+%d) outside [0,%d)", first_pair, n_pairs, s->n_list);
    if (prm->lm_points < 1 || prm->lm_points > 64) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "lm_points must be in [1,64]");
    if (prm->method != EPIVO_RANSAC && prm->method != EPIVO_LMEDS) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "method");
    if (prm->match_mode < 0 || prm->match_mode > 2) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "match_mode");
    if (prm->norm != EPIVO_NORM_HAMMING && prm->norm != EPIVO_NORM_HAMMING2) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "norm");
    EPV_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t main_stream = ctx->stream;
    EpvRange r_seq(ctx, h_kps ? "epivo_seq_process" : "epivo_seq_run");
    // an explicit pair list may reference any frame: host buffers are then uploaded whole before the first group
    const bool upload_all = h_kps != nullptr && s->pairs_set;
    const bool upload = h_kps != nullptr && !upload_all;
    const bool overlap = s->overlap && !upload && !upload_all;
    if (upload || upload_all) s->frames_hi = std::max(s->frames_hi, first_pair + n_frames_up);
    if (s->pairs_set && s->frames_hi == 0) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "pair list set but no frames uploaded");
    if (s->pairs_set && s->list_max >= s->frames_hi)          // a slot never uploaded would be matched as garbage
        EPV_FAIL(ctx, EPIVO_ERR_INVALID, "the pair list references frame %d but only frames [0,%d) have been uploaded",
                 s->list_max, s->frames_hi);
    // matcher groups / geometry groups (event slots: matcher [0, HALF), geometry [HALF, 2*HALF))
    constexpr int HALF = SEQ_MAX_CHUNKS / 2;
    // matcher groups.  Resident data: uniform groups.  Host buffers: the upload is cut into pieces of at most one wave
    // of matcher CTAs, every matcher launch waiting only for its own frames (and the launches alternate between
    // two streams, see below, so a piece boundary costs nothing).  Small pieces are what matters when the copy is
    // slower than the matcher: alone on a box the PCIe copy delivers frames 2x faster than the matcher consumes
    // them (55 GB/s against 26 GB/s) and any schedule hides it, but with eight ranks pulling at once a rank gets
    // 23 GB/s (profiles/r2_h2d_ceiling_8gpu.json), the matcher runs behind the copy, and the step ends one piece
    // of matching after the last byte lands (round 1's 1, 2, 4, rest schedule left 2468 pairs = 7.5 ms there).
    std::vector<std::pair<int, int> > mg;     // (first pair, pairs)
    {
        const int mchunk = overlap ? SEQ_CHUNK_OVERLAP : SEQ_CHUNK;
        int wave = upload ? epv_match_pairs_per_wave(ctx, s->kp) : mchunk;
        int max_pieces = HALF, cap_waves = 4;
        if (upload) {                                   // tuning knobs (environment): first piece = wave / div, piece count, cap
            // default: a quarter wave first (the matcher starts 0.1 ms after the call instead of 0.43), doubling up to
            // one wave: 74, 148, 296, 296, ... pairs (measured 17.17 -> 16.94 ms per step against 16.65 device-resident)
            int div = 4;
            if (const char* e = getenv("EPIVO_UPLOAD_DIV")) div = std::max(1, atoi(e));
            wave = std::max(1, wave / div);
            if (const char* e = getenv("EPIVO_UPLOAD_PIECES")) max_pieces = std::min(HALF, std::max(1, atoi(e)));
            if (const char* e = getenv("EPIVO_UPLOAD_CAP")) cap_waves = std::max(1, atoi(e));
            // never more pieces than event slots: widen the cap for very long sequences
            while ((n_pairs + (int64_t)wave * cap_waves - 1) / ((int64_t)wave * cap_waves) + 2 > max_pieces && cap_waves < (1 << 20))
                cap_waves *= 2;
        }
        int p0 = first_pair, left = n_pairs, waves = 1;
        while (left > 0) {
            int np = upload ? wave * waves : mchunk;
            if (upload && ((int)mg.size() >= max_pieces - 1 || left - np < wave)) np = left;    // the last piece takes the rest
            np = std::min(np, left);
            mg.push_back(std::make_pair(p0, np));
            p0 += np;
            left -= np;
            waves = std::min(2 * waves, cap_waves);
        }
    }
    const int gchunk = overlap ? SEQ_CHUNK_OVERLAP : SEQ_CHUNK;
    const int n_m = (int)mg.size(), n_g = (n_pairs + gchunk - 1) / gchunk;
    if (n_m > HALF || n_g > HALF) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "too many pair groups");
    s->last_mgroups = n_m;
    s->last_ggroups = n_g;
    s->last_frames = false;
    s->last_run = epivo_seq::RUN_DESC;
    s->last_n_pairs = n_pairs;
    s->last_first = first_pair;
    // Host-buffer path: the geometry of the pairs already matched CAN run between the matcher pieces (four groups, own
    // high-priority stream: epivo_seq_set_overlap(seq, 2)), which looks attractive when the copy is the limiter and
    // the GPU idles between pieces.  Measured, it loses in every regime -- 17.2 -> 18.9 ms per step with the copy at
    // full rate, 22.4 -> 23.1 ms with the copy throttled to the rate of an 8-rank run (EPIVO_UPLOAD_DELAY_US), and
    // 19.7 -> 20.8 ms on 8 GPUs: a geometry group is a chain of ~70 short dependent launches whose CTAs take slots
    // and issue cycles from the matcher wave that has just become ready, and the matcher then falls behind the copy.
    // So the default stays: geometry after the last matcher piece.
    int geo_mode = s->geo_mode;
    if (const char* e = getenv("EPIVO_GEO_MODE")) geo_mode = atoi(e);      // tuning / experiments: 2 = interleave
    const bool interleave = upload && n_m >= 8 && geo_mode == 2;
    if (upload && getenv("EPIVO_DEBUG_SCHED"))
        fprintf(stderr, "[epivo dev %d] host-buffer call: %d pieces, interleave %d\n", ctx->device, n_m, (int)interleave);
    EPV_CUDA(ctx, cudaEventRecord(s->ev_begin, main_stream));
    int rc = EPIVO_OK;
    const size_t kp = s->kp;
    const bool planes_on_copy = upload && prm->norm == EPIVO_NORM_HAMMING2;
    if (upload) {
        // all pieces are queued on the copy stream at once; they run back to back at PCIe rate.  HAMMING2: the bit
        // planes of a piece's frames are made right behind its copy, on the copy stream, so that a matcher launch
        // depends on nothing but its own event (no pre-pass in front of it, no frame converted twice).
        EPV_CUDA(ctx, cudaStreamWaitEvent(s->stream2, s->ev_begin, 0));
        EPV_CUDA(ctx, cudaStreamWaitEvent(s->stream3, s->ev_begin, 0));
        const char* de = getenv("EPIVO_UPLOAD_DELAY_US");
        const int delay_us = de ? atoi(de) : 0;
        for (int c = 0; c < n_m; ++c) {
            const int p0 = mg[c].first, np = mg[c].second;
            const int f0 = (c == 0) ? p0 : p0 + 1;                  // frame p0 came with the previous piece
            const int nf = p0 + np + 1 - f0;
            const size_t ho = (size_t)(f0 - first_pair);            // host arrays start at frame first_pair
            EPV_CUDA(ctx, cudaMemcpyAsync(s->d_kps + (size_t)f0 * kp * 2, h_kps + ho * kp * 2, (size_t)nf * kp * 8,
                                          cudaMemcpyHostToDevice, s->stream2));
            EPV_CUDA(ctx, cudaMemcpyAsync(s->d_desc + (size_t)f0 * kp * 8, h_desc + ho * kp * 32, (size_t)nf * kp * 32,
                                          cudaMemcpyHostToDevice, s->stream2));
            if (planes_on_copy) {
                rc = epv_planes_launch(ctx, s->d_desc + (size_t)f0 * kp * 8, s->d_planes + (size_t)f0 * kp * 8,
                                       (int64_t)nf * kp, 8, s->stream2);
                if (rc) return rc;
            }
            if (delay_us > 0) upload_delay_kernel<<<1, 1, 0, s->stream2>>>((unsigned)delay_us);
            EPV_CUDA(ctx, cudaEventRecord(s->ev_matched[c], s->stream2));
        }
        if (interleave) EPV_CUDA(ctx, cudaStreamWaitEvent(s->stream4, s->ev_begin, 0));
    }
    if (upload_all) {
        EPV_CUDA(ctx, cudaStreamWaitEvent(s->stream2, s->ev_begin, 0));
        EPV_CUDA(ctx, cudaMemcpyAsync(s->d_kps, h_kps, (size_t)n_frames_up * kp * 8, cudaMemcpyHostToDevice, s->stream2));
        EPV_CUDA(ctx, cudaMemcpyAsync(s->d_desc, h_desc, (size_t)n_frames_up * kp * 32, cudaMemcpyHostToDevice, s->stream2));
        EPV_CUDA(ctx, cudaEventRecord(s->ev_matched[0], s->stream2));
        EPV_CUDA(ctx, cudaStreamWaitEvent(main_stream, s->ev_matched[0], 0));
    }
    if (overlap) EPV_CUDA(ctx, cudaStreamWaitEvent(s->stream2, s->ev_begin, 0));
    int n_geo = 0;                       // geometry groups already issued (interleaved mode)
    for (int c = 0; c < n_m && !rc; ++c) {
        const int p0 = mg[c].first, np = mg[c].second;
        cudaStream_t piece_stream = main_stream;
        if (upload) {
            // the matcher pieces alternate between two streams: piece c+1 (its frames have landed) fills the SMs
            // that the draining CTAs of piece c free up, and its finalize / key-fill kernels run beside piece c+1's
            // tiles -- on one stream every piece boundary cost ~0.1 ms of drained GPU
            piece_stream = (c & 1) ? s->stream3 : main_stream;
            EPV_CUDA(ctx, cudaStreamWaitEvent(piece_stream, s->ev_matched[c], 0));
        }
        ctx->stream = piece_stream;
        rc = seq_run_match(s, prm, c, p0, np, planes_on_copy);
        ctx->stream = main_stream;
        if (rc) break;
        if (interleave) {
            EPV_CUDA(ctx, cudaEventRecord(s->ev_piece[c], piece_stream));
            const int per = (n_m + 3) / 4;                          // pieces per geometry group
            if ((c + 1) % per == 0 || c == n_m - 1) {
                const int c0 = (c / per) * per;                     // the group's first piece
                const int gp0 = mg[c0].first, gnp = p0 + np - gp0;
                EPV_CUDA(ctx, cudaStreamWaitEvent(s->stream4, s->ev_piece[c], 0));
                if (c > 0) EPV_CUDA(ctx, cudaStreamWaitEvent(s->stream4, s->ev_piece[c - 1], 0));   // the other stream's last piece
                ctx->stream = s->stream4;
                rc = seq_run_geometry(s, prm, HALF + n_geo, gp0, gnp);
                ctx->stream = main_stream;
                if (rc) break;
                ++n_geo;
            }
        }
        if (overlap) {      // optional two-stream compute: geometry of group c under the matcher of c+1
            EPV_CUDA(ctx, cudaEventRecord(s->ev_matched[c], main_stream));
            EPV_CUDA(ctx, cudaStreamWaitEvent(s->stream2, s->ev_matched[c], 0));
            ctx->stream = s->stream2;
            rc = seq_run_geometry(s, prm, HALF + c, p0, np);
            ctx->stream = main_stream;
        }
    }
    if (upload && n_m > 1 && !rc) {     // the odd pieces join the context stream before the geometry
        EPV_CUDA(ctx, cudaEventRecord(s->ev_geo_done, s->stream3));
        EPV_CUDA(ctx, cudaStreamWaitEvent(main_stream, s->ev_geo_done, 0));
    }
    ctx->stream = main_stream;
    if (rc) return rc;
    if (interleave) {       // every group's geometry is already queued on stream4: join it
        s->last_ggroups = n_geo;
        EPV_CUDA(ctx, cudaEventRecord(s->ev_geo_done, s->stream4));
        EPV_CUDA(ctx, cudaStreamWaitEvent(main_stream, s->ev_geo_done, 0));
    } else if (overlap) {   // later work on the context stream (download) is ordered after the geometry
        EPV_CUDA(ctx, cudaEventRecord(s->ev_geo_done, s->stream2));
        EPV_CUDA(ctx, cudaStreamWaitEvent(main_stream, s->ev_geo_done, 0));
    } else {
        for (int c = 0; c < n_g && !rc; ++c) {
            const int p0 = first_pair + c * gchunk;
            const int np = std::min(gchunk, first_pair + n_pairs - p0);
            rc = seq_run_geometry(s, prm, HALF + c, p0, np);
        }
        if (rc) return rc;
    }
    EPV_CUDA(ctx, cudaEventRecord(s->ev_end, main_stream));
    return EPIVO_OK;
}

int epivo_seq_run(epivo_seq* s, const epivo_pipeline_params* prm, int first_pair, int n_pairs) {
    if (!s || !prm) return EPIVO_ERR_INVALID;
    return seq_execute(s, prm, first_pair, n_pairs, nullptr, nullptr, 0);
}

int epivo_seq_process(epivo_seq* s, const epivo_pipeline_params* prm, int n_frames, const float* kps,
                      const uint8_t* descs, epivo_pair_result* out) {
    if (!s || !prm) return EPIVO_ERR_INVALID;
    epivo_ctx* ctx = s->ctx;
    if (!kps || !descs || !out) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "null buffer");
    if (n_frames < 2 || n_frames > s->max_frames) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "n_frames %d outside [2,%d]", n_frames, s->max_frames);
    // consecutive pairs: n_frames - 1 of them; explicit pair list (epivo_seq_set_pairs): the whole list
    if (s->pairs_set && s->list_max >= n_frames)
        EPV_FAIL(ctx, EPIVO_ERR_INVALID, "the pair list references frame %d but only %d frames are given", s->list_max, n_frames);
    const int n_pairs = s->pairs_set ? s->n_list : n_frames - 1;
    int rc = seq_execute(s, prm, 0, n_pairs, kps, descs, n_frames);
    if (rc) return rc;
    return epivo_seq_download(s, out, 0, n_pairs);
}

int epivo_seq_process_points(epivo_seq* s, const epivo_pipeline_params* prm, int n_pairs, const float* p0, const float* p1,
                             const int32_t* counts, int max_pts, epivo_pair_result* out) {
    if (!s || !prm) return EPIVO_ERR_INVALID;
    epivo_ctx* ctx = s->ctx;
    if (n_pairs < 0 || n_pairs > s->n_list) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "n_pairs %d outside [0,%d]", n_pairs, s->n_list);
    if (n_pairs == 0) return EPIVO_OK;
    if (!p0 || !p1 || !counts || !out) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "null buffer");
    if (max_pts < 1 || max_pts > s->kp) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "max_pts %d outside [1,%d]", max_pts, s->kp);
    if (prm->lm_points < 1 || prm->lm_points > 64) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "lm_points must be in [1,64]");
    if (prm->method != EPIVO_RANSAC && prm->method != EPIVO_LMEDS) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "method");
    for (int i = 0; i < n_pairs; ++i)
        if (counts[i] < 0 || counts[i] > max_pts) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "counts[%d] = %d outside [0,%d]", i, counts[i], max_pts);
    EPV_CUDA(ctx, cudaSetDevice(ctx->device));
    EpvRange r_seq(ctx, "epivo_seq_process_points");
    const size_t np = (size_t)n_pairs * max_pts;
    int rc = epv_ws_reserve(ctx, np * 16 + (size_t)n_pairs * 4 + 4096);
    if (rc) return rc;
    float* d_p0 = epv_ws_take<float>(ctx, np * 2);
    float* d_p1 = epv_ws_take<float>(ctx, np * 2);
    int32_t* d_cnt = epv_ws_take<int32_t>(ctx, n_pairs);
    cudaStream_t st = ctx->stream;
    EPV_CUDA(ctx, cudaEventRecord(s->ev_begin, st));
    EPV_CUDA(ctx, cudaMemcpyAsync(d_p0, p0, np * 8, cudaMemcpyHostToDevice, st));
    EPV_CUDA(ctx, cudaMemcpyAsync(d_p1, p1, np * 8, cudaMemcpyHostToDevice, st));
    EPV_CUDA(ctx, cudaMemcpyAsync(d_cnt, counts, (size_t)n_pairs * 4, cudaMemcpyHostToDevice, st));
    const double ax = 1.0 / prm->K[0], ay = 1.0 / prm->K[4];
    points_in_kernel<<<dim3((max_pts + 255) / 256, n_pairs), 256, 0, st>>>(d_p0, d_p1, d_cnt, max_pts, s->stride, ax,
                                                                            -prm->K[2] * ax, ay, -prm->K[5] * ay, s->d_xn,
                                                                            s->d_nmatch, s->d_mq, s->d_mt);
    EPV_LAUNCHED(ctx);
    constexpr int HALF = SEQ_MAX_CHUNKS / 2;
    const int n_g = (n_pairs + SEQ_CHUNK - 1) / SEQ_CHUNK;
    if (n_g > HALF) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "too many pair groups");
    s->last_mgroups = 0;
    s->last_ggroups = n_g;
    s->last_n_pairs = n_pairs;
    s->last_first = 0;
    s->last_frames = false;
    s->last_run = epivo_seq::RUN_POINTS;
    for (int c = 0; c < n_g; ++c) {
        const int g0 = c * SEQ_CHUNK, gn = std::min(SEQ_CHUNK, n_pairs - g0);
        rc = seq_run_geometry(s, prm, HALF + c, g0, gn);
        if (rc) return rc;
    }
    EPV_CUDA(ctx, cudaEventRecord(s->ev_end, st));
    return epivo_seq_download(s, out, 0, n_pairs);
}

// The optical-flow loop body from frames (kitti_E.cpp:54-201, kitti.cpp, euroc_E.cpp:169-208).  The frames go through
// the front end in windows of at most G frames, so that the workspace stays bounded on long sequences: per window one
// upload, [remap], FAST capped at kp_per_frame, the pyramids and Scharr derivatives of every frame of the window, LK for
// the pairs of the window and the status compaction into the sequence's correspondence buffers.  Consecutive windows
// share S = max |ft - fq| frames, so every pair lies inside a window; a pair is tracked in the first window that holds
// both of its frames.  The geometry then runs over all pairs as in epivo_seq_process_points (not interleaved with the
// front end: overlapping the geometry with other work measured slower, see epivo_seq_set_overlap).
namespace {
constexpr int FRAMES_MAX_WINDOW = 256;
constexpr size_t FRAMES_WS_BUDGET = (size_t)3 << 29;        // 1.5 GiB of front-end workspace per window
constexpr int LK_WINDOW = 21, LK_MAX_LEVEL = 3, LK_MAX_COUNT = 30;   // calcOpticalFlowPyrLK's defaults, which every
constexpr double LK_EPSILON = 0.01, LK_MIN_EIG = 1e-4;              // reference call site uses

struct FramesWs {
    size_t src, img, maps, fast, lk, kps;
    size_t total() const { return src + img + maps + fast + lk + kps; }
};
FramesWs frames_ws(int g, int rows, int cols, int R, int C, bool maps, int kp) {
    FramesWs w;
    w.src = maps ? epv_align((size_t)g * rows * cols) : 0;
    w.img = epv_align((size_t)g * R * C);
    w.maps = maps ? epv_align((size_t)R * C * 4) + epv_align((size_t)R * C * 2) : 0;
    w.fast = epv_align(epv_fast_work_bytes(g, R, C));
    w.lk = epv_align(epv_lk_work_bytes(g, R, C, LK_MAX_LEVEL));
    w.kps = epv_align((size_t)g * kp * 8);
    return w;
}
}  // namespace

int epivo_seq_process_frames(epivo_seq* s, const epivo_pipeline_params* prm, int n_frames, const uint8_t* images, int rows,
                             int cols, const int16_t* map_xy, const uint16_t* map_frac, int drows, int dcols,
                             int fast_threshold, int32_t* corners_out, epivo_pair_result* out) {
    if (!s || !prm) return EPIVO_ERR_INVALID;
    epivo_ctx* ctx = s->ctx;
    // every check before the first launch
    if (!images || !out) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "null buffer");
    if (n_frames < 2 || n_frames > s->max_frames) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "n_frames %d outside [2,%d]", n_frames, s->max_frames);
    if (rows <= 0 || cols <= 0) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "empty frames (%d x %d)", cols, rows);
    const bool maps = map_xy != nullptr || map_frac != nullptr;
    if (maps && (!map_xy || !map_frac || drows <= 0 || dcols <= 0))
        EPV_FAIL(ctx, EPIVO_ERR_INVALID, "remap needs both maps and a positive size (%d x %d)", dcols, drows);
    const int R = maps ? drows : rows, C = maps ? dcols : cols;
    if (R <= LK_WINDOW || C <= LK_WINDOW)
        EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "image %d x %d not larger than the %d x %d LK window", C, R, LK_WINDOW, LK_WINDOW);
    if (fast_threshold < 0 || fast_threshold > 255) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "fast_threshold %d outside [0, 255]", fast_threshold);
    if (prm->lm_points < 1 || prm->lm_points > 64) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "lm_points must be in [1,64]");
    if (prm->method != EPIVO_RANSAC && prm->method != EPIVO_LMEDS) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "method");
    if (s->pairs_set && s->list_max >= n_frames)
        EPV_FAIL(ctx, EPIVO_ERR_INVALID, "the pair list references frame %d but only %d frames are given", s->list_max, n_frames);
    const int n_pairs = s->pairs_set ? s->n_list : n_frames - 1;
    constexpr int HALF = SEQ_MAX_CHUNKS / 2;
    const int n_g = (n_pairs + SEQ_CHUNK - 1) / SEQ_CHUNK;
    if (n_g > HALF) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "too many pair groups");
    const int kp = s->kp, st = s->stride;
    // window size G: at most 256 frames, and no more than the workspace budget holds
    int G = std::min(FRAMES_MAX_WINDOW, n_frames);
    while (G > 2 && frames_ws(G, rows, cols, R, C, maps, kp).total() > FRAMES_WS_BUDGET) --G;
    int S = 0;
    for (int p = 0; p < n_pairs; ++p) S = std::max(S, std::abs(s->h_ft[p] - s->h_fq[p]));
    if (S >= G)
        EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "a pair spans %d frames; the front end tracks in windows of %d frames", S, G);
    const int step = G - S;
    const int n_win = 1 + (n_frames > G ? (n_frames - G + step - 1) / step : 0);
    // pairs by window (list order inside a window): meta block of window k at 3 * first[k]
    std::vector<int> win(n_pairs), first(n_win + 1, 0);
    for (int p = 0; p < n_pairs; ++p) {
        const int hi = std::max(s->h_fq[p], s->h_ft[p]);
        win[p] = hi < G ? 0 : (hi - G + 1 + step - 1) / step;
        ++first[win[p] + 1];
    }
    int max_wp = 0;
    for (int k = 0; k < n_win; ++k) {
        max_wp = std::max(max_wp, first[k + 1]);
        first[k + 1] += first[k];
    }
    if (max_wp > 65535) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "%d pairs in one frame window (at most 65535)", max_wp);
    std::vector<int32_t> meta((size_t)3 * n_pairs);
    {
        std::vector<int> fill(first.begin(), first.end() - 1);
        for (int p = 0; p < n_pairs; ++p) {
            const int k = win[p], nk = first[k + 1] - first[k], j = fill[k]++ - first[k];
            int32_t* m = meta.data() + (size_t)3 * first[k];
            m[j] = s->h_fq[p] - k * step;             // window-local frames
            m[nk + j] = s->h_ft[p] - k * step;
            m[2 * nk + j] = p;
        }
    }
    EPV_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!s->d_trk) {
        const int rc = seq_alloc(s, &s->d_trk, (size_t)s->max_pairs * st * 4);
        if (rc) return rc;
    }
    const FramesWs w = frames_ws(G, rows, cols, R, C, maps, kp);
    const size_t np = (size_t)max_wp * kp;
    int rc = epv_ws_reserve(ctx, w.total() + epv_align((size_t)n_frames * 4) + epv_align(meta.size() * 4 + 4) +
                                     epv_align(np * 8) + epv_align(np) + epv_align(np * 4) + 4096);
    if (rc) return rc;
    uint8_t* d_src = maps ? epv_ws_take<uint8_t>(ctx, w.src) : nullptr;
    uint8_t* d_img = epv_ws_take<uint8_t>(ctx, w.img);
    int16_t* d_mxy = maps ? epv_ws_take<int16_t>(ctx, (size_t)R * C * 2) : nullptr;
    uint16_t* d_mfr = maps ? epv_ws_take<uint16_t>(ctx, (size_t)R * C) : nullptr;
    uint8_t* d_fast = epv_ws_take<uint8_t>(ctx, w.fast);
    uint8_t* d_lk = epv_ws_take<uint8_t>(ctx, w.lk);
    float* d_kps = epv_ws_take<float>(ctx, (size_t)G * kp * 2);
    int32_t* d_found = epv_ws_take<int32_t>(ctx, n_frames);
    int32_t* d_meta = epv_ws_take<int32_t>(ctx, meta.size() + 1);
    float* d_next = epv_ws_take<float>(ctx, np * 2);
    uint8_t* d_status = epv_ws_take<uint8_t>(ctx, np);
    float* d_err = epv_ws_take<float>(ctx, np);       // passed as every reference call site does: it gates the status
    cudaStream_t cs = ctx->stream;
    EpvRange r_seq(ctx, "epivo_seq_process_frames");
    EPV_CUDA(ctx, cudaEventRecord(s->ev_begin, cs));
    if (maps) {
        EPV_CUDA(ctx, cudaMemcpyAsync(d_mxy, map_xy, (size_t)R * C * 4, cudaMemcpyHostToDevice, cs));
        EPV_CUDA(ctx, cudaMemcpyAsync(d_mfr, map_frac, (size_t)R * C * 2, cudaMemcpyHostToDevice, cs));
    }
    EPV_CUDA(ctx, cudaMemcpyAsync(d_meta, meta.data(), meta.size() * 4, cudaMemcpyHostToDevice, cs));
    const double ax = 1.0 / prm->K[0], ay = 1.0 / prm->K[4];
    const double bx = -prm->K[2] * ax, by = -prm->K[5] * ay;
    for (int k = 0; k < n_win; ++k) {
        const int f0 = k * step, g = std::min(G, n_frames - f0), nk = first[k + 1] - first[k];
        const size_t fb = (size_t)rows * cols;
        EPV_CUDA(ctx, cudaMemcpyAsync(maps ? d_src : d_img, images + (size_t)f0 * fb, (size_t)g * fb, cudaMemcpyHostToDevice, cs));
        if (maps) {
            rc = epv_remap_launch(ctx, d_src, g, rows, cols, d_mxy, d_mfr, R, C, 0, d_img);
            if (rc) return rc;
        }
        // a frame shared with the previous window is detected again: the same corners, the same count
        rc = epv_fast_launch(ctx, d_img, g, R, C, fast_threshold, 1, kp, d_kps, nullptr, d_found + f0, d_fast);
        if (rc) return rc;
        if (nk == 0) continue;
        rc = epv_lk_pyramids(ctx, d_img, g, R, C, LK_MAX_LEVEL, g, d_lk);
        if (rc) return rc;
        const int32_t* m = d_meta + (size_t)3 * first[k];
        rc = epv_lk_track_launch(ctx, d_lk, g, R, C, LK_MAX_LEVEL, nk, m, d_kps, d_found + f0, kp, LK_MAX_COUNT, LK_EPSILON,
                                 LK_MIN_EIG, d_next, d_status, d_err);
        if (rc) return rc;
        track_compact_kernel<<<nk, 256, 0, cs>>>(m, nk, d_kps, d_found + f0, kp, d_next, d_status, st, ax, bx, ay, by,
                                                 s->d_trk, s->d_xn, s->d_nmatch, s->d_mq, s->d_mt, s->d_md);
        EPV_LAUNCHED(ctx);
    }
    s->last_mgroups = 0;
    s->last_ggroups = n_g;
    s->last_n_pairs = n_pairs;
    s->last_first = 0;
    s->last_frames = true;
    s->last_run = epivo_seq::RUN_FRAMES;
    for (int c = 0; c < n_g; ++c) {
        const int g0 = c * SEQ_CHUNK, gn = std::min(SEQ_CHUNK, n_pairs - g0);
        rc = seq_run_geometry(s, prm, HALF + c, g0, gn);
        if (rc) return rc;
    }
    EPV_CUDA(ctx, cudaEventRecord(s->ev_end, cs));
    if (corners_out) EPV_CUDA(ctx, cudaMemcpyAsync(corners_out, d_found, (size_t)n_frames * 4, cudaMemcpyDeviceToHost, cs));
    return epivo_seq_download(s, out, 0, n_pairs);
}

int epivo_seq_get_points(epivo_seq* s, int pair, float* p0, float* p1, int* n_out) {
    if (!s || !n_out) return EPIVO_ERR_INVALID;
    epivo_ctx* ctx = s->ctx;
    if (!s->last_frames) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "the last run was not epivo_seq_process_frames");
    if (pair < 0 || pair >= s->last_n_pairs) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "pair %d outside [0,%d)", pair, s->last_n_pairs);
    EPV_CUDA(ctx, cudaSetDevice(ctx->device));
    int32_t n = 0;
    const float* t = s->d_trk + (size_t)pair * 4 * s->stride;
    EPV_CUDA(ctx, cudaMemcpyAsync(&n, s->d_nmatch + pair, 4, cudaMemcpyDeviceToHost, ctx->stream));
    EPV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (p0) EPV_CUDA(ctx, cudaMemcpyAsync(p0, t, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (p1) EPV_CUDA(ctx, cudaMemcpyAsync(p1, t + 2 * (size_t)s->stride, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    EPV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *n_out = n;
    return EPIVO_OK;
}

int epivo_seq_download(epivo_seq* s, epivo_pair_result* out, int first_pair, int n_pairs) {
    if (!s || !out) return EPIVO_ERR_INVALID;
    epivo_ctx* ctx = s->ctx;
    if (first_pair < 0 || n_pairs < 0 || first_pair + n_pairs > s->n_list)
        EPV_FAIL(ctx, EPIVO_ERR_INVALID, "pair range");
    EPV_CUDA(ctx, cudaSetDevice(ctx->device));
    // a pinned caller buffer takes the DMA directly; pageable memory goes through the pinned staging copy
    cudaPointerAttributes pa;
    const bool pinned = cudaPointerGetAttributes(&pa, out) == cudaSuccess && pa.type == cudaMemoryTypeHost;
    if (!pinned) (void)cudaGetLastError();
    epivo_pair_result* dst = pinned ? out : s->h_results;
    EPV_CUDA(ctx, cudaMemcpyAsync(dst, s->d_results + first_pair, (size_t)n_pairs * sizeof(epivo_pair_result),
                                  cudaMemcpyDeviceToHost, ctx->stream));
    EPV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (!pinned) memcpy(out, s->h_results, (size_t)n_pairs * sizeof(epivo_pair_result));
    return EPIVO_OK;
}

int epivo_seq_cloud(epivo_seq* s, const double* scales, int first_pair, int n_pairs, double* poses, double* points,
                    int64_t cap, int64_t* limits, int64_t* n_points) {
    if (!s) return EPIVO_ERR_INVALID;
    epivo_ctx* ctx = s->ctx;
    if (first_pair < 0 || n_pairs < 0 || first_pair + n_pairs > s->n_list)
        EPV_FAIL(ctx, EPIVO_ERR_INVALID, "pair range [%d,+%d) outside [0,%d)", first_pair, n_pairs, s->n_list);
    if (first_pair < s->last_first || first_pair + n_pairs > s->last_first + s->last_n_pairs)
        EPV_FAIL(ctx, EPIVO_ERR_INVALID, "pairs [%d,+%d) were not part of the last run", first_pair, n_pairs);
    if (n_points) *n_points = 0;
    if (n_pairs == 0) {
        if (poses) { for (int i = 0; i < 16; ++i) poses[i] = (i % 5 == 0) ? 1.0 : 0.0; }
        return EPIVO_OK;
    }
    EPV_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t np = (size_t)n_pairs;
    if (cap < 0 || !points) cap = 0;
    size_t need = epv_align(np * 8) + epv_align((np + 1) * 128) + epv_align(np * 4) + epv_align((np + 1) * 8) +
                  epv_align((size_t)cap * 24) + 4096;
    int rc = epv_ws_reserve(ctx, need);
    if (rc) return rc;
    double* d_scales = scales ? epv_ws_take<double>(ctx, np) : nullptr;
    double* d_poses = epv_ws_take<double>(ctx, (np + 1) * 16);
    int32_t* d_counts = epv_ws_take<int32_t>(ctx, np);
    int64_t* d_limits = epv_ws_take<int64_t>(ctx, np + 1);
    double* d_points = cap > 0 ? epv_ws_take<double>(ctx, (size_t)cap * 3) : nullptr;
    if (scales) EPV_CUDA(ctx, cudaMemcpyAsync(d_scales, scales, np * 8, cudaMemcpyHostToDevice, ctx->stream));
    const size_t o = (size_t)first_pair;
    rc = epv_chain_launch(ctx, s->d_results + o, d_scales, n_pairs, d_poses);
    if (rc) return rc;
    rc = epv_cloud_launch(ctx, n_pairs, s->stride, s->d_results + o, d_scales, d_poses, s->d_xin + o * 4 * s->stride,
                          s->d_ninl + o, d_counts, d_limits, nullptr, 0, 0);
    if (rc) return rc;
    if (cap > 0) {
        rc = epv_cloud_launch(ctx, n_pairs, s->stride, s->d_results + o, d_scales, d_poses,
                              s->d_xin + o * 4 * s->stride, s->d_ninl + o, d_counts, d_limits, d_points, cap, 1);
        if (rc) return rc;
    }
    std::vector<int64_t> h_limits(np + 1);
    EPV_CUDA(ctx, cudaMemcpyAsync(h_limits.data(), d_limits, (np + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (poses) EPV_CUDA(ctx, cudaMemcpyAsync(poses, d_poses, (np + 1) * 128, cudaMemcpyDeviceToHost, ctx->stream));
    EPV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const int64_t total = h_limits[np];
    if (limits) memcpy(limits, h_limits.data(), np * 8);
    if (n_points) *n_points = total;
    if (cap > 0) {
        const int64_t w = std::min<int64_t>(total, cap);
        EPV_CUDA(ctx, cudaMemcpyAsync(points, d_points, (size_t)w * 24, cudaMemcpyDeviceToHost, ctx->stream));
        EPV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return EPIVO_OK;
}

int epivo_seq_stage_ms(epivo_seq* s, float* ms, int n) {
    if (!s || !ms) return EPIVO_ERR_INVALID;
    epivo_ctx* ctx = s->ctx;
    EPV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    constexpr int HALF = SEQ_MAX_CHUNKS / 2;
    for (int c = 0; c < s->last_mgroups; ++c) {
        float t = 0;
        EPV_CUDA(ctx, cudaEventElapsedTime(&t, s->ev[c][0], s->ev[c][1]));
        acc[1] += t;                // [1] match: plane pre-pass + key init + tile kernel
        EPV_CUDA(ctx, cudaEventElapsedTime(&t, s->evk[c][0], s->evk[c][1]));
        acc[7] += t;                // [7] matcher tile kernel alone, summed over the group launches
    }
    for (int c = 0; c < s->last_ggroups; ++c) {
        {                               // [2] sample + presolve (part of [3])
            float t = 0;
            EPV_CUDA(ctx, cudaEventElapsedTime(&t, s->ev[HALF + c][2], s->evp[HALF + c]));
            acc[2] += t;
        }
        for (int k = 2; k < 6; ++k) {   // [3] essential [4] pose [5] lm [6] finish
            float t = 0;
            EPV_CUDA(ctx, cudaEventElapsedTime(&t, s->ev[HALF + c][k], s->ev[HALF + c][k + 1]));
            acc[k + 1] += t;
        }
    }
    float tot = 0;
    if (s->last_mgroups > 0) EPV_CUDA(ctx, cudaEventElapsedTime(&tot, s->ev_begin, s->ev_end));
    acc[0] = tot;
    for (int i = 0; i < n; ++i) ms[i] = i < 8 ? acc[i] : (i == 8 ? (float)s->last_mgroups : 0.f);
    return EPIVO_OK;
}

int epivo_seq_get_matches(epivo_seq* s, int pair, int32_t* query_idx, int32_t* train_idx, int32_t* dist, int* n_out) {
    if (!s || !n_out) return EPIVO_ERR_INVALID;
    epivo_ctx* ctx = s->ctx;
    if (pair < 0 || pair >= s->n_list) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "pair index");
    int32_t n = 0;
    const size_t o = (size_t)pair * s->stride;
    EPV_CUDA(ctx, cudaMemcpyAsync(&n, s->d_nmatch + pair, 4, cudaMemcpyDeviceToHost, ctx->stream));
    EPV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (query_idx) EPV_CUDA(ctx, cudaMemcpyAsync(query_idx, s->d_mq + o, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (train_idx) EPV_CUDA(ctx, cudaMemcpyAsync(train_idx, s->d_mt + o, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (dist) EPV_CUDA(ctx, cudaMemcpyAsync(dist, s->d_md + o, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    EPV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *n_out = n;
    return EPIVO_OK;
}

int epivo_seq_get_masks(epivo_seq* s, int pair, uint8_t* e_mask, int* n_e, uint8_t* pose_mask, int* n_pose) {
    if (!s) return EPIVO_ERR_INVALID;
    epivo_ctx* ctx = s->ctx;
    if (pair < 0 || pair >= s->n_list) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "pair index");
    int32_t nm = 0, ni = 0;
    const size_t o = (size_t)pair * s->stride;
    EPV_CUDA(ctx, cudaMemcpyAsync(&nm, s->d_nmatch + pair, 4, cudaMemcpyDeviceToHost, ctx->stream));
    EPV_CUDA(ctx, cudaMemcpyAsync(&ni, s->d_ninl + pair, 4, cudaMemcpyDeviceToHost, ctx->stream));
    EPV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (e_mask) EPV_CUDA(ctx, cudaMemcpyAsync(e_mask, s->d_emask + o, (size_t)nm, cudaMemcpyDeviceToHost, ctx->stream));
    if (pose_mask) EPV_CUDA(ctx, cudaMemcpyAsync(pose_mask, s->d_pmask + o, (size_t)ni, cudaMemcpyDeviceToHost, ctx->stream));
    EPV_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (n_e) *n_e = nm;
    if (n_pose) *n_pose = ni;
    return EPIVO_OK;
}

// kitti_ba.cpp:757-905 (bundle_adjustment, mono) and 908-1068 (bundle_adjustment_stereo) over the pairs of the last run:
// ba.match_kp + ba.bundle_adjustment without the per-pair downloads.  Host: window plan and (node, node) -> pair lookup,
// every refusal before the first launch.  Device: ba_assemble_kernel (one launch) -> the batched window LM (epv_lm_launch,
// as epivo_lm_rt_batch calls it).  Host again: the sequential tail of ba.finish on the downloaded chains, O(windows x
// n_zeta).  Mono: a node is a frame, full reps weigh 1, translations carry the scale.  Stereo: frame f is nodes 2f (left)
// and 2f + 1 (right), each window entry becomes three reps (kitti_ba.cpp:934-941), a full rep weighs its pair's pair_w
// (NULL: 1), and there is no scale carry (:1054-1066).
static int seq_bundle_adjust(epivo_seq* s, bool stereo, int n_entry, const int32_t* first, const int32_t* second,
                             int stride, int num_frames, const double* pair_w, const double Kinv[9], double huber_delta,
                             double* opt_T, double* win_T, epivo_lm_res* lm, int32_t* iters, uint8_t* reverted,
                             int32_t* n_windows) {
    if (!s) return EPIVO_ERR_INVALID;
    epivo_ctx* ctx = s->ctx;
    if (!first || !second || !Kinv || !opt_T || !n_windows) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "null argument");
    if (n_entry < 1) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "n_rep = %d: the window needs at least one pair", n_entry);
    if (stride < 1) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "stride = %d < 1", stride);
    const int step = stereo ? 2 : 1;    // nodes per frame
    if (num_frames < 2 || num_frames > s->max_frames / step)
        EPV_FAIL(ctx, EPIVO_ERR_INVALID, "num_frames %d outside [2,%d]", num_frames, s->max_frames / step);
    if (s->last_run == epivo_seq::RUN_NONE)
        EPV_FAIL(ctx, EPIVO_ERR_INVALID, "no run over the current pair list (epivo_seq_run / _process / _process_frames)");
    if (s->last_run == epivo_seq::RUN_POINTS)
        EPV_FAIL(ctx, EPIVO_ERR_INVALID, "the last run was epivo_seq_process_points, which keeps no pixels");
    // window entries -> node pairs (stereo: ba.expand_stereo_window)
    std::vector<int32_t> na, nb;
    for (int j = 0; j < n_entry; ++j) {
        const int a = first[j], c = second[j];
        if (a < 0 || c < 0) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "window entry %d = (%d,%d) has a negative offset", j, a, c);
        if (a == c) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "window entry %d = (%d,%d) pairs a frame with itself", j, a, c);
        if (!stereo) {
            na.push_back(a);
            nb.push_back(c);
            continue;
        }
        if (a >= s->max_frames / 2 || c >= s->max_frames / 2)     // also keeps 2a + 1 in range
            EPV_FAIL(ctx, EPIVO_ERR_INVALID, "window entry %d = (%d,%d) reaches past the %d frames of the sequence", j, a,
                     c, s->max_frames / 2);
        na.insert(na.end(), {2 * a, 2 * a + 1, 2 * a});
        nb.insert(nb.end(), {2 * c, 2 * c, 2 * a + 1});
    }
    const int n_rep = (int)na.size();
    // window offsets -> reps and chain span (ba.window_reps, kitti_ba.cpp:810-815)
    int lo = INT32_MAX, hi = 0;
    std::vector<int32_t> reps((size_t)n_rep * 2);
    for (int j = 0; j < n_rep; ++j) {
        const int a = na[j], c = nb[j];
        reps[2 * j] = c > a ? a : a - 1;
        reps[2 * j + 1] = c > a ? c - 1 : c;
        lo = std::min(lo, std::min(a, c));
        hi = std::max(hi, std::max(a, c));
    }
    const int n_zeta = hi - lo;
    for (int j = 0; j < n_rep; ++j)      // ba.bundle_adjustment passes the reps unshifted: a window must start at offset 0
        if (reps[2 * j] >= n_zeta || reps[2 * j + 1] >= n_zeta)
            EPV_FAIL(ctx, EPIVO_ERR_INVALID, "rep %d = (%d,%d) outside the chain [0,%d)", j, reps[2 * j], reps[2 * j + 1], n_zeta);
    int rc = epv_lm_check_n32(ctx, n_zeta, n_rep);
    if (rc) return rc;
    if (pair_w)
        for (int p = 0; p < s->n_list; ++p)
            if (!std::isfinite(pair_w[p])) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "pair_w[%d] = %g is not finite", p, pair_w[p]);
    // window starts in frames (ba.window_starts, kitti_ba.cpp:780-801 / 943-963): span = the largest node offset
    const int nodes = step * num_frames;
    std::vector<int> starts;
    for (int i = 0; i < num_frames; i += stride) {
        if (step * i + hi >= nodes) break;
        starts.push_back(i);
    }
    const int B = (int)starts.size();
    // (node, node) -> the first pair of the list with that key; every key must lie in the last run
    std::unordered_map<int64_t, int> key;
    key.reserve(s->h_fq.size() * 2);
    for (size_t p = 0; p < s->h_fq.size(); ++p) key.emplace(((int64_t)s->h_fq[p] << 32) | (uint32_t)s->h_ft[p], (int)p);
    std::vector<int32_t> tab((size_t)B * (n_rep + n_zeta));
    auto lookup = [&](int b, int f0, int f1, int32_t* out) -> int {
        const auto it = key.find(((int64_t)f0 << 32) | (uint32_t)f1);
        if (it == key.end())
            EPV_FAIL(ctx, EPIVO_ERR_INVALID, "window %d (start %d) needs the pair (%d,%d), which is not in the pair list", b,
                     starts[b], f0, f1);
        if (it->second < s->last_first || it->second >= s->last_first + s->last_n_pairs)
            EPV_FAIL(ctx, EPIVO_ERR_INVALID, "the pair (%d,%d) is pair %d of the list, outside the last run [%d,+%d)", f0, f1,
                     it->second, s->last_first, s->last_n_pairs);
        *out = it->second;
        return EPIVO_OK;
    };
    for (int b = 0; b < B && !rc; ++b) {
        const int i = step * starts[b];
        for (int j = 0; j < n_rep && !rc; ++j) rc = lookup(b, i + na[j], i + nb[j], &tab[(size_t)b * n_rep + j]);
        for (int k = 0; k < n_zeta && !rc; ++k)
            rc = lookup(b, i + lo + k, i + lo + k + 1, &tab[(size_t)B * n_rep + (size_t)b * n_zeta + k]);
    }
    if (rc) return rc;
    for (int f = 0; f < nodes; ++f)
        for (int e = 0; e < 16; ++e) opt_T[(size_t)f * 16 + e] = (e % 5 == 0) ? 1.0 : 0.0;
    *n_windows = B;
    if (B == 0) return EPIVO_OK;
    // ---- device: assembly + LM
    EPV_CUDA(ctx, cudaSetDevice(ctx->device));
    EpvRange r_ba(ctx, stereo ? "epivo_seq_bundle_adjust_stereo" : "epivo_seq_bundle_adjust");
    const size_t nT = (size_t)B * n_zeta * 16, nP = (size_t)B * n_rep * BA_MIN_PT * 3, nW = (size_t)B * n_rep;
    const size_t n_tab = tab.size() + reps.size(), n_pw = pair_w ? (size_t)s->n_list : 0;
    rc = epv_ws_reserve(ctx, epv_align(n_tab * 4) + epv_align(n_pw * 8) + 2 * epv_align(nT * 8) + 2 * epv_align(nP * 8) +
                                 epv_align(nW * 8) + epv_align((size_t)B * sizeof(epivo_lm_res)) + epv_align((size_t)B * 4) +
                                 4096);
    if (rc) return rc;
    rc = epv_pin_reserve(ctx, epv_align(n_tab * 4) + epv_align(n_pw * 8) + 2 * epv_align(nT * 8) +
                                  epv_align((size_t)B * sizeof(epivo_lm_res)) + epv_align((size_t)B * 4) + 4096);
    if (rc) return rc;
    int32_t* d_tab = epv_ws_take<int32_t>(ctx, n_tab);
    double* d_pw = pair_w ? epv_ws_take<double>(ctx, n_pw) : nullptr;
    double* d_T0 = epv_ws_take<double>(ctx, nT);
    double* d_T = epv_ws_take<double>(ctx, nT);
    double* d_pr = epv_ws_take<double>(ctx, nP);
    double* d_p_r = epv_ws_take<double>(ctx, nP);
    double* d_w = epv_ws_take<double>(ctx, nW);
    epivo_lm_res* d_lm = epv_ws_take<epivo_lm_res>(ctx, B);
    int32_t* d_it = epv_ws_take<int32_t>(ctx, B);
    int32_t* h_tab = epv_pin_take<int32_t>(ctx, n_tab);
    double* h_pw = pair_w ? epv_pin_take<double>(ctx, n_pw) : nullptr;
    double* h_T0 = epv_pin_take<double>(ctx, nT);
    double* h_T = epv_pin_take<double>(ctx, nT);
    epivo_lm_res* h_lm = epv_pin_take<epivo_lm_res>(ctx, B);
    int32_t* h_it = epv_pin_take<int32_t>(ctx, B);
    memcpy(h_tab, tab.data(), tab.size() * 4);
    memcpy(h_tab + tab.size(), reps.data(), reps.size() * 4);
    cudaStream_t st = ctx->stream;
    EPV_CUDA(ctx, cudaMemcpyAsync(d_tab, h_tab, n_tab * 4, cudaMemcpyHostToDevice, st));
    if (pair_w) {
        memcpy(h_pw, pair_w, n_pw * 8);
        EPV_CUDA(ctx, cudaMemcpyAsync(d_pw, h_pw, n_pw * 8, cudaMemcpyHostToDevice, st));
    }
    BaKinv ki;
    memcpy(ki.k, Kinv, sizeof(ki.k));
    const bool tracks = s->last_run == epivo_seq::RUN_FRAMES;
    ba_assemble_kernel<<<dim3(n_rep, B), 256, 0, st>>>(d_tab, n_rep, n_zeta, s->stride, s->kp, ki, s->d_nmatch, s->d_ninl,
                                                       s->d_emask, s->d_pmask, s->d_R, s->d_t, s->d_fq, s->d_ft, s->d_mq,
                                                       s->d_mt, s->d_kps, tracks ? s->d_trk : nullptr, d_pw, d_T0, d_T,
                                                       d_pr, d_p_r, d_w);
    EPV_LAUNCHED(ctx);
    LmPlan lp{};
    lp.B = B;
    lp.n_zeta = n_zeta;
    lp.n_rep = n_rep;
    lp.N = BA_MIN_PT;
    lp.reps = d_tab + tab.size();
    lp.wreps = d_w;
    lp.epsilon = 1e-8;                   // kitti_ba.cpp:881
    lp.lambda0 = 1e-2;
    lp.huber_delta = huber_delta;
    lp.max_iters = 30;
    lp.T0s = d_T;
    lp.pr = d_pr;
    lp.p_r = d_p_r;
    lp.out = d_lm;
    lp.iters = d_it;
    lp.active = nullptr;
    // the kernel choice of epivo_lm_rt_batch for the same reps, so both routes run the same code on the same bytes
    lp.single_pair = (n_zeta == 1 && n_rep == 1 && reps[0] == 0 && reps[1] == 0) ? 1 : 0;
    {
        EpvRange r(ctx, "epivo: Levenberg_Marquardt (windows)");
        rc = epv_lm_launch(ctx, lp);
    }
    if (rc) return rc;
    EPV_CUDA(ctx, cudaMemcpyAsync(h_T0, d_T0, nT * 8, cudaMemcpyDeviceToHost, st));
    EPV_CUDA(ctx, cudaMemcpyAsync(h_T, d_T, nT * 8, cudaMemcpyDeviceToHost, st));
    EPV_CUDA(ctx, cudaMemcpyAsync(h_lm, d_lm, (size_t)B * sizeof(epivo_lm_res), cudaMemcpyDeviceToHost, st));
    EPV_CUDA(ctx, cudaMemcpyAsync(h_it, d_it, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    EPV_CUDA(ctx, cudaStreamSynchronize(st));
    // ---- host: ba.finish (kitti_ba.cpp:853-856, 889-903 / 1054-1066).  A window whose r_norm exceeds 1e-2 keeps its
    // initial chain (NaN does not revert, as in the reference's comparison); mono: a window that starts on an optimized
    // frame divides its translations by that frame's translation norm (stereo keeps scale 1, an exact division); later
    // windows overwrite the overlap.
    std::vector<uint8_t> optimized((size_t)nodes, 0);
    for (int b = 0; b < B; ++b) {
        const int w0 = step * starts[b] + lo;
        double scale = 1.0;
        if (!stereo && optimized[w0]) {
            const double* tw = opt_T + (size_t)w0 * 16;
            const double xx = tw[3] * tw[3], yy = tw[7] * tw[7], zz = tw[11] * tw[11];
            scale = std::sqrt((xx + yy) + zz);
        }
        const bool rev = h_lm[b].r_norm > 1e-2;
        const double* Ts = (rev ? h_T0 : h_T) + (size_t)b * n_zeta * 16;
        for (int k = 0; k < n_zeta; ++k) {
            double* o = opt_T + (size_t)(w0 + k) * 16;
            memcpy(o, Ts + (size_t)k * 16, 128);
            o[3] /= scale;
            o[7] /= scale;
            o[11] /= scale;
            optimized[w0 + k] = 1;
        }
        if (reverted) reverted[b] = rev ? 1 : 0;
    }
    if (win_T) memcpy(win_T, h_T, nT * 8);
    if (lm) memcpy(lm, h_lm, (size_t)B * sizeof(epivo_lm_res));
    if (iters) memcpy(iters, h_it, (size_t)B * 4);
    return EPIVO_OK;
}

int epivo_seq_bundle_adjust(epivo_seq* s, int n_rep, const int32_t* first, const int32_t* second, int stride,
                            int num_frames, const double Kinv[9], double huber_delta, double* opt_T, double* win_T,
                            epivo_lm_res* lm, int32_t* iters, uint8_t* reverted, int32_t* n_windows) {
    return seq_bundle_adjust(s, false, n_rep, first, second, stride, num_frames, nullptr, Kinv, huber_delta, opt_T, win_T,
                             lm, iters, reverted, n_windows);
}

int epivo_seq_bundle_adjust_stereo(epivo_seq* s, int n_rep, const int32_t* first, const int32_t* second, int stride,
                                   int num_frames, const double* pair_w, const double Kinv[9], double huber_delta,
                                   double* opt_T, double* win_T, epivo_lm_res* lm, int32_t* iters, uint8_t* reverted,
                                   int32_t* n_windows) {
    return seq_bundle_adjust(s, true, n_rep, first, second, stride, num_frames, pair_w, Kinv, huber_delta, opt_T, win_T,
                             lm, iters, reverted, n_windows);
}

}  // extern "C"
