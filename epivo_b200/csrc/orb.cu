// N4 front end, descriptor extractor: cv::ORB::detectAndCompute as the reference configures it
//     Ptr<ORB> orb = ORB::create(10000, 1.2f, 8, 15, 0, 2, ORB::FAST_SCORE);   kitti_ba.cpp:128
//     orb->detect(src, kp); orb->compute(src, kp, desc);                        kitti_ba.cpp:131-152
// for a batch of 8-bit images, bit-exact with OpenCV (modules/features2d/src/orb.cpp restated): keypoint coordinates,
// order, size, angle, response, octave and the 256-bit descriptors.  Byte / integer work except for two short float32
// chains (the angle polynomial, the Gaussian blur) that are spelled with round-to-nearest intrinsics in OpenCV's order.
//
//   pyramid      level k = INTER_LINEAR_EXACT resize of level k-1 (8.8 fixed-point weights, one rounding)    orb_resize_kernel
//   detection    FAST-9/16 (fastThreshold, non-max suppression) per level                                     frontend.cu
//   selection    border filter (edgeThreshold) + KeyPointsFilter::retainBest(nfeaturesPerLevel): keeps every
//                corner whose score is >= the n-th best one, in the order libstdc++'s std::nth_element +
//                std::partition leave them in -- reproduced by running those two algorithms, each partition
//                pass as two ordered compactions + independent swaps on a block of threads                    orb_select_kernel
//   orientation  intensity centroid of the radius-15 disc, fastAtan2's polynomial                             orb_describe_kernel
//   blur         GaussianBlur(7 x 7, sigma 2) as OpenCV runs it on a ROI: sepFilter2D in float32              orb_blur_kernel
//   descriptor   256 steered BRIEF tests (WTA_K 2) on the blurred level; samples that leave the level read
//                its unblurred BORDER_REFLECT_101 margin, as OpenCV's level-with-margin buffer holds it       orb_describe_kernel
#include <math.h>

#include <vector>

#include "orb_select.cuh"
#include "stages.cuh"

namespace {

constexpr int ORB_MAX_LEVELS = 16;
constexpr int ORB_PATCH_RADIUS = 15;
constexpr int ORB_PATCH = 31;

struct OrbGeom {
    int nlevels, n_images, edge, max_kp;
    int rows[ORB_MAX_LEVELS], cols[ORB_MAX_LEVELS];
    int nfeat[ORB_MAX_LEVELS];          // retainBest budget per level
    int cap[ORB_MAX_LEVELS];            // candidate slots per image and level (no FAST result can exceed it)
    int64_t img_off[ORB_MAX_LEVELS];    // byte offset of level l's block [n_images][rows][cols]
    int64_t cand_off[ORB_MAX_LEVELS];   // element offset of level l's block [n_images][cap] in the candidate arrays
    float scale[ORB_MAX_LEVELS];
};

// ---- pyramid ------------------------------------------------------------------------------------------------------------
// tab = ofs << 9 | c1: source offset and the 8.8 weight of the second tap (c0 = 256 - c1); the edge-copy ranges of
// OpenCV's resize (destination indices whose source falls outside) are folded in as c1 = 0 on the edge pixel.
__global__ void __launch_bounds__(256) orb_resize_kernel(const uint8_t* __restrict__ src, int srows, int scols,
                                                         uint8_t* __restrict__ dst, int drows, int dcols,
                                                         const uint32_t* __restrict__ xtab, const uint32_t* __restrict__ ytab) {
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x >= dcols || y >= drows) return;
    const uint8_t* s = src + (size_t)blockIdx.z * srows * scols;
    const uint32_t tx = xtab[x], ty = ytab[y];
    const int ox = tx >> 9, x1 = tx & 511, x0 = 256 - x1;
    const int oy = ty >> 9, y1 = ty & 511, y0 = 256 - y1;
    const int ox1 = min(ox + 1, scols - 1), oy1 = min(oy + 1, srows - 1);
    const int top = s[(size_t)oy * scols + ox] * x0 + s[(size_t)oy * scols + ox1] * x1;      // ufixedpoint16 rows
    const int bot = s[(size_t)oy1 * scols + ox] * x0 + s[(size_t)oy1 * scols + ox1] * x1;
    const int v = (top * y0 + bot * y1 + (1 << 15)) >> 16;                                   // ufixedpoint32 -> uchar
    dst[(size_t)blockIdx.z * drows * dcols + (size_t)y * dcols + x] = (uint8_t)min(v, 255);
}

// borderInterpolate(i, n, BORDER_REFLECT_101), any distance outside
__device__ __forceinline__ int reflect101(int i, int n) {
    if (n == 1) return 0;
    while ((unsigned)i >= (unsigned)n) i = i < 0 ? -i : 2 * (n - 1) - i;
    return i;
}

// ---- blur ---------------------------------------------------------------------------------------------------------------
// getGaussianKernel(7, 2, CV_32F)
__constant__ float c_gauss7[7] = {0x1.1f5f62p-4f, 0x1.0c70fcp-3f, 0x1.869472p-3f, 0x1.ba95cp-3f,
                                  0x1.869472p-3f, 0x1.0c70fcp-3f, 0x1.1f5f62p-4f};
constexpr int BL_X = 32, BL_Y = 16;

// rows:  s = k[0]*p[0]; s = fma(k[i], p[i], s), i = 1..6        (filter.simd.hpp RowFilter<uchar, float>, AVX2 build)
// cols:  s = k[3]*r[0]; s = fma(k[3+i], r[i] + r[-i], s), i = 1..3; cvRound, saturate   (SymmColumnFilter<float, uchar>)
__global__ void __launch_bounds__(BL_X * BL_Y) orb_blur_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst,
                                                               int rows, int cols) {
    __shared__ uint8_t tile[BL_Y + 6][BL_X + 8];
    __shared__ float H[BL_Y + 6][BL_X];
    const int x0 = blockIdx.x * BL_X, y0 = blockIdx.y * BL_Y;
    const uint8_t* s = src + (size_t)blockIdx.z * rows * cols;
    const int tid = threadIdx.y * BL_X + threadIdx.x;
    for (int i = tid; i < (BL_Y + 6) * (BL_X + 6); i += BL_X * BL_Y) {
        const int ty = i / (BL_X + 6), tx = i % (BL_X + 6);
        const int gx = reflect101(x0 + tx - 3, cols), gy = reflect101(y0 + ty - 3, rows);
        tile[ty][tx] = s[(size_t)gy * cols + gx];
    }
    __syncthreads();
    for (int i = tid; i < (BL_Y + 6) * BL_X; i += BL_X * BL_Y) {
        const int ty = i / BL_X, tx = i % BL_X;
        float a = __fmul_rn(c_gauss7[0], (float)tile[ty][tx]);
#pragma unroll
        for (int k = 1; k < 7; ++k) a = __fmaf_rn(c_gauss7[k], (float)tile[ty][tx + k], a);
        H[ty][tx] = a;
    }
    __syncthreads();
    const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
    if (x >= cols || y >= rows) return;
    const int ty = threadIdx.y + 3, tx = threadIdx.x;
    float a = __fmul_rn(c_gauss7[3], H[ty][tx]);
#pragma unroll
    for (int k = 1; k <= 3; ++k) a = __fmaf_rn(c_gauss7[3 + k], __fadd_rn(H[ty + k][tx], H[ty - k][tx]), a);
    const int q = __float2int_rn(a);
    dst[(size_t)blockIdx.z * rows * cols + (size_t)y * cols + x] = (uint8_t)min(max(q, 0), 255);
}

// ---- selection ------------------------------------------------------------------------------------------------------------
// orb_retain_best_block (orb_select.cuh): libstdc++'s std::nth_element + std::partition on packed keys
constexpr int SEL_T = 512;                                    // threads of the selection CTA

// the block of threads orb_retain_best_block runs on (orb_select.cuh)
struct OrbSelectBlockExec {
    int* s_cnt;                                               // 2 x 16 warp counts + 2 running offsets, shared memory
    __device__ int tid() const { return threadIdx.x; }
    __device__ int nthreads() const { return SEL_T; }
    __device__ void sync() const { __syncthreads(); }
    __device__ void imin(int* p, int v) const { atomicMin(p, v); }
    // A gets every c in [0, m) with fa(c) in ascending order, B likewise with fb
    template <class FA, class FB>
    __device__ void compact2(int m, FA fa, FB fb, uint32_t* A, uint32_t* B, int* nA, int* nB) const {
        const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
        int* wa = s_cnt;
        int* wb = s_cnt + SEL_T / 32;
        int* off = s_cnt + 2 * (SEL_T / 32);
        if (t == 0) off[0] = off[1] = 0;
        __syncthreads();
        for (int base = 0; base < m; base += SEL_T) {
            const int c = base + t;
            const bool a = c < m && fa(c), b = c < m && fb(c);
            const unsigned ba = __ballot_sync(0xFFFFFFFFu, a), bb = __ballot_sync(0xFFFFFFFFu, b);
            if (lane == 0) {
                wa[warp] = __popc(ba);
                wb[warp] = __popc(bb);
            }
            __syncthreads();
            int oa = off[0], ob = off[1];
            for (int w = 0; w < warp; ++w) {
                oa += wa[w];
                ob += wb[w];
            }
            const unsigned lt = (1u << lane) - 1;
            if (a) A[oa + __popc(ba & lt)] = (uint32_t)c;
            if (b) B[ob + __popc(bb & lt)] = (uint32_t)c;
            __syncthreads();
            if (t == SEL_T - 1) {
                off[0] = oa + __popc(ba);
                off[1] = ob + __popc(bb);
            }
            __syncthreads();
        }
        if (t == 0) {
            *nA = off[0];
            *nB = off[1];
        }
        __syncthreads();
    }
};

// one CTA per (image, level): border filter in FAST's order, then retainBest.  sel[level block][image][k] = candidate
// index of the k-th kept keypoint; sel_cnt[image][level] = how many.  Keys and the two stop lists of a partition pass
// live in shared memory when the level's candidates fit (smem_keys each), else in HBM (the sel slot and scratch).
__global__ void __launch_bounds__(SEL_T) orb_select_kernel(OrbGeom g, const float* __restrict__ cand_kps,
                                                           const float* __restrict__ cand_resp,
                                                           const int32_t* __restrict__ cand_cnt, uint32_t* __restrict__ sel,
                                                           uint32_t* __restrict__ scratch, int32_t* __restrict__ sel_cnt,
                                                           int smem_keys) {
    extern __shared__ uint32_t s_keys[];
    __shared__ int s_cnt[2 * (SEL_T / 32) + 2];
    __shared__ OrbSelectShared s_sh;
    const int img = blockIdx.x, lv = blockIdx.y;
    const int tid = threadIdx.x;
    const int cap = g.cap[lv], rows = g.rows[lv], cols = g.cols[lv], edge = g.edge;
    const int n = min(cand_cnt[lv * g.n_images + img], cap);
    const float* kp = cand_kps + (g.cand_off[lv] + (int64_t)img * cap) * 2;
    const float* rs = cand_resp + g.cand_off[lv] + (int64_t)img * cap;
    uint32_t* out = sel + g.cand_off[lv] + (int64_t)img * cap;
    uint32_t* scr = scratch + (g.cand_off[lv] + (int64_t)img * cap) * 2;
    const bool room = rows > 2 * edge && cols > 2 * edge;
    OrbSelectBlockExec ex{s_cnt};
    // survivors of the border filter, in FAST's order (A; B is not needed here)
    uint32_t* A = scr;
    uint32_t* B = scr + cap;
    ex.compact2(n, [&](int j) {
        const float x = kp[2 * j], y = kp[2 * j + 1];
        return room && x >= edge && x < cols - edge && y >= edge && y < rows - edge;              // Rect::contains
    }, [](int) { return false; }, A, B, &s_sh.nA, &s_sh.nB);
    const int nf = s_sh.nA;
    const bool in_smem = nf <= smem_keys;
    uint32_t* keys = in_smem ? s_keys : out;
    for (int i = tid; i < nf; i += SEL_T) {
        const uint32_t j = A[i];
        keys[i] = ((uint32_t)rs[j] << 24) | j;
    }
    __syncthreads();
    if (in_smem) {
        A = s_keys + smem_keys;
        B = s_keys + 2 * smem_keys;
    }
    const int n_points = g.nfeat[lv];
    int kept = nf;
    if (nf > n_points) kept = n_points == 0 ? 0 : orb_retain_best_block(ex, keys, nf, n_points, A, B, &s_sh);
    __syncthreads();
    if (tid == 0) sel_cnt[img * g.nlevels + lv] = kept;
    for (int i = tid; i < kept; i += SEL_T) out[i] = keys[i] & 0xFFFFFFu;
}

// one thread per image: where each level's keypoints start in the image's output, and the total
__global__ void orb_offsets_kernel(OrbGeom g, const int32_t* __restrict__ sel_cnt, int32_t* __restrict__ base,
                                   int32_t* __restrict__ counts) {
    const int img = blockIdx.x * blockDim.x + threadIdx.x;
    if (img >= g.n_images) return;
    int acc = 0;
    for (int l = 0; l < g.nlevels; ++l) {
        base[img * (ORB_MAX_LEVELS + 1) + l] = acc;
        acc += sel_cnt[img * g.nlevels + l];
    }
    base[img * (ORB_MAX_LEVELS + 1) + g.nlevels] = acc;
    counts[img] = acc;
}

// ---- orientation + descriptor ---------------------------------------------------------------------------------------------
__constant__ int8_t c_umax[16] = {15, 15, 15, 15, 14, 14, 14, 13, 13, 12, 11, 10, 9, 8, 6, 3};
// ORB's learned sampling pattern for patch size 31 (orb.cpp bit_pattern_31_): 256 tests x (x0, y0, x1, y1)
__constant__ int8_t c_pattern[256 * 4] = {
#include "orb_pattern.inc"
};

// cv::fastAtan2 (mathfuncs_core atan_f32), degrees; every operation rounded on its own, as cv2 evaluates it
__device__ __forceinline__ float orb_fast_atan2(float y, float x) {
    const float p1 = 0x1.ca44dep+5f, p3 = -0x1.2aaddcp+4f, p5 = 0x1.1d3f7ep+3f, p7 = -0x1.4515b2p+1f;
    const float eps = 0x1p-52f;                                          // (float)DBL_EPSILON
    const float ax = fabsf(x), ay = fabsf(y);
    float a, c, c2;
    if (ax >= ay) {
        c = __fdiv_rn(ay, __fadd_rn(ax, eps));
        c2 = __fmul_rn(c, c);
        a = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c);
    } else {
        c = __fdiv_rn(ax, __fadd_rn(ay, eps));
        c2 = __fmul_rn(c, c);
        a = __fsub_rn(90.f, __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c));
    }
    if (x < 0) a = __fsub_rn(180.f, a);
    if (y < 0) a = __fsub_rn(360.f, a);
    return a;
}

struct OrbKp {             // = cv::KeyPoint's memory layout (epivo_keypoint in the header)
    float x, y, size, angle, response;
    int32_t octave, class_id;
};

// one warp per kept keypoint: orientation (ICAngles), KeyPoint fields, 32 descriptor bytes (one per lane)
__global__ void __launch_bounds__(256) orb_describe_kernel(OrbGeom g, const uint8_t* __restrict__ pyr,
                                                           const uint8_t* __restrict__ blur, const float* __restrict__ cand_kps,
                                                           const float* __restrict__ cand_resp, const uint32_t* __restrict__ sel,
                                                           const int32_t* __restrict__ base, OrbKp* __restrict__ kps_out,
                                                           uint8_t* __restrict__ desc_out) {
    __shared__ int8_t s_pat[256 * 4];
    for (int i = threadIdx.x; i < 256 * 4; i += 256) s_pat[i] = c_pattern[i];
    __syncthreads();
    const int img = blockIdx.y, lane = threadIdx.x & 31;
    const int32_t* b = base + img * (ORB_MAX_LEVELS + 1);
    const int total = min(b[g.nlevels], g.max_kp);
    for (int k = blockIdx.x * 8 + (threadIdx.x >> 5); k < total; k += gridDim.x * 8) {
        int lv = 0;
        while (lv + 1 < g.nlevels && k >= b[lv + 1]) ++lv;
        const int rows = g.rows[lv], cols = g.cols[lv], cap = g.cap[lv];
        const int64_t slot = g.cand_off[lv] + (int64_t)img * cap;
        const uint32_t j = sel[slot + (k - b[lv])];
        const float fx = cand_kps[(slot + j) * 2], fy = cand_kps[(slot + j) * 2 + 1];
        const int x = (int)fx, y = (int)fy;
        const uint8_t* im = pyr + g.img_off[lv] + (size_t)img * rows * cols;
        const uint8_t* bl = blur + g.img_off[lv] + (size_t)img * rows * cols;
        // ICAngles: m_10 = sum u I(u, v), m_01 = sum v I(u, v) over the disc; lane = column u + 15
        int m10 = 0, m01 = 0;
        if (lane < ORB_PATCH) {
            const int u = lane - ORB_PATCH_RADIUS, au = abs(u);
            const uint8_t* c = im + (size_t)y * cols + (x + u);
            int col = c[0];
            for (int v = 1; v <= ORB_PATCH_RADIUS; ++v) {
                if (au > c_umax[v]) break;                                // umax decreases with v
                const int plus = c[(ptrdiff_t)v * cols], minus = c[-(ptrdiff_t)v * cols];
                col += plus + minus;
                m01 += v * (plus - minus);
            }
            m10 = u * col;
        }
        m10 = __reduce_add_sync(0xFFFFFFFFu, m10);
        m01 = __reduce_add_sync(0xFFFFFFFFu, m01);
        const float angle = orb_fast_atan2((float)m01, (float)m10);
        const float sc = g.scale[lv];
        const float px = __fmul_rn(fx, sc), py = __fmul_rn(fy, sc);        // pt *= scale
        if (lane == 0) {
            OrbKp o;
            o.x = px;
            o.y = py;
            o.size = __fmul_rn((float)ORB_PATCH, sc);
            o.angle = angle;
            o.response = cand_resp[slot + j];
            o.octave = lv;
            o.class_id = -1;
            kps_out[(size_t)img * g.max_kp + k] = o;
        }
        // computeOrbDescriptors
        const float inv = __fdiv_rn(1.f, sc);
        const float ang = __fmul_rn(angle, 0x1.1df46ap-6f);                // angle *= (float)(CV_PI/180.f)
        const float ca = (float)cos((double)ang), sa = (float)sin((double)ang);
        const int cx = __float2int_rn(__fmul_rn(px, inv)), cy = __float2int_rn(__fmul_rn(py, inv));
        unsigned byte = 0;
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            const int8_t* p = s_pat + (lane * 8 + t) * 4;
            int val[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const float qx = (float)p[2 * h], qy = (float)p[2 * h + 1];
                const int ix = __float2int_rn(__fsub_rn(__fmul_rn(qx, ca), __fmul_rn(qy, sa)));
                const int iy = __float2int_rn(__fadd_rn(__fmul_rn(qx, sa), __fmul_rn(qy, ca)));
                const int sx = cx + ix, sy = cy + iy;
                if (sx >= 0 && sx < cols && sy >= 0 && sy < rows) val[h] = bl[(size_t)sy * cols + sx];
                else val[h] = im[(size_t)reflect101(sy, rows) * cols + reflect101(sx, cols)];   // the unblurred margin
            }
            byte |= (val[0] < val[1] ? 1u : 0u) << t;
        }
        desc_out[((size_t)img * g.max_kp + k) * 32 + lane] = (uint8_t)byte;
    }
}

// interpolationLinear<ufixedpoint16>::getCoeffs (resize.cpp) for every destination index, in double as OpenCV's
// softdouble computes it; edge-copy ranges folded in
void orb_resize_table(int src, int dst, uint32_t* tab) {
    const double inv_scale = (double)dst / (double)src;
    const double scale = 1.0 / inv_scale;
    std::vector<int> ofs(dst, 0), c1(dst, 0);
    int lo = 0, hi = dst;
    for (int v = 0; v < dst; ++v) {
        const double fval = scale * ((double)v + 0.5) - 0.5;
        const int iv = (int)floor(fval);
        if (iv >= 0 && src > 1) {
            if (iv < src - 1) {
                ofs[v] = iv;
                c1[v] = (int)nearbyint((fval - iv) * 256.0);
            } else {
                ofs[v] = src - 1;
                hi = std::min(hi, v);
            }
        } else {
            lo = std::max(lo, v + 1);
        }
    }
    for (int v = 0; v < dst; ++v) {
        if (v < lo) tab[v] = 0;
        else if (v >= hi) tab[v] = (uint32_t)(src - 1) << 9;
        else tab[v] = ((uint32_t)ofs[v] << 9) | (uint32_t)c1[v];
    }
}

}  // namespace

// ORB_Impl::detectAndCompute's host-side set-up: level scales (getScale), level sizes, feature budget per level
int epv_orb_plan(epivo_ctx* ctx, int n_images, int rows, int cols, int nfeatures, float scale_factor, int nlevels,
                 int edge_threshold, int max_kp, EpvOrbPlan* plan) {
    if (nlevels < 1 || nlevels > ORB_MAX_LEVELS) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "nlevels %d outside [1, %d]", nlevels, ORB_MAX_LEVELS);
    if (!(scale_factor > 1.0f) || scale_factor > 2.0f) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "scale_factor %g outside (1, 2]", scale_factor);
    if (edge_threshold < ORB_PATCH_RADIUS)       // the orientation disc must stay inside the level
        EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "edge_threshold %d below the patch radius %d", edge_threshold, ORB_PATCH_RADIUS);
    if (nfeatures < 0) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "negative nfeatures");
    OrbGeom& g = *reinterpret_cast<OrbGeom*>(plan->geom);
    static_assert(sizeof(OrbGeom) <= sizeof(plan->geom), "EpvOrbPlan::geom too small");
    g.nlevels = nlevels;
    g.n_images = n_images;
    g.edge = edge_threshold;
    g.max_kp = max_kp;
    int64_t img_off = 0, cand_off = 0;
    plan->tab_entries = 0;
    for (int l = 0; l < nlevels; ++l) {
        const float s = (float)pow((double)scale_factor, (double)l);      // getScale(level, firstLevel = 0, scaleFactor)
        g.scale[l] = s;
        const float inv = 1.f / s;                                         // float inv_scale = 1.f / scale;
        g.cols[l] = (int)lrintf((float)cols * inv);                        // Size sz(cvRound(cols*inv_scale), cvRound(rows*inv_scale)):
        g.rows[l] = (int)lrintf((float)rows * inv);                        // 285 columns at 1.2f are 238 this way, 237 by division
        if (g.rows[l] < 1 || g.cols[l] < 1) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "level %d of a %d x %d image is empty", l, rows, cols);
        g.cap[l] = ((g.rows[l] + 1) / 2) * ((g.cols[l] + 1) / 2) + 1;      // suppressed corners are never 8-neighbours
        if (g.cap[l] >= (1 << 24)) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "image too large");
        g.img_off[l] = img_off;
        g.cand_off[l] = cand_off;
        img_off += (int64_t)epv_align((size_t)n_images * g.rows[l] * g.cols[l]);
        cand_off += (int64_t)n_images * g.cap[l];
        if (l > 0) plan->tab_entries += g.rows[l] + g.cols[l];
    }
    plan->pyr_bytes = (size_t)img_off;
    plan->cand_total = (size_t)cand_off;
    // computeKeyPoints: nfeatures split geometrically over the levels, float arithmetic as in orb.cpp
    const float factor = (float)(1.0 / (double)scale_factor);
    float nd = (float)nfeatures * (1 - factor) / (1 - (float)pow((double)factor, (double)nlevels));
    int sum = 0;
    for (int l = 0; l < nlevels - 1; ++l) {
        g.nfeat[l] = (int)lrintf(nd);
        sum += g.nfeat[l];
        nd *= factor;
    }
    g.nfeat[nlevels - 1] = std::max(nfeatures - sum, 0);
    return EPIVO_OK;
}

int epivo_orb_level_geometry(int rows, int cols, int nfeatures, float scale_factor, int nlevels, int32_t* level_rows,
                             int32_t* level_cols, int32_t* level_features) {
    if (rows <= 0 || cols <= 0 || !level_rows || !level_cols || !level_features) return EPIVO_ERR_INVALID;
    epivo_ctx scratch;                         // host-only: carries the error text of epv_orb_plan, no CUDA call is made
    EpvOrbPlan plan;
    const int rc = epv_orb_plan(&scratch, 1, rows, cols, nfeatures, scale_factor, nlevels, ORB_PATCH_RADIUS, 0, &plan);
    if (rc) return rc;
    const OrbGeom& g = *reinterpret_cast<const OrbGeom*>(plan.geom);
    for (int l = 0; l < nlevels; ++l) {
        level_rows[l] = g.rows[l];
        level_cols[l] = g.cols[l];
        level_features[l] = g.nfeat[l];
    }
    return EPIVO_OK;
}

size_t epv_orb_work_bytes(const EpvOrbPlan& plan) {
    const OrbGeom& g = *reinterpret_cast<const OrbGeom*>(plan.geom);
    return 2 * plan.pyr_bytes + epv_fast_work_bytes(g.n_images, g.rows[0], g.cols[0]) + plan.cand_total * 24 +
           (size_t)plan.tab_entries * 4 + (size_t)g.n_images * (ORB_MAX_LEVELS * 3 + 2) * 4 + 16 * 4096;
}

// d_pyr: plan.pyr_bytes with the images already at offset 0 ([n_images][rows][cols]); d_kps: [n_images][max_kp] of
// epivo_keypoint; d_desc: [n_images][max_kp][32]; d_counts: [n_images] keypoints FOUND (only the first max_kp stored).
// h_tab: pinned host staging for the resize tables (plan.tab_entries words), must stay valid until the stream drains.
int epv_orb_launch(epivo_ctx* ctx, const EpvOrbPlan& plan, int fast_threshold, uint8_t* d_pyr, void* d_kps,
                   uint8_t* d_desc, int32_t* d_counts, uint32_t* h_tab) {
    const OrbGeom& g = *reinterpret_cast<const OrbGeom*>(plan.geom);
    const int n_images = g.n_images;
    if (n_images <= 0) return EPIVO_OK;
    if (n_images > 65535) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "more than 65535 images per call");
    cudaStream_t st = ctx->stream;
    uint8_t* d_blur = epv_ws_take<uint8_t>(ctx, plan.pyr_bytes);
    uint8_t* d_fast = epv_ws_take<uint8_t>(ctx, epv_fast_work_bytes(n_images, g.rows[0], g.cols[0]));
    float* cand_kps = epv_ws_take<float>(ctx, plan.cand_total * 2);
    float* cand_resp = epv_ws_take<float>(ctx, plan.cand_total);
    uint32_t* sel = epv_ws_take<uint32_t>(ctx, plan.cand_total);
    uint32_t* scratch = epv_ws_take<uint32_t>(ctx, plan.cand_total * 2);
    uint32_t* d_tab = epv_ws_take<uint32_t>(ctx, plan.tab_entries + 1);
    int32_t* cand_cnt = epv_ws_take<int32_t>(ctx, (size_t)n_images * ORB_MAX_LEVELS);
    int32_t* sel_cnt = epv_ws_take<int32_t>(ctx, (size_t)n_images * ORB_MAX_LEVELS);
    int32_t* base = epv_ws_take<int32_t>(ctx, (size_t)n_images * (ORB_MAX_LEVELS + 1));
    // pyramid
    {
        EpvRange r(ctx, "orb_pyramid");
        size_t at = 0;
        for (int l = 1; l < g.nlevels; ++l) {
            orb_resize_table(g.cols[l - 1], g.cols[l], h_tab + at);
            orb_resize_table(g.rows[l - 1], g.rows[l], h_tab + at + g.cols[l]);
            at += g.cols[l] + g.rows[l];
        }
        if (at) EPV_CUDA(ctx, cudaMemcpyAsync(d_tab, h_tab, at * 4, cudaMemcpyHostToDevice, st));
        at = 0;
        for (int l = 1; l < g.nlevels; ++l) {
            const dim3 grid((g.cols[l] + 31) / 32, (g.rows[l] + 7) / 8, n_images);
            orb_resize_kernel<<<grid, dim3(32, 8), 0, st>>>(d_pyr + g.img_off[l - 1], g.rows[l - 1], g.cols[l - 1],
                                                            d_pyr + g.img_off[l], g.rows[l], g.cols[l], d_tab + at,
                                                            d_tab + at + g.cols[l]);
            EPV_LAUNCHED(ctx);
            at += g.cols[l] + g.rows[l];
        }
    }
    // FAST per level + blur per level
    {
        EpvRange r(ctx, "orb_fast_blur");
        EPV_CUDA(ctx, cudaMemsetAsync(cand_cnt, 0, (size_t)n_images * ORB_MAX_LEVELS * 4, st));
        for (int l = 0; l < g.nlevels; ++l) {
            if (g.rows[l] >= 7 && g.cols[l] >= 7) {
                const int rc = epv_fast_launch(ctx, d_pyr + g.img_off[l], n_images, g.rows[l], g.cols[l], fast_threshold, 1,
                                               g.cap[l], cand_kps + g.cand_off[l] * 2, cand_resp + g.cand_off[l],
                                               cand_cnt + (size_t)l * n_images, d_fast);
                if (rc) return rc;
            }
            const dim3 grid((g.cols[l] + BL_X - 1) / BL_X, (g.rows[l] + BL_Y - 1) / BL_Y, n_images);
            orb_blur_kernel<<<grid, dim3(BL_X, BL_Y), 0, st>>>(d_pyr + g.img_off[l], d_blur + g.img_off[l], g.rows[l], g.cols[l]);
            EPV_LAUNCHED(ctx);
        }
    }
    {
        EpvRange r(ctx, "orb_select_describe");
        int max_cap = 0;
        for (int l = 0; l < g.nlevels; ++l) max_cap = std::max(max_cap, g.cap[l]);
        const int smem_keys = std::min(max_cap, 16 * 1024);                // keys + two stop lists: 192 KB at most; larger sets select in HBM
        EPV_CUDA(ctx, cudaFuncSetAttribute(orb_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_keys * 12));
        orb_select_kernel<<<dim3(n_images, g.nlevels), SEL_T, (size_t)smem_keys * 12, st>>>(g, cand_kps, cand_resp, cand_cnt, sel,
                                                                                            scratch, sel_cnt, smem_keys);
        EPV_LAUNCHED(ctx);
        orb_offsets_kernel<<<(n_images + 127) / 128, 128, 0, st>>>(g, sel_cnt, base, d_counts);
        EPV_LAUNCHED(ctx);
        if (g.max_kp > 0) {
            const int bx = std::max(1, std::min((g.max_kp + 7) / 8, 4 * ctx->sm_count));
            orb_describe_kernel<<<dim3(bx, n_images), 256, 0, st>>>(g, d_pyr, d_blur, cand_kps, cand_resp, sel, base,
                                                                    (OrbKp*)d_kps, d_desc);
            EPV_LAUNCHED(ctx);
        }
    }
    return EPIVO_OK;
}
