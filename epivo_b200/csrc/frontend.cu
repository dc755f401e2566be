// N4 front end, detector part: cv::FastFeatureDetector (FAST-9/16, OpenCV features2d/src/fast.cpp FAST_t<16>)
// for a batch of 8-bit images, as the reference calls it:
//   FastFeatureDetector::create(40)->detect(src, kp0, Mat())   kitti_E.cpp:71-74, kitti_ba.cpp:49,62
//   FastFeatureDetector::create()  ->detect(...)  (threshold 10) kitti_ba.cpp:98,117-118
// Integer / byte work bound by HBM (one read of the image, one 2-byte score write and read per pixel): the
// result -- keypoint coordinates, their order and the response -- is bit-exact with OpenCV.
//
// OpenCV's loop, restated:  a pixel (x, y) with 3 <= x < cols-3, 3 <= y < rows-3 is a corner when 9 contiguous
// pixels of its 16-pixel Bresenham circle are all darker than v - t or all brighter than v + t (the pair-wise
// rejection cascade in front of that test never rejects a corner: 9 contiguous of 16 contain one pixel of every
// antipodal pair).  With non-maximum suppression a corner is kept when its score -- cornerScore<16>: the largest
// threshold for which it is still a corner -- is strictly greater than the scores of its 8 neighbours (0 where the
// neighbour is not a corner); the response is the score, or 0 without suppression.  Keypoints come out row by row,
// left to right.
#include <limits.h>

#include "stages.cuh"

namespace {

constexpr int FT_BX = 32, FT_BY = 8;                     // pixels per CTA of the score pass
constexpr int FT_TW = FT_BX + 6, FT_TH = FT_BY + 6;      // tile with the radius-3 halo

// circle offsets (dx, dy) in OpenCV's order (makeOffsets, patternSize 16)
__constant__ int8_t c_circle[16][2] = {{0, 3},  {1, 3},   {2, 2},   {3, 1},   {3, 0},  {3, -1}, {2, -2}, {1, -3},
                                       {0, -3}, {-1, -3}, {-2, -2}, {-3, -1}, {-3, 0}, {-3, 1}, {-2, 2}, {-1, 3}};

// 9 contiguous set bits in a circular 16-bit mask
__device__ __forceinline__ bool arc9(unsigned m) {
    const unsigned mm = m | (m << 16);
    unsigned r = mm & (mm >> 1);          // runs of 2
    r &= r >> 2;                          // 4
    r &= r >> 4;                          // 8
    r &= mm >> 8;                         // 9
    return (r & 0xFFFFu) != 0;
}

// cornerScore<16> (fast_score.cpp): d[k] = v - p[k];
//   a0 = max(threshold, max over the 16 arcs of 9 of min d);  b0 = min(-a0, min over the arcs of max d);  -b0 - 1
__device__ __forceinline__ int corner_score(const int (&d)[16], int threshold) {
    int lo2[16], hi2[16], lo4[16], hi4[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) { lo2[i] = min(d[i], d[(i + 1) & 15]); hi2[i] = max(d[i], d[(i + 1) & 15]); }
#pragma unroll
    for (int i = 0; i < 16; ++i) { lo4[i] = min(lo2[i], lo2[(i + 2) & 15]); hi4[i] = max(hi2[i], hi2[(i + 2) & 15]); }
    int a0 = threshold;
#pragma unroll
    for (int i = 0; i < 16; ++i) a0 = max(a0, min(min(lo4[i], lo4[(i + 4) & 15]), d[(i + 8) & 15]));
    int b0 = -a0;
#pragma unroll
    for (int i = 0; i < 16; ++i) b0 = min(b0, max(max(hi4[i], hi4[(i + 4) & 15]), d[(i + 8) & 15]));
    return -b0 - 1;
}

// score pass: S[img][y][x] = 0x100 | score for corners, 0 elsewhere
__global__ void __launch_bounds__(FT_BX * FT_BY) fast_score_kernel(const uint8_t* __restrict__ img, int rows, int cols,
                                                                   int threshold, int want_score, uint16_t* __restrict__ S) {
    __shared__ uint8_t tile[FT_TH][FT_TW + 2];
    const int x0 = blockIdx.x * FT_BX, y0 = blockIdx.y * FT_BY;
    const uint8_t* im = img + (size_t)blockIdx.z * rows * cols;
    uint16_t* s = S + (size_t)blockIdx.z * rows * cols;
    const int tid = threadIdx.y * FT_BX + threadIdx.x;
    for (int i = tid; i < FT_TH * FT_TW; i += FT_BX * FT_BY) {
        const int ty = i / FT_TW, tx = i % FT_TW;
        const int gx = min(max(x0 + tx - 3, 0), cols - 1), gy = min(max(y0 + ty - 3, 0), rows - 1);
        tile[ty][tx] = im[(size_t)gy * cols + gx];
    }
    __syncthreads();
    const int x = x0 + threadIdx.x, y = y0 + threadIdx.y;
    if (x >= cols || y >= rows) return;
    uint16_t out = 0;
    if (x >= 3 && x < cols - 3 && y >= 3 && y < rows - 3) {
        const int cx = threadIdx.x + 3, cy = threadIdx.y + 3;
        const int v = tile[cy][cx];
        int d[16];
        unsigned dark = 0, bright = 0;
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const int p = tile[cy + c_circle[k][1]][cx + c_circle[k][0]];
            d[k] = v - p;
            dark |= (d[k] > threshold ? 1u : 0u) << k;        // p < v - t
            bright |= (-d[k] > threshold ? 1u : 0u) << k;     // p > v + t
        }
        if (arc9(dark) || arc9(bright)) out = (uint16_t)(0x100 | (want_score ? corner_score(d, threshold) : 0));
    }
    s[(size_t)y * cols + x] = out;
}

__device__ __forceinline__ bool fast_keep(const uint16_t* __restrict__ s, int rows, int cols, int x, int y, int nonmax) {
    const int c = s[(size_t)y * cols + x];
    if (!(c & 0x100)) return false;
    if (!nonmax) return true;
    const int sc = c & 0xFF;
    // corners exist only for 3 <= x < cols-3, 3 <= y < rows-3: the 8 neighbours are inside the image
    const uint16_t* r0 = s + (size_t)(y - 1) * cols + x;
    const uint16_t* r1 = s + (size_t)y * cols + x;
    const uint16_t* r2 = s + (size_t)(y + 1) * cols + x;
    return sc > (r0[-1] & 0xFF) && sc > (r0[0] & 0xFF) && sc > (r0[1] & 0xFF) && sc > (r1[-1] & 0xFF) &&
           sc > (r1[1] & 0xFF) && sc > (r2[-1] & 0xFF) && sc > (r2[0] & 0xFF) && sc > (r2[1] & 0xFF);
}

// A row is cut into segments of FT_SEG pixels so that a single frame still fills the GPU with warps (one warp per
// segment: 8 steps of 32 pixels instead of a whole 1241-pixel row); counts / offsets are per (row, segment), in row-major
// order, which is OpenCV's keypoint order.
constexpr int FT_SEG = 256;

// one warp per (row segment, image): number of kept corners in the segment
__global__ void __launch_bounds__(128) fast_count_kernel(const uint16_t* __restrict__ S, int rows, int cols, int nseg, int nonmax,
                                                         int32_t* __restrict__ segcount) {
    const int item = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (item >= rows * nseg) return;
    const int row = item / nseg, x_lo = (item % nseg) * FT_SEG, x_hi = min(x_lo + FT_SEG, cols);
    const uint16_t* s = S + (size_t)blockIdx.y * rows * cols;
    int n = 0;
    if (row >= 3 && row < rows - 3)
        for (int x = x_lo + lane; x < x_hi; x += 32) n += fast_keep(s, rows, cols, x, row, nonmax) ? 1 : 0;
    n = __reduce_add_sync(0xFFFFFFFFu, n);
    if (lane == 0) segcount[(size_t)blockIdx.y * rows * nseg + item] = n;
}

// one CTA per image: exclusive scan of the row counts in place, total to counts[img]
__global__ void __launch_bounds__(256) fast_scan_kernel(int32_t* __restrict__ rowcount, int rows, int32_t* __restrict__ counts) {
    __shared__ int s_warp[8];
    __shared__ int s_carry;
    int32_t* rc = rowcount + (size_t)blockIdx.x * rows;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < rows; base += 256) {
        const int i = base + tid;
        const int v = i < rows ? rc[i] : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        int off = s_carry;
        for (int w = 0; w < warp; ++w) off += s_warp[w];
        if (i < rows) rc[i] = off + incl - v;
        __syncthreads();
        if (tid == 255) s_carry = off + incl;
        __syncthreads();
    }
    if (tid == 0) counts[blockIdx.x] = s_carry;
}

// one warp per (row segment, image): write the kept corners of the segment, left to right, at the segment's offset
__global__ void __launch_bounds__(128) fast_write_kernel(const uint16_t* __restrict__ S, int rows, int cols, int nseg, int nonmax,
                                                         const int32_t* __restrict__ segoff, int max_kp,
                                                         float* __restrict__ kps, float* __restrict__ resp) {
    const int item = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (item >= rows * nseg) return;
    const int row = item / nseg, x_lo = (item % nseg) * FT_SEG, x_hi = min(x_lo + FT_SEG, cols);
    if (row < 3 || row >= rows - 3) return;
    const uint16_t* s = S + (size_t)blockIdx.y * rows * cols;
    int pos = segoff[(size_t)blockIdx.y * rows * nseg + item];
    float* kp = kps + (size_t)blockIdx.y * max_kp * 2;
    float* rs = resp ? resp + (size_t)blockIdx.y * max_kp : nullptr;
    for (int x0 = x_lo; x0 < x_hi; x0 += 32) {
        const int x = x0 + lane;
        const bool keep = x < x_hi && fast_keep(s, rows, cols, x, row, nonmax);
        const unsigned bal = __ballot_sync(0xFFFFFFFFu, keep);
        if (keep) {
            const int k = pos + __popc(bal & ((1u << lane) - 1));
            if (k < max_kp) {
                kp[2 * k] = (float)x;
                kp[2 * k + 1] = (float)row;
                if (rs) rs[k] = nonmax ? (float)(s[(size_t)row * cols + x] & 0xFF) : 0.0f;
            }
        }
        pos += __popc(bal);
    }
}

}  // namespace

static inline int fast_nseg(int cols) { return (cols + FT_SEG - 1) / FT_SEG; }

size_t epv_fast_work_bytes(int n_images, int rows, int cols) {
    return (size_t)n_images * rows * cols * 2 + (size_t)n_images * rows * fast_nseg(cols) * 4 + 256;
}

// d_img: [n_images][rows][cols] bytes; d_kps: [n_images][max_kp][2]; d_resp: optional [n_images][max_kp];
// d_counts: [n_images] (the number FOUND, which may exceed max_kp: only the first max_kp are stored)
int epv_fast_launch(epivo_ctx* ctx, const uint8_t* d_img, int n_images, int rows, int cols, int threshold, int nonmax,
                    int max_kp, float* d_kps, float* d_resp, int32_t* d_counts, void* work) {
    if (n_images <= 0) return EPIVO_OK;
    uint16_t* S = (uint16_t*)work;
    int32_t* segcount = (int32_t*)((uint8_t*)work + (((size_t)n_images * rows * cols * 2 + 127) & ~(size_t)127));
    if (n_images > 65535) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "more than 65535 images per call");
    const int nseg = fast_nseg(cols), items = rows * nseg;
    const dim3 g((cols + FT_BX - 1) / FT_BX, (rows + FT_BY - 1) / FT_BY, n_images);
    fast_score_kernel<<<g, dim3(FT_BX, FT_BY), 0, ctx->stream>>>(d_img, rows, cols, threshold, nonmax, S);
    EPV_LAUNCHED(ctx);
    const dim3 gr((items + 3) / 4, n_images);
    fast_count_kernel<<<gr, 128, 0, ctx->stream>>>(S, rows, cols, nseg, nonmax, segcount);
    EPV_LAUNCHED(ctx);
    fast_scan_kernel<<<n_images, 256, 0, ctx->stream>>>(segcount, items, d_counts);
    EPV_LAUNCHED(ctx);
    fast_write_kernel<<<gr, 128, 0, ctx->stream>>>(S, rows, cols, nseg, nonmax, segcount, max_kp, d_kps, d_resp);
    EPV_LAUNCHED(ctx);
    return EPIVO_OK;
}

// =================================================================================================================
// N4 front end, tracker part: cv::calcOpticalFlowPyrLK with the defaults the reference uses
//     calcOpticalFlowPyrLK(src, tgt, pt0, pt1_, status, err);     kitti_E.cpp:79-84, kitti_ba.cpp:203-208,281-286
// (winSize 21 x 21, maxLevel 3, criteria COUNT+EPS (30, 0.01), flags 0, minEigThreshold 1e-4), OpenCV
// video/src/lkpyramid.cpp restated: buildOpticalFlowPyramid (pyrDown, BORDER_REFLECT_101), calcSharrDeriv, and
// LKTrackerInvoker level by level.  The integer parts -- pyramid, Scharr derivatives, the 14-bit fixed-point
// bilinear windows -- are exact; the 2 x 2 normal equations are summed in exact integers and rounded once to float
// (OpenCV accumulates them in float32 lanes; the sums of these integer products are almost always exactly
// representable, so the two agree bit for bit on most points and to ~1e-4 px otherwise); everything after that is
// OpenCV's float32 arithmetic spelled with round-to-nearest intrinsics (no FMA contraction).
namespace {

constexpr int LK_WIN = 21, LK_AREA = LK_WIN * LK_WIN, LK_PPL = (LK_AREA + 31) / 32;   // 14 window pixels per lane
constexpr int LK_MAX_LEVELS = 8;

struct LkGeom {
    int levels;                         // pyramid levels actually built (maxLevel + 1 or fewer)
    int rows[LK_MAX_LEVELS], cols[LK_MAX_LEVELS];
    int64_t off[LK_MAX_LEVELS];         // element offset of each level inside a frame's pyramid
    int64_t frame_stride;               // elements per frame pyramid
};

__device__ __forceinline__ int reflect101(int i, int n) {
    i = abs(i);
    return i >= n ? 2 * (n - 1) - i : i;
}

// cv::pyrDown, 8-bit: [1 4 6 4 1] x [1 4 6 4 1], BORDER_REFLECT_101, (sum + 128) >> 8; one thread per output pixel
__global__ void __launch_bounds__(256) pyr_down_kernel(uint8_t* __restrict__ pyr, LkGeom g, int level) {
    const int rows = g.rows[level - 1], cols = g.cols[level - 1], orow = g.rows[level], ocol = g.cols[level];
    const uint8_t* src = pyr + (size_t)blockIdx.y * g.frame_stride + g.off[level - 1];
    uint8_t* dst = pyr + (size_t)blockIdx.y * g.frame_stride + g.off[level];
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= orow * ocol) return;
    const int oy = i / ocol, ox = i % ocol;
    const int w[5] = {1, 4, 6, 4, 1};
    int sum = 0;
#pragma unroll
    for (int dy = 0; dy < 5; ++dy) {
        const uint8_t* r = src + (size_t)reflect101(2 * oy + dy - 2, rows) * cols;
        int h = 0;
#pragma unroll
        for (int dx = 0; dx < 5; ++dx) h += w[dx] * r[reflect101(2 * ox + dx - 2, cols)];
        sum += w[dy] * h;
    }
    dst[i] = (uint8_t)((sum + 128) >> 8);
}

// calcSharrDeriv: (dI/dx, dI/dy) as short2, 3-10-3 Scharr, BORDER_REFLECT_101; one thread per pixel
__global__ void __launch_bounds__(256) scharr_kernel(const uint8_t* __restrict__ pyr, short2* __restrict__ dpyr, LkGeom g,
                                                     int level) {
    const int rows = g.rows[level], cols = g.cols[level];
    const uint8_t* src = pyr + (size_t)blockIdx.y * g.frame_stride + g.off[level];
    short2* dst = dpyr + (size_t)blockIdx.y * g.frame_stride + g.off[level];
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= rows * cols) return;
    const int y = i / cols, x = i % cols;
    const uint8_t* r0 = src + (size_t)reflect101(y - 1, rows) * cols;
    const uint8_t* r1 = src + (size_t)y * cols;
    const uint8_t* r2 = src + (size_t)reflect101(y + 1, rows) * cols;
    const int xm = reflect101(x - 1, cols), xp = reflect101(x + 1, cols);
    const int t0m = (r0[xm] + r2[xm]) * 3 + r1[xm] * 10, t0p = (r0[xp] + r2[xp]) * 3 + r1[xp] * 10;
    const int t1m = r2[xm] - r0[xm], t1c = r2[x] - r0[x], t1p = r2[xp] - r0[xp];
    dst[i] = make_short2((short)(t0p - t0m), (short)((t1p + t1m) * 3 + t1c * 10));
}

// warp total of per-lane 32-bit partial sums (the total needs up to 37 bits): two REDUX on the halves instead of a
// five-step 64-bit shuffle chain -- the reduction sits on the dependent path of every LK iteration
__device__ __forceinline__ long long warp_sum_i32(int v) {
    const int hi = __reduce_add_sync(0xFFFFFFFFu, v >> 16);              // |v >> 16| <= 2^15 per lane
    const int lo = __reduce_add_sync(0xFFFFFFFFu, v & 0xFFFF);           // < 2^16 per lane
    return ((long long)hi << 16) + lo;
}

// cvFloor as the x86 build OpenCV ships: NaN and values beyond the int range convert to INT_MIN, which the range tests
// then reject (CUDA's conversion would give 0 for NaN and let the point through)
__device__ __forceinline__ int lk_floor(float v) {
    return (v == v && fabsf(v) < 2147483520.f) ? (int)floorf(v) : INT_MIN;
}
__device__ __forceinline__ void lk_weights(float a, float b, int& w00, int& w01, int& w10, int& w11) {
    const float s = 16384.0f;                                                   // 1 << W_BITS
    w00 = __float2int_rn(__fmul_rn(__fmul_rn(__fsub_rn(1.f, a), __fsub_rn(1.f, b)), s));   // cvRound: half to even
    w01 = __float2int_rn(__fmul_rn(__fmul_rn(a, __fsub_rn(1.f, b)), s));
    w10 = __float2int_rn(__fmul_rn(__fmul_rn(__fsub_rn(1.f, a), b), s));
    w11 = 16384 - w00 - w01 - w10;
}

// The 21 x 21 window is cut into 63 row segments of 7 pixels (3 per row); a lane owns segments `lane` and `lane + 32`.
// The bilinear samples of a segment share their source pixels -- 2 x 8 loads for 7 samples instead of 4 per sample --
// and the row / column border arithmetic is done once per segment.
constexpr int LK_SEG = 7, LK_NSEG = LK_AREA / LK_SEG;        // 63

template <bool INTERIOR>
__device__ __forceinline__ void lk_row8(const uint8_t* __restrict__ img, int rows, int cols, int y, int x0, int (&v)[8]) {
    if (INTERIOR) {
        const uint8_t* r = img + (size_t)y * cols + x0;
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = r[i];
    } else {                                                 // the pyramid's border: BORDER_REFLECT_101
        const uint8_t* r = img + (size_t)reflect101(y, rows) * cols;
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = r[reflect101(x0 + i, cols)];
    }
}
template <bool INTERIOR>
__device__ __forceinline__ void lk_drow8(const short2* __restrict__ d, int rows, int cols, int y, int x0, short2 (&v)[8]) {
    if (INTERIOR) {
        const short2* r = d + (size_t)y * cols + x0;
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = r[i];
    } else {                                                 // the derivative's border: BORDER_CONSTANT 0
        const bool yin = y >= 0 && y < rows;
        const short2* r = d + (size_t)(yin ? y : 0) * cols;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int x = x0 + i;
            v[i] = (yin && x >= 0 && x < cols) ? r[x] : make_short2(0, 0);
        }
    }
}
// window of the previous image: I and its derivatives for one segment, and the segment's part of the 2 x 2 system
template <bool INTERIOR, int BASE>
__device__ __forceinline__ void lk_patch_seg(const uint8_t* __restrict__ I, const short2* __restrict__ dI, int rows, int cols,
                                             int y, int x0, int w00, int w01, int w10, int w11, short (&Iw)[2 * LK_SEG],
                                             short (&Ix)[2 * LK_SEG], short (&Iy)[2 * LK_SEG], int& s11, int& s12, int& s22) {
    int a[8], b[8];
    short2 da[8], db[8];
    lk_row8<INTERIOR>(I, rows, cols, y, x0, a);
    lk_row8<INTERIOR>(I, rows, cols, y + 1, x0, b);
    lk_drow8<INTERIOR>(dI, rows, cols, y, x0, da);
    lk_drow8<INTERIOR>(dI, rows, cols, y + 1, x0, db);
#pragma unroll
    for (int i = 0; i < LK_SEG; ++i) {
        const int iv = a[i] * w00 + a[i + 1] * w01 + b[i] * w10 + b[i + 1] * w11;
        const int ixv = (da[i].x * w00 + da[i + 1].x * w01 + db[i].x * w10 + db[i + 1].x * w11 + (1 << 13)) >> 14;
        const int iyv = (da[i].y * w00 + da[i + 1].y * w01 + db[i].y * w10 + db[i + 1].y * w11 + (1 << 13)) >> 14;
        Iw[BASE + i] = (short)((iv + (1 << 8)) >> 9);                         // CV_DESCALE(., W_BITS1 - 5)
        Ix[BASE + i] = (short)ixv;
        Iy[BASE + i] = (short)iyv;
        s11 += ixv * ixv;
        s12 += ixv * iyv;
        s22 += iyv * iyv;
    }
}
// window of the next image at the current position against the stored one: the segment's part of the right-hand side
// (SAD = false) or of the absolute difference (SAD = true, the `err` pass)
template <bool INTERIOR, int BASE, bool SAD>
__device__ __forceinline__ void lk_diff_seg(const uint8_t* __restrict__ J, int rows, int cols, int y, int x0, int w00, int w01,
                                            int w10, int w11, const short (&Iw)[2 * LK_SEG], const short (&Ix)[2 * LK_SEG],
                                            const short (&Iy)[2 * LK_SEG], int& s1, int& s2) {
    int a[8], b[8];
    lk_row8<INTERIOR>(J, rows, cols, y, x0, a);
    lk_row8<INTERIOR>(J, rows, cols, y + 1, x0, b);
#pragma unroll
    for (int i = 0; i < LK_SEG; ++i) {
        const int jv = a[i] * w00 + a[i + 1] * w01 + b[i] * w10 + b[i + 1] * w11;
        const int diff = ((jv + (1 << 8)) >> 9) - Iw[BASE + i];
        if (SAD) {
            s1 += abs(diff);
        } else {
            s1 += diff * Ix[BASE + i];
            s2 += diff * Iy[BASE + i];
        }
    }
}

// one warp per point: all pyramid levels, all iterations
constexpr int LK_MINBLOCKS = 5;
__global__ void __launch_bounds__(128, LK_MINBLOCKS) lk_kernel(const uint8_t* __restrict__ pyr, const short2* __restrict__ dpyr, LkGeom g,
                                                 const float* __restrict__ pts, const int32_t* __restrict__ counts,
                                                 int max_pts, int max_count, double eps2, float min_eig,
                                                 float* __restrict__ next_pts, uint8_t* __restrict__ status,
                                                 float* __restrict__ err, const int32_t* __restrict__ pair_frames) {
    const int pair = blockIdx.y, lane = threadIdx.x & 31;
    const int p = blockIdx.x * 4 + (threadIdx.x >> 5);
    // pair i tracks frame i into frame i + 1 with the points and count of slot i; with pair_frames (gridDim.y pairs:
    // previous frames, then next frames) it tracks the points of frame fi -- slot fi of pts / counts -- into frame fj
    const int fi = pair_frames ? pair_frames[pair] : pair;
    const int fj = pair_frames ? pair_frames[gridDim.y + pair] : pair + 1;
    if (p >= min(counts[fi], max_pts)) return;
    const float px = pts[((size_t)fi * max_pts + p) * 2], py = pts[((size_t)fi * max_pts + p) * 2 + 1];
    const float half = (LK_WIN - 1) * 0.5f;
    const float FLT_SCALE = 1.f / (1 << 20);
    float nx = 0.f, ny = 0.f;            // nextPts[ptidx]
    bool ok = true;
    short Iw[2 * LK_SEG], Ix[2 * LK_SEG], Iy[2 * LK_SEG];
    const int wyA = lane / 3, wxA = LK_SEG * (lane - 3 * wyA);                     // segment `lane`: window row, first column
    const bool segB = lane + 32 < LK_NSEG;                                         // segment `lane + 32` (lane 31 has none)
    const int wyB = (lane + 32) / 3, wxB = LK_SEG * (lane + 32 - 3 * wyB);
    for (int level = g.levels - 1; level >= 0; --level) {
        const int rows = g.rows[level], cols = g.cols[level];
        const uint8_t* I = pyr + (size_t)fi * g.frame_stride + g.off[level];
        const uint8_t* J = pyr + (size_t)fj * g.frame_stride + g.off[level];
        const short2* dI = dpyr + (size_t)fi * g.frame_stride + g.off[level];
        const float sc = 1.f / (float)(1 << level);
        float ppx = __fmul_rn(px, sc), ppy = __fmul_rn(py, sc);
        if (level == g.levels - 1) { nx = ppx; ny = ppy; } else { nx = __fmul_rn(nx, 2.f); ny = __fmul_rn(ny, 2.f); }
        ppx = __fsub_rn(ppx, half);
        ppy = __fsub_rn(ppy, half);
        const int ipx = lk_floor(ppx), ipy = lk_floor(ppy);
        if (ipx < -LK_WIN || ipx >= cols || ipy < -LK_WIN || ipy >= rows) {
            if (level == 0) ok = false;
            continue;
        }
        int w00, w01, w10, w11;
        lk_weights(__fsub_rn(ppx, (float)ipx), __fsub_rn(ppy, (float)ipy), w00, w01, w10, w11);
        int s11 = 0, s12 = 0, s22 = 0;                      // per lane: 14 x 4080^2 < 2^31
        if (ipx >= 0 && ipy >= 0 && ipx + LK_WIN < cols && ipy + LK_WIN < rows) {       // whole footprint inside: warp-uniform
            lk_patch_seg<true, 0>(I, dI, rows, cols, ipy + wyA, ipx + wxA, w00, w01, w10, w11, Iw, Ix, Iy, s11, s12, s22);
            if (segB) lk_patch_seg<true, LK_SEG>(I, dI, rows, cols, ipy + wyB, ipx + wxB, w00, w01, w10, w11, Iw, Ix, Iy, s11, s12, s22);
        } else {
            lk_patch_seg<false, 0>(I, dI, rows, cols, ipy + wyA, ipx + wxA, w00, w01, w10, w11, Iw, Ix, Iy, s11, s12, s22);
            if (segB) lk_patch_seg<false, LK_SEG>(I, dI, rows, cols, ipy + wyB, ipx + wxB, w00, w01, w10, w11, Iw, Ix, Iy, s11, s12, s22);
        }
        const float A11 = __fmul_rn(__ll2float_rn(warp_sum_i32(s11)), FLT_SCALE),
                    A12 = __fmul_rn(__ll2float_rn(warp_sum_i32(s12)), FLT_SCALE),
                    A22 = __fmul_rn(__ll2float_rn(warp_sum_i32(s22)), FLT_SCALE);
        float D = __fsub_rn(__fmul_rn(A11, A22), __fmul_rn(A12, A12));
        const float dA = __fsub_rn(A11, A22);
        const float root = __fsqrt_rn(__fadd_rn(__fmul_rn(dA, dA), __fmul_rn(__fmul_rn(4.f, A12), A12)));
        const float minEig = __fdiv_rn(__fsub_rn(__fadd_rn(A22, A11), root), (float)(2 * LK_WIN * LK_WIN));
        if (minEig < min_eig || D < 1.1920929e-07f) {                        // FLT_EPSILON
            if (level == 0) ok = false;
            continue;
        }
        D = __fdiv_rn(1.f, D);
        float tx = __fsub_rn(nx, half), ty = __fsub_rn(ny, half);             // nextPt -= halfWin
        float pdx = 0.f, pdy = 0.f;
        for (int j = 0; j < max_count; ++j) {
            const int inx = lk_floor(tx), iny = lk_floor(ty);
            if (inx < -LK_WIN || inx >= cols || iny < -LK_WIN || iny >= rows) {
                if (level == 0) ok = false;
                break;
            }
            lk_weights(__fsub_rn(tx, (float)inx), __fsub_rn(ty, (float)iny), w00, w01, w10, w11);
            // per lane |diff * I'| <= 8160 * 4080 over 14 pixels fits 32 bits; the warp total needs 64
            int s1 = 0, s2 = 0;
            if (inx >= 0 && iny >= 0 && inx + LK_WIN < cols && iny + LK_WIN < rows) {
                // the whole 22 x 22 footprint lies inside the image (the common case, warp-uniform): no border arithmetic
                lk_diff_seg<true, 0, false>(J, rows, cols, iny + wyA, inx + wxA, w00, w01, w10, w11, Iw, Ix, Iy, s1, s2);
                if (segB) lk_diff_seg<true, LK_SEG, false>(J, rows, cols, iny + wyB, inx + wxB, w00, w01, w10, w11, Iw, Ix, Iy, s1, s2);
            } else {
                lk_diff_seg<false, 0, false>(J, rows, cols, iny + wyA, inx + wxA, w00, w01, w10, w11, Iw, Ix, Iy, s1, s2);
                if (segB) lk_diff_seg<false, LK_SEG, false>(J, rows, cols, iny + wyB, inx + wxB, w00, w01, w10, w11, Iw, Ix, Iy, s1, s2);
            }
            const long long b1 = warp_sum_i32(s1), b2 = warp_sum_i32(s2);
            const float fb1 = __fmul_rn(__ll2float_rn(b1), FLT_SCALE), fb2 = __fmul_rn(__ll2float_rn(b2), FLT_SCALE);
            const float dx = __fmul_rn(__fsub_rn(__fmul_rn(A12, fb2), __fmul_rn(A22, fb1)), D);
            const float dy = __fmul_rn(__fsub_rn(__fmul_rn(A12, fb1), __fmul_rn(A11, fb2)), D);
            tx = __fadd_rn(tx, dx);
            ty = __fadd_rn(ty, dy);
            nx = __fadd_rn(tx, half);
            ny = __fadd_rn(ty, half);
            if (__dadd_rn(__dmul_rn((double)dx, (double)dx), __dmul_rn((double)dy, (double)dy)) <= eps2) break;
            if (j > 0 && fabs((double)__fadd_rn(dx, pdx)) < 0.01 && fabs((double)__fadd_rn(dy, pdy)) < 0.01) {
                nx = __fsub_rn(nx, __fmul_rn(dx, 0.5f));
                ny = __fsub_rn(ny, __fmul_rn(dy, 0.5f));
                break;
            }
            pdx = dx;
            pdy = dy;
        }
        if (level == 0 && ok && err != nullptr) {
            // lkpyramid.cpp, after the iterations, when the caller passes `err` (every reference call site does): the
            // mean absolute window difference at the FINAL position -- which the loop did not range-check after its
            // last update: outside [-win, size) the status is cleared
            const float ex = __fsub_rn(nx, half), ey = __fsub_rn(ny, half);
            const int iex = lk_floor(ex), iey = lk_floor(ey);
            if (iex < -LK_WIN || iex >= cols || iey < -LK_WIN || iey >= rows) {
                ok = false;
            } else {
                lk_weights(__fsub_rn(ex, (float)iex), __fsub_rn(ey, (float)iey), w00, w01, w10, w11);
                int sad = 0, unused = 0;
                lk_diff_seg<false, 0, true>(J, rows, cols, iey + wyA, iex + wxA, w00, w01, w10, w11, Iw, Ix, Iy, sad, unused);
                if (segB) lk_diff_seg<false, LK_SEG, true>(J, rows, cols, iey + wyB, iex + wxB, w00, w01, w10, w11, Iw, Ix, Iy, sad, unused);
                sad = __reduce_add_sync(0xFFFFFFFFu, sad);          // < 2^24: the float sum OpenCV forms is exact, in any order
                if (lane == 0) err[(size_t)pair * max_pts + p] = __fdiv_rn((float)sad, (float)(32 * LK_AREA));
            }
        }
    }
    if (lane == 0) {
        next_pts[((size_t)pair * max_pts + p) * 2] = nx;
        next_pts[((size_t)pair * max_pts + p) * 2 + 1] = ny;
        status[(size_t)pair * max_pts + p] = ok ? 1 : 0;
    }
}

LkGeom lk_geometry(int rows, int cols, int max_level) {
    LkGeom g{};
    int64_t off = 0;
    int r = rows, c = cols;
    for (int l = 0; l <= max_level && l < LK_MAX_LEVELS; ++l) {
        if (l > 0) {                                     // buildOpticalFlowPyramid: stop when a side would not exceed the window
            const int nr = (r + 1) / 2, nc = (c + 1) / 2;
            if (nc <= LK_WIN || nr <= LK_WIN) break;
            r = nr;
            c = nc;
        }
        g.rows[l] = r;
        g.cols[l] = c;
        g.off[l] = off;
        off += ((int64_t)r * c + 63) & ~(int64_t)63;
        g.levels = l + 1;
    }
    g.frame_stride = off;
    return g;
}

}  // namespace

// bytes of device scratch for n_frames frames: 8-bit pyramids + short2 derivative pyramids
size_t epv_lk_work_bytes(int n_frames, int rows, int cols, int max_level) {
    const LkGeom g = lk_geometry(rows, cols, max_level);
    return (size_t)n_frames * g.frame_stride * (1 + 4) + 1024;
}

// d_images: [n_frames][rows][cols] -> the pyramids of every frame in `work`, and the derivative pyramids of frames
// [0, n_deriv) (the frames that are the previous image of some pair)
int epv_lk_pyramids(epivo_ctx* ctx, const uint8_t* d_images, int n_frames, int rows, int cols, int max_level, int n_deriv,
                    void* work) {
    if (rows <= LK_WIN || cols <= LK_WIN)
        EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "image %d x %d not larger than the %d x %d window", cols, rows, LK_WIN, LK_WIN);
    if (n_frames > 65535) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "more than 65535 frames per call");
    const LkGeom g = lk_geometry(rows, cols, max_level);
    uint8_t* pyr = (uint8_t*)work;
    short2* dpyr = (short2*)(pyr + (((size_t)n_frames * g.frame_stride + 255) & ~(size_t)255));
    // level 0 = the frames themselves (one strided copy), then level by level
    EPV_CUDA(ctx, cudaMemcpy2DAsync(pyr, (size_t)g.frame_stride, d_images, (size_t)rows * cols, (size_t)rows * cols, n_frames,
                                    cudaMemcpyDeviceToDevice, ctx->stream));
    for (int l = 1; l < g.levels; ++l) {
        const int n = g.rows[l] * g.cols[l];
        pyr_down_kernel<<<dim3((n + 255) / 256, n_frames), 256, 0, ctx->stream>>>(pyr, g, l);
        EPV_LAUNCHED(ctx);
    }
    for (int l = 0; l < g.levels && n_deriv > 0; ++l) {
        const int n = g.rows[l] * g.cols[l];
        scharr_kernel<<<dim3((n + 255) / 256, n_deriv), 256, 0, ctx->stream>>>(pyr, dpyr, g, l);
        EPV_LAUNCHED(ctx);
    }
    return EPIVO_OK;
}

// LK over the pyramids epv_lk_pyramids left in `work` (built for n_frames frames): pair i < n_pairs tracks
// d_pts[i][0..min(d_counts[i], max_pts)) from frame i into frame i + 1, or, with d_pair_frames (2 x n_pairs: previous
// frames, then next frames), d_pts[fi][..d_counts[fi]) from frame fi = d_pair_frames[i] into d_pair_frames[n_pairs + i].
// Outputs are [n_pairs][max_pts].
int epv_lk_track_launch(epivo_ctx* ctx, const void* work, int n_frames, int rows, int cols, int max_level, int n_pairs,
                        const int32_t* d_pair_frames, const float* d_pts, const int32_t* d_counts, int max_pts, int max_count,
                        double epsilon, double min_eig, float* d_next, uint8_t* d_status, float* d_err) {
    if (n_pairs <= 0 || max_pts <= 0) return EPIVO_OK;
    if (n_pairs > 65535) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "more than 65535 pairs per call");
    const LkGeom g = lk_geometry(rows, cols, max_level);
    const uint8_t* pyr = (const uint8_t*)work;
    const short2* dpyr = (const short2*)(pyr + (((size_t)n_frames * g.frame_stride + 255) & ~(size_t)255));
    lk_kernel<<<dim3((max_pts + 3) / 4, n_pairs), 128, 0, ctx->stream>>>(pyr, dpyr, g, d_pts, d_counts, max_pts, max_count,
                                                                       epsilon * epsilon, (float)min_eig, d_next, d_status,
                                                                       d_err, d_pair_frames);
    EPV_LAUNCHED(ctx);
    return EPIVO_OK;
}

// d_images: [n_frames][rows][cols]; pair i tracks d_pts[i][0..counts[i]) from frame i into frame i + 1
int epv_lk_launch(epivo_ctx* ctx, const uint8_t* d_images, int n_frames, int rows, int cols, const float* d_pts,
                  const int32_t* d_counts, int max_pts, int max_level, int max_count, double epsilon, double min_eig,
                  float* d_next, uint8_t* d_status, float* d_err, void* work) {
    if (n_frames < 2 || max_pts <= 0) return EPIVO_OK;
    // derivatives of the PREVIOUS image of every pair: frames 0 .. n-2
    int rc = epv_lk_pyramids(ctx, d_images, n_frames, rows, cols, max_level, n_frames - 1, work);
    if (rc) return rc;
    return epv_lk_track_launch(ctx, work, n_frames, rows, cols, max_level, n_frames - 1, nullptr, d_pts, d_counts, max_pts,
                               max_count, epsilon, min_eig, d_next, d_status, d_err);
}

// =================================================================================================================
// N4 front end, undistortion: cv::remap(src, dst, map1, map2, INTER_LINEAR) with the fixed-point maps that
// initUndistortRectifyMap hands the EuRoC driver (euroc_E.cpp:105-113 builds them once -- m1type 0 selects CV_16SC2 +
// CV_16UC1 --, :169-174 remaps every frame): map_xy holds the integer source position of every destination pixel,
// map_frac the 5 + 5 fraction bits.  OpenCV's bilinear table for fractions (fx, fy) / 32 is
// w = {(32-fx)(32-fy), fx(32-fy), (32-fx)fy, fx fy} * 32 (sum 2^15; its saturation of the single 32768 entry to 32767
// does not change any 8-bit result), the pixel is (sum w p + 2^14) >> 15, and with BORDER_CONSTANT a source pixel
// outside the image is the border value.  Integer work, one byte written per 6 bytes of map read: HBM-bound, bit-exact.
namespace {

__global__ void __launch_bounds__(256) remap_kernel(const uint8_t* __restrict__ img, int rows, int cols,
                                                    const short2* __restrict__ map_xy, const uint16_t* __restrict__ map_frac,
                                                    int drows, int dcols, int border, uint8_t* __restrict__ out) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= drows * dcols) return;
    const uint8_t* s = img + (size_t)blockIdx.y * rows * cols;
    const short2 xy = map_xy[i];
    const int f = map_frac[i] & 1023, fx = f & 31, fy = f >> 5;
    const int sx = xy.x, sy = xy.y;
    const int w00 = (32 - fx) * (32 - fy) * 32, w01 = fx * (32 - fy) * 32, w10 = (32 - fx) * fy * 32, w11 = fx * fy * 32;
    int v;
    if ((unsigned)sx < (unsigned)max(cols - 1, 0) && (unsigned)sy < (unsigned)max(rows - 1, 0)) {
        const uint8_t* p = s + (size_t)sy * cols + sx;
        v = p[0] * w00 + p[1] * w01 + p[cols] * w10 + p[cols + 1] * w11;
    } else if (sx >= cols || sx + 1 < 0 || sy >= rows || sy + 1 < 0) {
        out[(size_t)blockIdx.y * drows * dcols + i] = (uint8_t)border;
        return;
    } else {
        const bool x0 = sx >= 0 && sx < cols, x1 = sx + 1 >= 0 && sx + 1 < cols;
        const bool y0 = sy >= 0 && sy < rows, y1 = sy + 1 >= 0 && sy + 1 < rows;
        const int p00 = (x0 && y0) ? s[(size_t)sy * cols + sx] : border;
        const int p01 = (x1 && y0) ? s[(size_t)sy * cols + sx + 1] : border;
        const int p10 = (x0 && y1) ? s[(size_t)(sy + 1) * cols + sx] : border;
        const int p11 = (x1 && y1) ? s[(size_t)(sy + 1) * cols + sx + 1] : border;
        v = p00 * w00 + p01 * w01 + p10 * w10 + p11 * w11;
    }
    out[(size_t)blockIdx.y * drows * dcols + i] = (uint8_t)min(max((v + (1 << 14)) >> 15, 0), 255);
}

}  // namespace

// d_img: [n_images][rows][cols]; maps: [drows][dcols] (shared by all images); d_out: [n_images][drows][dcols]
int epv_remap_launch(epivo_ctx* ctx, const uint8_t* d_img, int n_images, int rows, int cols, const int16_t* d_map_xy,
                     const uint16_t* d_map_frac, int drows, int dcols, int border, uint8_t* d_out) {
    if (n_images <= 0 || drows <= 0 || dcols <= 0) return EPIVO_OK;
    if (n_images > 65535) EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "more than 65535 images per call");
    const int n = drows * dcols;
    remap_kernel<<<dim3((n + 255) / 256, n_images), 256, 0, ctx->stream>>>(d_img, rows, cols, (const short2*)d_map_xy, d_map_frac,
                                                                        drows, dcols, border, d_out);
    EPV_LAUNCHED(ctx);
    return EPIVO_OK;
}
