// E1/E2: cv::findEssentialMat(RANSAC | LMEDS) on the GPU, batched over frame pairs.
//
// Replaces kitti.cpp:98-104, kitti_E.cpp:98-104, euroc_E.cpp:202-208, kitti_ba.cpp:232,308,702.
// OpenCV's estimator (modules/calib3d/src/ptsetreg.cpp) is a sequential loop
//     sample 5 -> solve (<= 10 models) -> score every model -> keep strictly better -> shrink niters
// whose sample stream does not depend on the data (cv::RNG seeded with -1).  Those semantics are
// kept exactly, but the work is done in rounds (see "Rounds" below): the next R samples of every
// running pair are drawn from the same RNG stream and solved at full occupancy (fivept.cuh), then
// one CTA per pair scores the models (Sampson error in OpenCV's operation order, float32
// compare) and replays the sequential "strictly better / update niters" bookkeeping in sample
// order, stopping where the sequential loop would have stopped.  The result is the model the
// sequential loop returns.
#include <float.h>
#include <math.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "fivept.cuh"
#include "stages.cuh"

namespace {

constexpr int ES_THREADS = 256;
constexpr int ES_WARPS = ES_THREADS / 32;
constexpr int ES_SUB = 32;           // samples per scoring sub-chunk, at most (one lane of warp 0 per sample in the replay)

struct CvRng {   // cv::RNG: multiply-with-carry
    unsigned long long state;
    __device__ unsigned next() {
        state = (unsigned long long)(unsigned)state * 4164903690ULL + (unsigned)(state >> 32);
        return (unsigned)state;
    }
    __device__ int uniform(int a, int b) { return a == b ? a : (int)(next() % (unsigned)(b - a)) + a; }
};

// ptsetreg.cpp getSubset: 5 distinct indices, redraw on duplicates
__device__ __forceinline__ void draw_subset(CvRng& rng, int n, int* idx) {
    for (int i = 0; i < 5; ++i) {
        int v;
        bool dup;
        do {
            v = rng.uniform(0, n);
            dup = false;
            for (int k = 0; k < i; ++k) dup |= (idx[k] == v);
        } while (dup);
        idx[i] = v;
    }
}

// ptsetreg.cpp RANSACUpdateNumIters
__device__ int update_num_iters(double p, double ep, int model_points, int max_iters) {
    p = fmax(p, 0.0);
    p = fmin(p, 1.0);
    ep = fmax(ep, 0.0);
    ep = fmin(ep, 1.0);
    double num = fmax(1.0 - p, DBL_MIN);
    double denom;
    if (model_points == 5) {                   // the only call shape here; x^5 by multiplication instead of pow()
        const double x = 1.0 - ep, x2 = x * x;
        denom = 1.0 - x2 * x2 * x;
    } else {
        denom = 1.0 - pow(1.0 - ep, (double)model_points);
    }
    if (denom < DBL_MIN) return 0;
    num = log(num);
    denom = log(denom);
    return (denom >= 0 || -num >= max_iters * (-denom)) ? max_iters : (int)rint(num / denom);
}

// EMEstimatorCallback::computeError for one correspondence, OpenCV's operation order
// (Matx products accumulate left to right from 0; OpenCV's calib3d is built without FMA
// contraction, so every operation here is an explicit round-to-nearest intrinsic).
__device__ __forceinline__ float sampson_f32(const double* __restrict__ E, double a1, double b1, double a2,
                                             double b2) {
    // explicit round-to-nearest multiplies and adds: never contracted into FMAs
    const double ex0 = __dadd_rn(__dadd_rn(__dmul_rn(E[0], a1), __dmul_rn(E[1], b1)), E[2]);
    const double ex1 = __dadd_rn(__dadd_rn(__dmul_rn(E[3], a1), __dmul_rn(E[4], b1)), E[5]);
    const double ex2 = __dadd_rn(__dadd_rn(__dmul_rn(E[6], a1), __dmul_rn(E[7], b1)), E[8]);
    const double et0 = __dadd_rn(__dadd_rn(__dmul_rn(E[0], a2), __dmul_rn(E[3], b2)), E[6]);
    const double et1 = __dadd_rn(__dadd_rn(__dmul_rn(E[1], a2), __dmul_rn(E[4], b2)), E[7]);
    const double x2tEx1 = __dadd_rn(__dadd_rn(__dmul_rn(a2, ex0), __dmul_rn(b2, ex1)), ex2);
    const double den = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(ex0, ex0), __dmul_rn(ex1, ex1)), __dmul_rn(et0, et0)),
                                 __dmul_rn(et1, et1));
    return (float)__ddiv_rn(__dmul_rn(x2tEx1, x2tEx1), den);
}

// Inlier test  (float)(num/den) <= thr32  without the FP64 division.
// Let B be the largest double whose float rounding is <= thr32 (the midpoint between thr32 and the
// next float up, or its predecessor when the tie would round up).  Then
//     num/den <= B                =>  RN64(num/den) <= B        => inlier      (RN is monotone)
//     num/den >  B (1 + 2^-50)    =>  RN64(num/den) >  B        => outlier
// and the sign of B*den - num is exact in one FMA.  Only quotients within 2^-50 of B (or
// den == 0 / NaN) take the division; num and den are the same un-fused values OpenCV computes.
// high 32 bits of a double: for positive normal x, y:  hi(x) > hi(y)  =>  x > y,  and hi(y 2^e) = hi(y) + (e << 20)
__host__ __device__ inline int samp_hi(double x) {
#ifdef __CUDA_ARCH__
    return __double2hiint(x);
#else
    long long b;
    memcpy(&b, &x, 8);
    return (int)(b >> 32);
#endif
}

struct SampThr {
    double B, C;     // C = B * 2^-50
    double Blo, Bhi, dmin;   // pre-filter of sampson_inlier_unit: B (1 -+ 2e-6); smallest trusted denominator
    int eoff, hdmin;         // integer form of the pre-filter: see prefilter_decide()
    float thr32;
};
__host__ __device__ inline SampThr make_samp_thr(float thr32) {
    SampThr t;
    t.thr32 = thr32;
    unsigned bits;
#ifdef __CUDA_ARCH__
    bits = __float_as_uint(thr32);
    const float up = __uint_as_float(bits + 1u);
#else
    memcpy(&bits, &thr32, 4);
    const unsigned ub = bits + 1u;
    float up;
    memcpy(&up, &ub, 4);
#endif
    double mid = 0.5 * ((double)thr32 + (double)up);          // exact: two adjacent floats
    if ((bits & 1u) && mid > 0.0 && mid < 1e300) {            // odd mantissa: the tie rounds away from thr32
#ifdef __CUDA_ARCH__
        mid = __longlong_as_double(__double_as_longlong(mid) - 1);
#else
        long long mb;
        memcpy(&mb, &mid, 8);
        mb -= 1;
        memcpy(&mid, &mb, 8);
#endif
    }
    if (!(thr32 >= 0.0f) || !(thr32 < 3e38f)) mid = -1.0;     // negative / NaN / huge: always take the exact path
    t.B = mid;
    t.C = mid * 8.881784197001252e-16;                         // 2^-50
    t.Blo = mid * (1.0 - 2e-6);
    t.Bhi = mid * (1.0 + 2e-6);
    t.dmin = mid > 0.0 ? fmax(1e-8, 1e-13 / mid) : 1e300;     // invalid threshold: the pre-filter never decides
    // integer pre-filter: 2^e = the smallest power of two >= 2.1e-6 B, as an offset on the high word of a double
    {
        int e = 0;
        if (mid > 1e-200) {
            const double m = frexp(mid * 2.1e-6, &e);          // mid * 2.1e-6 = m 2^e, 0.5 <= m < 1  =>  2^e > B 2.1e-6
            (void)m;
        } else {
            t.dmin = 1e300;                                     // absurdly small threshold: exact path only
        }
        t.eoff = e * (1 << 20);
        t.hdmin = samp_hi(t.dmin);
    }
    return t;
}

__device__ __forceinline__ bool sampson_inlier(const double* __restrict__ E, double a1, double b1, double a2,
                                               double b2, const SampThr& T) {
    const double ex0 = __dadd_rn(__dadd_rn(__dmul_rn(E[0], a1), __dmul_rn(E[1], b1)), E[2]);
    const double ex1 = __dadd_rn(__dadd_rn(__dmul_rn(E[3], a1), __dmul_rn(E[4], b1)), E[5]);
    const double ex2 = __dadd_rn(__dadd_rn(__dmul_rn(E[6], a1), __dmul_rn(E[7], b1)), E[8]);
    const double et0 = __dadd_rn(__dadd_rn(__dmul_rn(E[0], a2), __dmul_rn(E[3], b2)), E[6]);
    const double et1 = __dadd_rn(__dadd_rn(__dmul_rn(E[1], a2), __dmul_rn(E[4], b2)), E[7]);
    const double x2tEx1 = __dadd_rn(__dadd_rn(__dmul_rn(a2, ex0), __dmul_rn(b2, ex1)), ex2);
    const double den = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(ex0, ex0), __dmul_rn(ex1, ex1)), __dmul_rn(et0, et0)),
                                 __dmul_rn(et1, et1));
    const double num = __dmul_rn(x2tEx1, x2tEx1);
    const double r = __fma_rn(T.B, den, -num);
    if (r >= 0.0 && den > 0.0 && T.B > 0.0) return true;
    if (-r > __dmul_rn(T.C, den) && T.B > 0.0) return false;
    return (float)__ddiv_rn(num, den) <= T.thr32;
}

// out-of-line copy for the pre-filter's fallback: a call keeps the compiler from predicating the
// 36-instruction exact path into the fast path (where it would be issued, masked off, every time)
__device__ __noinline__ bool sampson_inlier_slow(const double* E, double a1, double b1, double a2, double b2,
                                                 const SampThr& T) {
    return sampson_inlier(E, a1, b1, a2, b2, T);
}

// The same test for UNIT-NORM models (what the solver emits), with a fused pre-filter: the Sampson
// numerator and denominator are first evaluated with FMAs (22 instructions instead of 36).  With
// |E_ij| <= 1 and S1 = |a1|+|b1|+1, S2 = |a2|+|b2|+1 the fused s = x2'Ex1 is within eps_s = 12 u S1 S2
// of the exact value (u = 2^-53) and den within a relative 24 u S sqrt(2/den) + 4u.  A decision is
// taken from the fused values only if num lies outside [B (1 - 2e-6) den, B (1 + 2e-6) den] -- i.e. |s|
// differs from the boundary sqrt(B den) by a relative 1e-6 -- and the quantities are far from
// degenerate: den > 1e-8 (relative error of den below 1e-9 for S <= 20) and B den > 1e-13 (then
// eps_s < 5e-7 sqrt(B den) for S1 S2 <= 130, i.e. normalised coordinates up to ~10: any real camera).
// Everything else -- every borderline point included -- runs the exact OpenCV-order evaluation, so
// the result is always that of sampson_inlier().
// dmin: smallest denominator the pre-filter trusts = T.dmin * |E|_F^2 (T.dmin for the unit-norm models
// the solver emits; every quantity of the test is homogeneous in the scale of E)
// E: the model in registers; Emem: the same nine values in (shared / global) memory, read only by the
// out-of-line fallback -- passing the register copy there would force it onto the stack.
// Decision of the pre-filter from the fused num, den.  t = RN(num - B den); the point is decided when
//     |t| > den 2^e  (2^e >= 2.1e-6 B: num is outside [B (1 - 2e-6) den, B (1 + 2e-6) den], the band the error
//                     analysis above needs),   den > dmin,   and t, den are finite,
// and all three are tested on the HIGH WORDS as integers: hi(|t|) > hi(den) + (e << 20) implies |t| > den 2^e
// for normal numbers (den 2^e is normal because den > dmin >= 1e-13 / B), hi(den) > hi(dmin) implies
// den > dmin, and hi(|t|) < 0x7ff00000 excludes inf / NaN in num or den.  The integer tests are slightly
// stricter than the real-number ones (by at most 2^-20 relative), which only sends a few more points to the
// exact path.  They issue on the integer ALU, which this FP64-bound loop leaves idle: 17 FP64 instructions per
// (model, correspondence) instead of 21 (two threshold products and three FP64 compares before).
__device__ __forceinline__ bool prefilter_decide(double num, double den, const SampThr& T, int hdmin, bool& in) {
    const double t = fma(-den, T.B, num);
    const int ht = __double2hiint(t), hd = __double2hiint(den);
    const int at = ht & 0x7FFFFFFF;
    in = ht < 0;
    return at > hd + T.eoff && at < 0x7FF00000 && hd > hdmin;
}

__device__ __forceinline__ bool sampson_inlier_scaled(const double (&E)[9], const double* Emem, double a1, double b1,
                                                      double a2, double b2, const SampThr& T, int hdmin) {
    const double ex0 = fma(E[0], a1, fma(E[1], b1, E[2]));
    const double ex1 = fma(E[3], a1, fma(E[4], b1, E[5]));
    const double ex2 = fma(E[6], a1, fma(E[7], b1, E[8]));
    const double et0 = fma(E[0], a2, fma(E[3], b2, E[6]));
    const double et1 = fma(E[1], a2, fma(E[4], b2, E[7]));
    const double sx = fma(a2, ex0, fma(b2, ex1, ex2));
    const double den = fma(ex0, ex0, fma(ex1, ex1, fma(et0, et0, et1 * et1)));
    const double num = sx * sx;
    // Branch-free: the integer comparisons feed one (practically never taken) branch.
    bool in;
    if (prefilter_decide(num, den, T, hdmin, in)) return in;
    return sampson_inlier_slow(Emem, a1, b1, a2, b2, T);
}

__device__ __forceinline__ bool sampson_inlier_unit(const double (&E)[9], const double* Emem, double a1, double b1,
                                                    double a2, double b2, const SampThr& T) {
    return sampson_inlier_scaled(E, Emem, a1, b1, a2, b2, T, T.hdmin);
}

// Pre-filter alone: returns true if the fused evaluation decides the test (then `in` is the answer).
__device__ __forceinline__ bool sampson_fast(const double (&E)[9], double a1, double b1, double a2, double b2,
                                             const SampThr& T, int hdmin, bool& in) {
    const double ex0 = fma(E[0], a1, fma(E[1], b1, E[2]));
    const double ex1 = fma(E[3], a1, fma(E[4], b1, E[5]));
    const double ex2 = fma(E[6], a1, fma(E[7], b1, E[8]));
    const double et0 = fma(E[0], a2, fma(E[3], b2, E[6]));
    const double et1 = fma(E[1], a2, fma(E[4], b2, E[7]));
    const double sx = fma(a2, ex0, fma(b2, ex1, ex2));
    const double den = fma(ex0, ex0, fma(ex1, ex1, fma(et0, et0, et1 * et1)));
    const double num = sx * sx;
    return prefilter_decide(num, den, T, hdmin, in);
}

__device__ __forceinline__ int warp_sum(int v) { return __reduce_add_sync(0xFFFFFFFFu, v); }

// k-th smallest (0-based) of n non-negative floats in buf, by bitwise binary search on the
// IEEE bit pattern (OpenCV sorts the float errors as ints: ptsetreg.cpp nth_element on int*).
__device__ float warp_select(const float* buf, int n, int k, int lane) {
    unsigned result = 0;
    for (int bit = 30; bit >= 0; --bit) {
        const unsigned cand = result | (1u << bit);
        int cnt = 0;
        for (int i = lane; i < n; i += 32) cnt += (__float_as_uint(buf[i]) < cand);
        cnt = warp_sum(cnt);
        if (cnt <= k) result = cand;
    }
    return __uint_as_float(result);
}

// =====================================================================================
// Rounds.  OpenCV's estimator is a sequential loop whose sample stream does not depend on
// the data, so samples can be solved ahead of the bookkeeping.  A round r handles the next
// R_r samples of every pair that is still running:
//     ess_sample_kernel   one thread per running pair draws the samples (cv::RNG stream)
//     solve_a_kernel      one lane per (pair, sample): null space, constraints, elimination
//     solve_b1_kernel     one lane per (pair, sample): polynomial, roots -> compact list of real roots
//     solve_b2_kernel     one lane per real root: model + refinement
//     ess_round_kernel    one CTA per running pair: scores the models, replays the sequential
//                         "strictly better -> update niters" bookkeeping in sample order, and
//                         either finishes the pair (mask, compaction) or queues it for round r+1
// Pairs that have stopped drop out of the work list; samples at or beyond a pair's current
// niters are never solved or scored.  The host enqueues enough rounds to cover max_iters;
// rounds with an empty work list cost a few microseconds (grid-stride kernels, small grids:
// five ~3 us launches per empty round).
// =====================================================================================
constexpr int ES_RMAX = 128;         // samples per pair per round, at most
constexpr int ES_MAX_ROUNDS = 40;
constexpr size_t ES_SLOW_CAP = 1 << 18;   // slow-pass slots per round (a few per cent of a round's hypotheses at most)

struct RansacState {
    double best_score;
    double bestE[9];
    unsigned long long rng;
    int iter, niters, have, total_models;
};

struct EssWork {
    RansacState* state;      // [n_pairs]
    int32_t* wl[2];          // work lists (pair indices), ping-pong
    int32_t* ctl;            // [ES_MAX_ROUNDS + 1] running pairs per round
    int32_t* idx;            // [n_pairs * ES_RMAX][5]
    double* rec;             // [EB_DOUBLES][cap]  stage A -> stage B records, SoA
    double* models;          // [cap][10][9], model j of a slot is valid iff bit j of mflags[slot]
    uint32_t* mflags;        // [cap]
    uint32_t* items;         // [cap * 10] real roots of the round, compacted: slot << 4 | root index
    double* item_z;          // [cap * 10] the root itself
    int32_t* nitems;         // [ES_MAX_ROUNDS] roots per round
    uint32_t* slow;          // [cap] hypotheses of the round whose root iteration was not settled by the fast path
    double* slow_state;      // [DK_STATE][cap] their iterates (indexed by position in `slow`), SoA
    int32_t* nslow;          // [ES_MAX_ROUNDS]
    size_t cap;              // n_pairs * ES_RMAX slots
};

size_t ess_work_carve(EssWork* w, char* base, int n_pairs) {
    size_t off = 0;
    auto take = [&](size_t bytes) {
        char* p = base ? base + off : nullptr;
        off += epv_align(bytes);
        return p;
    };
    const size_t cap = (size_t)n_pairs * ES_RMAX;
    RansacState* st = reinterpret_cast<RansacState*>(take((size_t)n_pairs * sizeof(RansacState)));
    int32_t* wl0 = reinterpret_cast<int32_t*>(take((size_t)n_pairs * 4));
    int32_t* wl1 = reinterpret_cast<int32_t*>(take((size_t)n_pairs * 4));
    int32_t* ctl = reinterpret_cast<int32_t*>(take((ES_MAX_ROUNDS + 1) * 4));
    int32_t* idx = reinterpret_cast<int32_t*>(take(cap * 5 * 4));
    double* rec = reinterpret_cast<double*>(take(cap * fivept::EB_DOUBLES * 8));
    double* models = reinterpret_cast<double*>(take(cap * 90 * 8));
    uint32_t* mf = reinterpret_cast<uint32_t*>(take(cap * 4));
    uint32_t* items = reinterpret_cast<uint32_t*>(take(cap * 10 * 4));
    double* item_z = reinterpret_cast<double*>(take(cap * 10 * 8));
    int32_t* nitems = reinterpret_cast<int32_t*>(take(ES_MAX_ROUNDS * 4));
    uint32_t* slow = reinterpret_cast<uint32_t*>(take(cap * 4));
    double* slow_state = reinterpret_cast<double*>(take(ES_SLOW_CAP * fivept::DK_STATE * 8));
    int32_t* nslow = reinterpret_cast<int32_t*>(take(ES_MAX_ROUNDS * 4));
    if (w) {
        w->slow = slow; w->slow_state = slow_state; w->nslow = nslow;
        w->state = st; w->wl[0] = wl0; w->wl[1] = wl1; w->ctl = ctl; w->idx = idx; w->rec = rec;
        w->models = models; w->mflags = mf; w->items = items; w->item_z = item_z; w->nitems = nitems; w->cap = cap;
    }
    return off;
}

struct EssArgs {
    int n_pairs;
    int stride;                 // per-pair row stride of xn / masks
    const double* xn;           // [pair][4][stride] K-normalised x1 y1 x2 y2
    const int32_t* n;           // [pair] correspondences
    int method;
    double prob, thresh;        // thresh already divided by the focal length (OpenCV: threshold /= (fx+fy)/2)
    int max_iters;
    const int32_t* samples;     // optional injected samples [m][5] (shared by all pairs) or nullptr
    int m;
    float* errbuf;              // LMedS scratch [pair][ES_WARPS][stride]
    EssWork w;
    // outputs
    double* E;                  // [pair][9]
    uint8_t* mask;              // [pair][stride] {0,1}
    int32_t* n_inliers;         // [pair]
    int32_t* iters;             // [pair]
    int32_t* n_models;          // [pair]
    int32_t* status;            // [pair] 0 ok, EPIVO_ERR_NOMODEL
    double* xin;                // optional compacted inliers [pair][4][stride] (E3, kitti_E.cpp:106-112)
};

__global__ void ess_init_kernel(EssArgs a) {
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair == 0) {
        a.w.ctl[0] = a.n_pairs;
        for (int r = 1; r <= ES_MAX_ROUNDS; ++r) a.w.ctl[r] = 0;
        for (int r = 0; r < ES_MAX_ROUNDS; ++r) { a.w.nitems[r] = 0; a.w.nslow[r] = 0; }
    }
    if (pair >= a.n_pairs) return;
    const int n = a.n[pair];
    const bool lmeds = a.method == EPIVO_LMEDS;
    RansacState s;
    s.best_score = lmeds ? DBL_MAX : 0.0;
    for (int i = 0; i < 9; ++i) s.bestE[i] = 0.0;
    s.rng = 0xFFFFFFFFFFFFFFFFULL;                                      // RNG rng((uint64)-1)
    s.iter = 0;
    s.have = 0;
    s.total_models = 0;
    int ni = lmeds ? max(update_num_iters(a.prob, 0.45, 5, a.max_iters), 3) : max(a.max_iters, 1);
    if (a.samples) ni = min(ni, a.m);
    if (n < 5) ni = 0;
    if (n == 5) ni = 1;                                                 // count == modelPoints: one solve on all points
    s.niters = ni;
    a.w.state[pair] = s;
    a.w.wl[0][pair] = pair;
}

// one thread per running pair: the next min(R, niters - iter) samples of its stream
__global__ void ess_sample_kernel(EssArgs a, int round, int R) {
    const int count = a.w.ctl[round];
    const int32_t* wl = a.w.wl[round & 1];
    for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < count; w += gridDim.x * blockDim.x) {
        const int pair = wl[w];
        RansacState& st = a.w.state[pair];
        const int n = a.n[pair];
        const int ns = min(R, st.niters - st.iter);
        int32_t* out = a.w.idx + (size_t)w * R * 5;
        if (n == 5) {
            for (int s = 0; s < ns; ++s)
                for (int k = 0; k < 5; ++k) out[s * 5 + k] = k;
        } else if (a.samples) {
            for (int s = 0; s < ns; ++s)
                for (int k = 0; k < 5; ++k) out[s * 5 + k] = a.samples[(size_t)(st.iter + s) * 5 + k];
        } else {
            CvRng rng{st.rng};
            for (int s = 0; s < ns; ++s) {
                int v[5];
                draw_subset(rng, n, v);
                for (int k = 0; k < 5; ++k) out[s * 5 + k] = v[k];
            }
            st.rng = rng.state;
        }
    }
}

// ---- stage A: one warp = 32 hypotheses, 10x20 matrices lane-strided in shared memory -------
constexpr int SA_SMEM = 10 * 20 * 32 * 8;   // 51200 bytes per warp

__global__ void __launch_bounds__(32) solve_a_kernel(EssArgs a, int round, int R) {
    extern __shared__ __align__(16) double s_A[];
    const int lane = threadIdx.x;
    const int count = a.w.ctl[round];
    const int32_t* wl = a.w.wl[round & 1];
    const long long total = (long long)count * R;
    for (long long g = blockIdx.x; g * 32 < total; g += gridDim.x) {
        const long long slot = g * 32 + lane;
        bool valid = slot < total;
        int pair = 0, s = 0;
        if (valid) {
            const int w = (int)(slot / R);
            s = (int)(slot % R);
            pair = wl[w];
            const RansacState& st = a.w.state[pair];
            valid = st.iter + s < st.niters;
        }
        if (valid) {
            const int32_t* id = a.w.idx + slot * 5;
            const double* X1 = a.xn + (size_t)pair * 4 * a.stride;
            double x1[5][2], x2[5][2];
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                const int i = id[k];
                x1[k][0] = X1[i]; x1[k][1] = X1[a.stride + i];
                x2[k][0] = X1[2 * a.stride + i]; x2[k][1] = X1[3 * a.stride + i];
            }
            fivept::stage_a(x1, x2, fivept::SmemMat{s_A + lane}, a.w.rec + slot, a.w.cap);
        }
        __syncwarp();
    }
}

// ---- stage B1: one lane per hypothesis (polynomial + roots); real roots -> compact work list ----
constexpr int SB1_THREADS = 128;
constexpr int SB1_MINBLOCKS = 4;

// the warp's real roots are appended to the round's item list with one atomic per warp
__device__ __forceinline__ void append_roots(int count, const double (&zs)[10], uint32_t slot, uint32_t* items,
                                             double* item_z, int32_t* total) {
    const int lane = threadIdx.x & 31;
    int incl = count;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if (lane >= o) incl += v;
    }
    const int warp_total = __shfl_sync(0xFFFFFFFFu, incl, 31);
    int base = 0;
    if (lane == 31 && warp_total > 0) base = atomicAdd(total, warp_total);
    base = __shfl_sync(0xFFFFFFFFu, base, 31);
    const int off = base + incl - count;
#pragma unroll
    for (int k = 0; k < 10; ++k) {
        if (k < count) {
            items[off + k] = slot << 4 | (uint32_t)k;
            item_z[off + k] = zs[k];
        }
    }
}

// warp-aggregated reservation of one slow-pass slot per lane that asks for one; -1 when the list is full
__device__ __forceinline__ int reserve_slow(bool want, int32_t* total, int cap) {
    const unsigned m = __ballot_sync(0xFFFFFFFFu, want);
    if (!m) return -1;
    const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(total, __popc(m));
    base = __shfl_sync(0xFFFFFFFFu, base, leader);
    const int pos = base + __popc(m & ((1u << lane) - 1));
    return (want && pos < cap) ? pos : -1;
}

__global__ void __launch_bounds__(SB1_THREADS, SB1_MINBLOCKS) solve_b1_kernel(EssArgs a, int round, int R) {
    const int count = a.w.ctl[round];
    const int32_t* wl = a.w.wl[round & 1];
    const long long total = (long long)count * R;
    // whole warps iterate together (the append is a warp collective)
    for (long long base = (long long)blockIdx.x * SB1_THREADS; base < total; base += (long long)gridDim.x * SB1_THREADS) {
        const long long slot = base + threadIdx.x;
        bool valid = slot < total;
        if (valid) {
            const int w = (int)(slot / R), s = (int)(slot % R);
            const RansacState& st = a.w.state[wl[w]];
            valid = st.iter + s < st.niters;
        }
        double zs[10];
        int nz = 0;
        __shared__ double s_state[fivept::DK_STATE * SB1_THREADS];       // iterates of a lane that gives up
        if (valid) {
            nz = fivept::stage_b1<false>(a.w.rec + slot, a.w.cap, zs, s_state + threadIdx.x, SB1_THREADS);
            a.w.mflags[slot] = 0;
        }
        const int pos = reserve_slow(nz < 0, a.w.nslow + round, (int)ES_SLOW_CAP);
        if (nz < 0) {
            if (pos >= 0) {
                a.w.slow[pos] = (uint32_t)slot;
                for (int k = 0; k < fivept::DK_STATE; ++k) a.w.slow_state[(size_t)k * ES_SLOW_CAP + pos] = s_state[k * SB1_THREADS + threadIdx.x];
            } else {
                // list full (never seen: it holds 2^18 per round): finish in place, stalling only this warp
                nz = fivept::stage_b1<true>(a.w.rec + slot, a.w.cap, zs, s_state + threadIdx.x, SB1_THREADS);
            }
        }
        append_roots(max(nz, 0), zs, (uint32_t)slot, a.w.items, a.w.item_z, a.w.nitems + round);
    }
}

// the hypotheses stage B1 could not settle within DK_FAST_SWEEPS sweeps, one lane each, continued from the saved
// iterates up to OpenCV's 300 sweeps (compacted: a warp here holds 32 slow hypotheses, not one among 31 finished)
__global__ void __launch_bounds__(SB1_THREADS) solve_b1_slow_kernel(EssArgs a, int round) {
    const int total = min(a.w.nslow[round], (int)ES_SLOW_CAP);
    for (int base = blockIdx.x * SB1_THREADS; base < total; base += gridDim.x * SB1_THREADS) {
        const int i = base + threadIdx.x;
        double zs[10];
        int nz = 0;
        uint32_t slot = 0;
        if (i < total) {
            slot = a.w.slow[i];
            nz = fivept::stage_b1<true>(a.w.rec + slot, a.w.cap, zs, a.w.slow_state + i, ES_SLOW_CAP);
        }
        append_roots(nz, zs, slot, a.w.items, a.w.item_z, a.w.nitems + round);
    }
}

// ---- stage B2: one lane per real root: model + refinement -----------------------------------------
constexpr int SB2_THREADS = 64;
constexpr int SB2_MINBLOCKS = 4;

__global__ void __launch_bounds__(SB2_THREADS, SB2_MINBLOCKS) solve_b2_kernel(EssArgs a, int round) {
    __shared__ double s_sh[36 * SB2_THREADS];
    const int n_items = a.w.nitems[round];
    for (int it = blockIdx.x * SB2_THREADS + threadIdx.x; it < n_items; it += gridDim.x * SB2_THREADS) {
        const uint32_t code = a.w.items[it];
        const size_t slot = code >> 4;
        const int j = code & 15;
        double E[9];
        if (fivept::stage_b2(a.w.rec + slot, a.w.cap, a.w.item_z[it], s_sh + threadIdx.x, SB2_THREADS, E)) {
            double* out = a.w.models + slot * 90 + j * 9;
#pragma unroll
            for (int k = 0; k < 9; ++k) out[k] = E[k];
            atomicOr(&a.w.mflags[slot], 1u << j);
        }
    }
}

// inlier counts of one or two unit-norm models over correspondences [first, n) in steps of `step`;
// P: pointer type of the point rows (the caller passes the shared-memory array itself when the
// points are staged there, so the loads compile to LDS rather than generic loads)
// The hot loop is branch-free (pre-filter only); points it cannot decide -- practically none -- are
// recounted with the exact test in a second loop that is normally skipped.
constexpr int ES_UNROLL = 3;   // correspondences in flight per lane in the scoring loops

// Inlier counts of two models over the correspondences first, first + step, ... (both models in registers, every
// correspondence tested against both).
// bound >= 0 (whole-model calls only: first = lane, step = 32): the caller needs a count only if it EXCEEDS `bound` --
// RANSAC: the best count before this sub-chunk (a model can only win with strictly more), LMedS: n/2 (the filter asks
// for more than half of the errors below the best median).  Every ES_CHECK iterations the warp adds up what both models
// have (undecided points counted as if they were inliers) plus what is still to come; when neither can exceed the bound
// any more the pass ends -- the returned counts are then partial, which the callers treat exactly like "not more than
// bound".  On the headline data a wrong model (30 % inliers against a best of 84 %) is out after a quarter of the
// points; the result of the estimator is unchanged by construction.
constexpr int ES_CHECK = 2 * ES_UNROLL;
template <class P>
__device__ __forceinline__ void count_two(P X1, int stride, int n, int first, int step, const double* M0,
                                          const double* M1, const SampThr& T, int& c0, int& c1, int bound = -1) {
    double E0[9], E1[9];
#pragma unroll
    for (int c = 0; c < 9; ++c) { E0[c] = M0[c]; E1[c] = M1[c]; }
    int und = 0;                                  // correspondences of this lane the fast test left open (either model)
    int i = first;
    if (bound >= 0) {
        while (i - first < n) {                   // warp-uniform (first = lane, step = 32): every lane reaches the warp sums below
#pragma unroll
            for (int u = 0; u < ES_CHECK; ++u, i += step) {
                if (i < n) {
                    const double a1 = X1[i], b1 = X1[stride + i], a2 = X1[2 * stride + i], b2 = X1[3 * stride + i];
                    bool in0, in1;
                    const bool d0 = sampson_fast(E0, a1, b1, a2, b2, T, T.hdmin, in0);
                    const bool d1 = sampson_fast(E1, a1, b1, a2, b2, T, T.hdmin, in1);
                    c0 += (d0 && in0) ? 1 : 0;
                    c1 += (d1 && in1) ? 1 : 0;
                    und += (d0 && d1) ? 0 : 1;
                }
            }
            // i - first is the same for all lanes: the warp has seen every index below base = i - lane
            const int left = max(n - (i - first), 0);                       // >= correspondences still to come
            const int best_possible = max(warp_sum(c0 + und), warp_sum(c1 + und)) + left;
            if (best_possible <= bound) return;                             // neither model can exceed the bound
        }
    } else {
#pragma unroll ES_UNROLL
        for (; i < n; i += step) {
            const double a1 = X1[i], b1 = X1[stride + i], a2 = X1[2 * stride + i], b2 = X1[3 * stride + i];
            bool in0, in1;
            const bool d0 = sampson_fast(E0, a1, b1, a2, b2, T, T.hdmin, in0);
            const bool d1 = sampson_fast(E1, a1, b1, a2, b2, T, T.hdmin, in1);
            c0 += (d0 && in0) ? 1 : 0;
            c1 += (d1 && in1) ? 1 : 0;
            und += (d0 && d1) ? 0 : 1;
        }
    }
    if (und) {
        for (int i = first; i < n; i += step) {
            const double a1 = X1[i], b1 = X1[stride + i], a2 = X1[2 * stride + i], b2 = X1[3 * stride + i];
            bool in0, in1;
            if (!sampson_fast(E0, a1, b1, a2, b2, T, T.hdmin, in0)) c0 += sampson_inlier_slow(M0, a1, b1, a2, b2, T) ? 1 : 0;
            if (!sampson_fast(E1, a1, b1, a2, b2, T, T.hdmin, in1)) c1 += sampson_inlier_slow(M1, a1, b1, a2, b2, T) ? 1 : 0;
        }
    }
}
template <class P>
__device__ __forceinline__ int count_one(P X1, int stride, int n, int first, int step, const double* M, const SampThr& T) {
    double E[9];
#pragma unroll
    for (int c = 0; c < 9; ++c) E[c] = M[c];
    int c = 0;
    bool undecided = false;
#pragma unroll ES_UNROLL
    for (int i = first; i < n; i += step) {
        bool in;
        const bool d = sampson_fast(E, X1[i], X1[stride + i], X1[2 * stride + i], X1[3 * stride + i], T, T.hdmin, in);
        c += (d && in) ? 1 : 0;
        undecided |= !d;
    }
    if (undecided) {
        for (int i = first; i < n; i += step) {
            const double a1 = X1[i], b1 = X1[stride + i], a2 = X1[2 * stride + i], b2 = X1[3 * stride + i];
            bool in;
            if (!sampson_fast(E, a1, b1, a2, b2, T, T.hdmin, in)) c += sampson_inlier_slow(M, a1, b1, a2, b2, T) ? 1 : 0;
        }
    }
    return c;
}

// ---- scoring + sequential replay + finish: one CTA per running pair -------------------------
// pts_in_smem: the pair's correspondences (4 x stride doubles) are staged in dynamic shared memory
// once and every scoring pass reads them from there; they are read 3+ times per pair and the
// whole batch (45 KB per pair) does not stay in L2.  Off when they do not fit.
__global__ void __launch_bounds__(ES_THREADS, 2) ess_round_kernel(EssArgs a, int round, int R, int last_round,
                                                                  int pts_in_smem) {
    extern __shared__ __align__(16) double s_pts[];
    __shared__ double s_models[ES_SUB][10][9];    // models of the sub-chunk being scored
    __shared__ unsigned s_flags[ES_SUB];           // valid-model bit masks of the sub-chunk's samples
    __shared__ unsigned short s_item[ES_SUB * 10];    // flattened (sample << 4 | model) list of the sub-chunk
    __shared__ int s_nitems;
    __shared__ int s_next;                         // next unclaimed pair of items (dynamic distribution over the warps)
    __shared__ float s_score[ES_SUB][10];         // LMedS: medians
    __shared__ int s_cnt[ES_SUB][10];             // RANSAC: inlier counts
    __shared__ double s_bestE[9];
    __shared__ double s_best_score;
    __shared__ int s_niters, s_iter, s_have, s_total_models;
    __shared__ int s_warpcnt[ES_WARPS];
    __shared__ int s_base;
    __shared__ float s_thr;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int count = a.w.ctl[round];
    const int32_t* wl = a.w.wl[round & 1];
    const bool lmeds = a.method == EPIVO_LMEDS;
    const float thr32 = (float)(a.thresh * a.thresh);
    const SampThr thrR = make_samp_thr(thr32);

    for (int w = blockIdx.x; w < count; w += gridDim.x) {
        const int pair = wl[w];
        const int n = a.n[pair];
        const int64_t so = (int64_t)pair * 4 * a.stride;
        const double* X1 = pts_in_smem ? s_pts : a.xn + so;
        const double* Y1 = X1 + a.stride;
        const double* X2 = Y1 + a.stride;
        const double* Y2 = X2 + a.stride;
        RansacState& st = a.w.state[pair];
        __syncthreads();                                     // previous pair of this CTA is completely done
        if (pts_in_smem) {
            const double* g = a.xn + so;
            for (int i = tid; i < n; i += ES_THREADS) {
                s_pts[i] = g[i];
                s_pts[a.stride + i] = g[a.stride + i];
                s_pts[2 * a.stride + i] = g[2 * a.stride + i];
                s_pts[3 * a.stride + i] = g[3 * a.stride + i];
            }
        }
        if (tid == 0) {
            s_iter = st.iter;
            s_niters = st.niters;
            s_have = st.have;
            s_total_models = st.total_models;
            s_best_score = st.best_score;
        }
        if (tid < 9) s_bestE[tid] = st.bestE[tid];
        __syncthreads();
        const int iter0 = s_iter;
        const int ch = min(R, s_niters - iter0);             // samples solved for this pair in this round
        const double* gmodels = a.w.models + (size_t)w * R * 90;
        const uint32_t* gfl = a.w.mflags + (size_t)w * R;

        // Sub-chunks: score, then replay.  RANSAC usually shrinks niters after the first few samples, so the
        // first two sub-chunks of a pair are 8 samples (samples at or beyond the current niters are never
        // scored), the next 16; a pair that is still running after 32 samples is in for a long run and takes 32
        // at a time (~140 models per barrier: the replay by warp 0 and the wait at the barrier are amortised).
        for (int sbase = 0, sub = 0; sbase < ch; sbase += sub) {
            const int done = iter0 + sbase;
            sub = done < 2 * ES_WARPS ? ES_WARPS : (done < ES_SUB ? 2 * ES_WARPS : ES_SUB);
            const int r = min(sub, min(ch, s_niters - iter0) - sbase);          // samples scored now (>= 1)
            // stage the models of these samples and flatten them into a work list
            for (int i = tid; i < r * 90; i += ES_THREADS) (&s_models[0][0][0])[i] = gmodels[(size_t)sbase * 90 + i];
            for (int i = tid; i < ES_SUB * 10; i += ES_THREADS) (&s_cnt[0][0])[i] = 0;
            if (tid == ES_THREADS - 1) s_next = 0;
            if (warp == 0) {
                const unsigned fl = lane < r ? gfl[sbase + lane] : 0u;
                const int c = __popc(fl);
                int incl = c;
#pragma unroll
                for (int o = 1; o < ES_SUB; o <<= 1) {
                    const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                    if (lane >= o) incl += v;
                }
                if (lane < r) {
                    s_flags[lane] = fl;
                    int pos = incl - c;
                    for (int j = 0; j < 10; ++j)
                        if (fl >> j & 1u) s_item[pos++] = (unsigned short)(lane << 4 | j);
                }
                if (lane == ES_SUB - 1) s_nitems = incl;
            }
            __syncthreads();
            const int M = s_nitems;
            if (n != 5 && M > 0) {
                if (!lmeds) {
                    // a model matters only with more inliers than the best before this sub-chunk (and more than 4).  The
                    // bounded pass pays a warp sum every ES_CHECK iterations, so it is used only where it can end early
                    // enough: with a best of 11 % of the correspondences (RANSAC at 0.05 px) a hopeless model is known
                    // to be hopeless only after 90 % of them and the check costs more than it saves.
                    int best_now = max((int)s_best_score, 4);
                    int first = 0;                                           // items [0, first) are already counted
                    if (s_have == 0 && M > 3 * ES_WARPS) {
                        // No best yet (the pair's first sub-chunk): the first 2 * ES_WARPS models are counted in full,
                        // one pair of models per warp; the largest of those counts is a lower bound of the best BEFORE
                        // every later model of the sub-chunk, which bounds their passes (as the LMedS branch does with
                        // the first medians).  CTA-uniform branch: shared state only.
                        first = 2 * ES_WARPS;
                        {
                            const int code0 = s_item[2 * warp], code1 = s_item[2 * warp + 1];
                            const double* M0 = s_models[code0 >> 4][code0 & 15];
                            const double* M1 = s_models[code1 >> 4][code1 & 15];
                            int c0 = 0, c1 = 0;
                            if (pts_in_smem) count_two(s_pts, a.stride, n, lane, 32, M0, M1, thrR, c0, c1);
                            else count_two(a.xn + so, a.stride, n, lane, 32, M0, M1, thrR, c0, c1);
                            c0 = warp_sum(c0);
                            c1 = warp_sum(c1);
                            if (lane == 0) {
                                s_cnt[code0 >> 4][code0 & 15] = c0;
                                s_cnt[code1 >> 4][code1 & 15] = c1;
                            }
                        }
                        __syncthreads();
                        for (int j = 0; j < first; ++j) best_now = max(best_now, s_cnt[s_item[j] >> 4][s_item[j] & 15]);
                    }
                    const int ransac_bound = 3 * best_now > n ? best_now : -1;
                    if (M >= ES_WARPS) {
                        // the warps claim items two at a time from a shared counter (models differ in nothing, but
                        // a static split leaves the barrier waiting for the warp with the odd item): both models
                        // live in registers and every correspondence (shared memory) is tested against both
                        for (;;) {
                            int j0 = 0;
                            if (lane == 0) j0 = first + 2 * atomicAdd(&s_next, 1);
                            j0 = __shfl_sync(0xFFFFFFFFu, j0, 0);
                            if (j0 >= M) break;
                            const int code0 = s_item[j0];
                            const bool two = j0 + 1 < M;
                            const int code1 = two ? s_item[j0 + 1] : code0;
                            const double* M0 = s_models[code0 >> 4][code0 & 15];
                            const double* M1 = s_models[code1 >> 4][code1 & 15];
                            int c0 = 0, c1 = 0;
                            if (two) {
                                if (pts_in_smem) count_two(s_pts, a.stride, n, lane, 32, M0, M1, thrR, c0, c1, ransac_bound);
                                else count_two(a.xn + so, a.stride, n, lane, 32, M0, M1, thrR, c0, c1, ransac_bound);
                            } else {
                                c0 = pts_in_smem ? count_one(s_pts, a.stride, n, lane, 32, M0, thrR)
                                                 : count_one(a.xn + so, a.stride, n, lane, 32, M0, thrR);
                            }
                            c0 = warp_sum(c0);
                            c1 = warp_sum(c1);
                            if (lane == 0) {
                                s_cnt[code0 >> 4][code0 & 15] = c0;
                                if (two) s_cnt[code1 >> 4][code1 & 15] = c1;
                            }
                        }
                    } else {
                        // fewer models than warps: split the correspondences of each model over several warps
                        const int slices = ES_WARPS / M;
                        const int it = warp / slices, slice = warp % slices;
                        if (it < M) {
                            const int code = s_item[it];
                            const double* E = s_models[code >> 4][code & 15];
                            int cnt = pts_in_smem ? count_one(s_pts, a.stride, n, lane + 32 * slice, 32 * slices, E, thrR)
                                                  : count_one(a.xn + so, a.stride, n, lane + 32 * slice, 32 * slices, E, thrR);
                            cnt = warp_sum(cnt);
                            if (lane == 0) atomicAdd(&s_cnt[code >> 4][code & 15], cnt);
                        }
                    }
                } else {
                    // LMedS.  A model can only become the best if its median is below the best median of
                    // the PREVIOUS sub-chunks, i.e. if more than n/2 of its errors are below it -- a RANSAC
                    // style count with threshold "largest float < best" (no division, no selection).  Only
                    // the few models that pass (and everything before a first best exists) pay for the
                    // exact median: errors to scratch, bitwise radix select.
                    float* buf = a.errbuf + ((int64_t)pair * ES_WARPS + warp) * a.stride;
                    bool have_best = s_best_score < 1e300;
                    float bestf = (float)s_best_score;                       // exact: medians are floats
                    int first = 0;                                           // items [0, first) already have their medians
                    if (!have_best) {
                        // No best yet (the pair's first sub-chunk).  The first ES_WARPS models get their exact medians,
                        // one warp each; the smallest of them is an upper bound of the best median BEFORE every later
                        // model of the sub-chunk, so those go through the same count filter as in the later sub-chunks
                        // instead of paying for ~34 exact medians (40 % of the LMedS scoring time before).
                        first = min(M, ES_WARPS);
                        if (warp < first) {
                            const int code = s_item[warp];
                            const double* E = s_models[code >> 4][code & 15];
                            for (int i = lane; i < n; i += 32) buf[i] = sampson_f32(E, X1[i], Y1[i], X2[i], Y2[i]);
                            __syncwarp();
                            const float med = warp_select(buf, n, n / 2, lane);
                            __syncwarp();
                            if (lane == 0) s_score[code >> 4][code & 15] = med;
                        }
                        __syncthreads();                                     // CTA-uniform branch (shared state only)
                        float t = 3.0e38f;
                        for (int j = 0; j < first; ++j) t = fminf(t, s_score[s_item[j] >> 4][s_item[j] & 15]);
                        bestf = t;
                        have_best = true;
                    }
                    const bool can_filter = have_best && bestf > 0.0f;
                    const SampThr thrL = make_samp_thr(can_filter ? __uint_as_float(__float_as_uint(bestf) - 1u) : 0.0f);
                    const int need = n / 2 + 1;                              // errors that must lie below the best
                    for (;;) {
                        int j0 = 0;
                        if (lane == 0) j0 = first + 2 * atomicAdd(&s_next, 1);
                        j0 = __shfl_sync(0xFFFFFFFFu, j0, 0);
                        if (j0 >= M) break;
                        const int code0 = s_item[j0];
                        const bool two = j0 + 1 < M;
                        const int code1 = two ? s_item[j0 + 1] : code0;
                        const double* M0 = s_models[code0 >> 4][code0 & 15];
                        const double* M1 = s_models[code1 >> 4][code1 & 15];
                        int c0 = need, c1 = need;                            // no best yet: every model needs its median
                        if (have_best && !can_filter) {
                            c0 = c1 = 0;                                     // best median is 0: nothing can beat it
                        } else if (can_filter) {
                            c0 = c1 = 0;
                            if (pts_in_smem) count_two(s_pts, a.stride, n, lane, 32, M0, M1, thrL, c0, c1, need - 1);
                            else count_two(a.xn + so, a.stride, n, lane, 32, M0, M1, thrL, c0, c1, need - 1);
                            c0 = warp_sum(c0);
                            c1 = warp_sum(c1);
                        }
#pragma unroll 1
                        for (int h = 0; h < (two ? 2 : 1); ++h) {
                            const int code = h ? code1 : code0;
                            const double* E = h ? M1 : M0;
                            float med = 3.0e38f;                             // cannot win
                            if ((h ? c1 : c0) >= need) {
                                for (int i = lane; i < n; i += 32) buf[i] = sampson_f32(E, X1[i], Y1[i], X2[i], Y2[i]);
                                __syncwarp();
                                med = warp_select(buf, n, n / 2, lane);
                                __syncwarp();
                            }
                            if (lane == 0) s_score[code >> 4][code & 15] = med;
                        }
                    }
                }
            }
            __syncthreads();
            // Bookkeeping of ptsetreg.cpp run(), which is sequential over (sample, model):
            //     RANSAC: if (good > max(best, 4)) { best = good; E = model; niters = update(ep, niters); }
            //     LMedS : if (median < best)       { best = median; E = model; }
            //     stop as soon as iter >= niters.
            // Replayed by warp 0 with lane q = sample q of the sub-chunk.  "Strictly better" makes the
            // winner the FIRST model that attains the best score, and RANSACUpdateNumIters is a
            // min(niters, f(best)) with f non-increasing in the count, so niters after sample q depends
            // only on the best count among samples <= q: one update per lane, all lanes in parallel.
            if (warp == 0) {
                const int q = lane;
                const bool live = q < r;
                const unsigned fl = live ? s_flags[q] : 0u;
                const int ni_in = s_niters;
                if (n == 5) {                                // minimal case: first solution, all inliers
                    if (lane == 0) {
                        if (!s_have && fl) {
                            const int k = __ffs(fl) - 1;
                            s_have = 1;
                            for (int c = 0; c < 9; ++c) s_bestE[c] = s_models[0][k][c];
                        }
                        s_total_models += __popc(fl);
                        s_iter = iter0 + sbase + r;
                    }
                } else if (!lmeds) {
                    const int b_in = (int)s_best_score;
                    int m = 0, kb = 0;                       // best count of this sample and its first model
                    for (int k = 0; k < 10; ++k)
                        if ((fl >> k & 1u) && s_cnt[q][k] > m) { m = s_cnt[q][k]; kb = k; }
                    const int c = m > 4 ? m : 0;             // a count <= 4 never wins
                    int pa = max(c, b_in);                   // inclusive prefix maximum: best after sample q
#pragma unroll
                    for (int o = 1; o < ES_SUB; o <<= 1) pa = max(pa, __shfl_up_sync(0xFFFFFFFFu, pa, o, ES_SUB));
                    const int ni_after = pa > b_in ? update_num_iters(a.prob, (double)(n - pa) / n, 5, ni_in) : ni_in;
                    int ni_before = __shfl_up_sync(0xFFFFFFFFu, ni_after, 1, ES_SUB);
                    if (q == 0) ni_before = ni_in;
                    const bool stop_here = live && !(iter0 + sbase + q < ni_before);
                    const unsigned stops = __ballot_sync(0xFFFFFFFFu, stop_here);
                    const int qstop = stops ? __ffs(stops) - 1 : r;          // samples [0, qstop) are counted
                    const int B = __shfl_sync(0xFFFFFFFFu, pa, max(qstop - 1, 0));
                    const int ni_out = __shfl_sync(0xFFFFFFFFu, ni_after, max(qstop - 1, 0));
                    const unsigned winners = __ballot_sync(0xFFFFFFFFu, live && q < qstop && c == B && B > b_in);
                    int nmod = (live && q < qstop) ? __popc(fl) : 0;
                    nmod = warp_sum(nmod);
                    if (winners && q == __ffs(winners) - 1) {
                        s_best_score = (double)B;
                        s_have = 1;
                        for (int cc = 0; cc < 9; ++cc) s_bestE[cc] = s_models[q][kb][cc];
                    }
                    if (lane == 0) {
                        s_total_models += nmod;
                        s_iter = iter0 + sbase + qstop;
                        s_niters = qstop > 0 ? ni_out : ni_in;
                    }
                } else {
                    float m = 3.0e38f;                       // smallest median of this sample and its first model
                    int kb = -1;
                    for (int k = 0; k < 10; ++k)
                        if ((fl >> k & 1u) && (kb < 0 || s_score[q][k] < m)) { m = s_score[q][k]; kb = k; }
                    // first (lowest q) sample with the smallest median
                    float mm = kb >= 0 ? m : 3.0e38f;
                    unsigned long long key = ((unsigned long long)__float_as_uint(mm) << 32) | (unsigned)q;   // medians are >= 0
                    if (kb < 0) key = ~0ULL;
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        const unsigned long long other = __shfl_xor_sync(0xFFFFFFFFu, key, o);
                        key = other < key ? other : key;
                    }
                    int nmod = live ? __popc(fl) : 0;
                    nmod = warp_sum(nmod);
                    if (key != ~0ULL && q == (int)(key & 0xFFFFFFFFu) && (double)m < s_best_score) {
                        s_best_score = (double)m;
                        s_have = 1;
                        for (int cc = 0; cc < 9; ++cc) s_bestE[cc] = s_models[q][kb][cc];
                    }
                    if (lane == 0) {
                        s_total_models += nmod;
                        s_iter = iter0 + sbase + r;
                    }
                }
            }
            __syncthreads();
            if (s_iter >= s_niters) break;                   // the sequential loop would have stopped here
        }
        __syncthreads();

        if (s_iter < s_niters && !last_round) {
            // not finished: save the state and queue the pair for the next round
            if (tid == 0) {
                st.iter = s_iter;
                st.niters = s_niters;
                st.have = s_have;
                st.total_models = s_total_models;
                st.best_score = s_best_score;
                const int pos = atomicAdd(&a.w.ctl[round + 1], 1);
                a.w.wl[(round + 1) & 1][pos] = pair;
            }
            if (tid < 9) st.bestE[tid] = s_bestE[tid];
            continue;
        }

        // final mask (ptsetreg.cpp findInliers on the best model), inlier compaction
        if (tid == 0) {
            float t = thr32;
            if (lmeds && s_have && n > 5) {
                double sigma = 2.5 * 1.4826 * (1 + 5. / (n - 5)) * sqrt(s_best_score);
                sigma = fmax(sigma, 0.001);
                t = (float)(sigma * sigma);
            }
            s_thr = t;
            s_base = 0;
        }
        __syncthreads();
        const bool have = s_have != 0;
        const SampThr thrF = make_samp_thr(s_thr);
        double bestE[9];
#pragma unroll
        for (int c = 0; c < 9; ++c) bestE[c] = s_bestE[c];
        uint8_t* mask = a.mask + (int64_t)pair * a.stride;
        double* xin = a.xin ? a.xin + so : nullptr;
        for (int start = 0; start < n; start += ES_THREADS) {
            const int i = start + tid;
            bool in = false;
            double p[4] = {0, 0, 0, 0};
            if (i < n && have) {
                p[0] = X1[i]; p[1] = Y1[i]; p[2] = X2[i]; p[3] = Y2[i];
                in = (n == 5) ? true : sampson_inlier_unit(bestE, s_bestE, p[0], p[1], p[2], p[3], thrF);
            }
            if (i < n) mask[i] = in ? 1 : 0;
            const unsigned bal = __ballot_sync(0xFFFFFFFFu, in);
            if (lane == 0) s_warpcnt[warp] = __popc(bal);
            __syncthreads();
            int off = s_base;
            for (int ww = 0; ww < warp; ++ww) off += s_warpcnt[ww];
            if (in && xin) {
                const int k = off + __popc(bal & ((1u << lane) - 1));
                xin[k] = p[0];
                xin[a.stride + k] = p[1];
                xin[2 * a.stride + k] = p[2];
                xin[3 * a.stride + k] = p[3];
            }
            __syncthreads();
            if (tid == 0) {
                int tot = 0;
                for (int ww = 0; ww < ES_WARPS; ++ww) tot += s_warpcnt[ww];
                s_base += tot;
            }
            __syncthreads();
        }
        if (tid == 0) {
            a.n_inliers[pair] = s_base;
            a.iters[pair] = s_iter;
            a.n_models[pair] = s_total_models;
            a.status[pair] = have ? 0 : EPIVO_ERR_NOMODEL;
        }
        if (tid < 9) a.E[(int64_t)pair * 9 + tid] = have ? s_bestE[tid] : 0.0;
    }
}

// ---- K2 alone: m hypotheses given as coordinates (x1, x2: m x 5 x 2) -------------------------
__global__ void __launch_bounds__(32) five_point_a_kernel(const double* __restrict__ x1, const double* __restrict__ x2,
                                                          int m, double* __restrict__ rec) {
    extern __shared__ __align__(16) double s_A[];
    const int lane = threadIdx.x;
    for (long long g = blockIdx.x; g * 32 < m; g += gridDim.x) {
        const long long i = g * 32 + lane;
        if (i < m) {
            double a[5][2], b[5][2];
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                a[k][0] = x1[(i * 5 + k) * 2];
                a[k][1] = x1[(i * 5 + k) * 2 + 1];
                b[k][0] = x2[(i * 5 + k) * 2];
                b[k][1] = x2[(i * 5 + k) * 2 + 1];
            }
            fivept::stage_a(a, b, fivept::SmemMat{s_A + lane}, rec + i, (size_t)m);
        }
        __syncwarp();
    }
}

// stage B1 + B2 for the stand-alone solver: flags[i] = valid-model mask, models at fixed positions
__global__ void __launch_bounds__(SB1_THREADS, SB1_MINBLOCKS)
five_point_b1_kernel(const double* __restrict__ rec, int m, uint32_t* __restrict__ flags, uint32_t* __restrict__ items,
                     double* __restrict__ item_z, int32_t* __restrict__ n_items) {
    for (long long base = (long long)blockIdx.x * SB1_THREADS; base < m; base += (long long)gridDim.x * SB1_THREADS) {
        const long long i = base + threadIdx.x;
        double zs[10];
        int nz = 0;
        if (i < m) {
            nz = fivept::stage_b1<false>(rec + i, (size_t)m, zs);                // no state buffer: all sweeps in place
            flags[i] = 0;
        }
        append_roots(nz, zs, (uint32_t)i, items, item_z, n_items);
    }
}

__global__ void __launch_bounds__(SB2_THREADS, SB2_MINBLOCKS)
five_point_b2_kernel(const double* __restrict__ rec, int m, const uint32_t* __restrict__ items,
                     const double* __restrict__ item_z, const int32_t* __restrict__ n_items, double* __restrict__ Eout,
                     uint32_t* __restrict__ flags) {
    __shared__ double s_sh[36 * SB2_THREADS];
    const int n = *n_items;
    for (int it = blockIdx.x * SB2_THREADS + threadIdx.x; it < n; it += gridDim.x * SB2_THREADS) {
        const uint32_t code = items[it];
        const size_t i = code >> 4;
        const int j = code & 15;
        double E[9];
        if (fivept::stage_b2(rec + i, (size_t)m, item_z[it], s_sh + threadIdx.x, SB2_THREADS, E)) {
#pragma unroll
            for (int k = 0; k < 9; ++k) Eout[i * 90 + j * 9 + k] = E[k];
            atomicOr(&flags[i], 1u << j);
        }
    }
}

// ---- K3 alone: fixed hypothesis set, m models x n correspondences ----------------------
// Every thread keeps four correspondences in registers; the CTA walks a block of models staged
// in shared memory (broadcast reads); votes are counted per warp with ballot + popc, per CTA
// in shared memory and per model with one global atomicAdd per (CTA, model).
constexpr int SC_THREADS = 256;
// correspondences per thread, in registers: 4, 5 or 6 (template parameter), whichever wastes the fewest point
// slots for the given n (more independent FP64 chains per thread hide more of the DFMA latency: 6 is preferred)
constexpr int SC_MODELS = 128;               // models per CTA tile, at most
constexpr int SC_KUNROLL = 1;   // models in flight per loop iteration
constexpr int SC_MINBLOCKS = 2;

template <int SC_PPT>
__global__ void __launch_bounds__(SC_THREADS, SC_MINBLOCKS)
score_count_kernel(const double* __restrict__ E, int m, int mtile, const double* __restrict__ xn, int stride, int n,
                   float thr32, int32_t* __restrict__ counts) {
    __shared__ double s_E[SC_MODELS][9];
    __shared__ int s_hdmin[SC_MODELS];
    __shared__ int s_cnt[SC_MODELS];
    const int tid = threadIdx.x, lane = tid & 31;
    const int m0 = blockIdx.y * mtile;
    const int mm = min(mtile, m - m0);
    const SampThr T = make_samp_thr(thr32);
    for (int i = tid; i < mm * 9; i += SC_THREADS) (&s_E[0][0])[i] = E[(int64_t)m0 * 9 + i];
    for (int i = tid; i < mm; i += SC_THREADS) s_cnt[i] = 0;
    __syncthreads();
    for (int k = tid; k < mm; k += SC_THREADS) {
        double f2 = 0.0;
#pragma unroll
        for (int c = 0; c < 9; ++c) f2 += s_E[k][c] * s_E[k][c];
        s_hdmin[k] = samp_hi(fabs(T.dmin * f2)) | (f2 > 0.0 ? 0 : 0x7FF00000);   // zero / NaN / inf scale: the pre-filter never decides
    }
    double a1[SC_PPT], b1[SC_PPT], a2[SC_PPT], b2[SC_PPT];
    bool valid[SC_PPT];
#pragma unroll
    for (int q = 0; q < SC_PPT; ++q) {
        const int i = (blockIdx.x * SC_PPT + q) * SC_THREADS + tid;
        valid[q] = i < n;
        const int ii = valid[q] ? i : 0;
        a1[q] = xn[ii]; b1[q] = xn[stride + ii]; a2[q] = xn[2 * stride + ii]; b2[q] = xn[3 * stride + ii];
    }
    __syncthreads();
    // Branch-free hot loop (as count_two): the SC_PPT correspondences of a thread are independent FP64 chains
    // that the compiler interleaves only when no branch separates them (with one branch per point the first
    // version exposed the full DFMA latency of every chain: 60 % of the FP64 pipe).  Points the pre-filter
    // cannot decide are flagged in bit 16 of the vote word; a set flag anywhere in the warp -- practically
    // never -- sends the whole warp through the exact test for that model.
#pragma unroll SC_KUNROLL
    for (int k = 0; k < mm; ++k) {
        double e[9];
#pragma unroll
        for (int c = 0; c < 9; ++c) e[c] = s_E[k][c];
        const int dmin = s_hdmin[k];
        int v = 0;
#pragma unroll
        for (int q = 0; q < SC_PPT; ++q) {
            bool in;
            const bool d = sampson_fast(e, a1[q], b1[q], a2[q], b2[q], T, dmin, in);
            v += (valid[q] && d && in) ? 1 : 0;
            v |= (valid[q] && !d) ? (1 << 16) : 0;
        }
        v = warp_sum(v);                     // counts <= 32 SC_PPT in the low half, undecided lanes in the high half
        if (v >> 16) {                       // warp-uniform
            int c = 0;
#pragma unroll
            for (int q = 0; q < SC_PPT; ++q)
                c += (valid[q] && sampson_inlier_scaled(e, s_E[k], a1[q], b1[q], a2[q], b2[q], T, dmin)) ? 1 : 0;
            v = warp_sum(c);
        }
        if (lane == 0 && v) atomicAdd(&s_cnt[k], v);
    }
    __syncthreads();
    for (int k = tid; k < mm; k += SC_THREADS)
        if (s_cnt[k]) atomicAdd(&counts[m0 + k], s_cnt[k]);
}

// LMedS medians of a fixed hypothesis set: one warp per model
__global__ void __launch_bounds__(256)
score_median_kernel(const double* __restrict__ E, int m, const double* __restrict__ xn, int stride, int n,
                    float* __restrict__ errbuf, float* __restrict__ medians) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= m) return;
    double e[9];
    for (int q = 0; q < 9; ++q) e[q] = E[(int64_t)warp * 9 + q];
    float* buf = errbuf + (int64_t)warp * stride;
    for (int i = lane; i < n; i += 32)
        buf[i] = sampson_f32(e, xn[i], xn[stride + i], xn[2 * stride + i], xn[3 * stride + i]);
    __syncwarp();
    const float med = warp_select(buf, n, n / 2, lane);
    if (lane == 0) medians[warp] = med;
}

// first model with the largest count (block-level argmax, lowest index wins ties)
__global__ void __launch_bounds__(256) argmax_first_kernel(const int32_t* __restrict__ counts, int m, int* best) {
    __shared__ unsigned long long s_key[8];
    unsigned long long key = 0;
    for (int i = threadIdx.x; i < m; i += 256) {
        // larger count wins; among equals the smaller index wins
        unsigned long long k = ((unsigned long long)(unsigned)counts[i] << 32) | (unsigned)(0x7FFFFFFF - i);
        key = k > key ? k : key;
    }
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long other = __shfl_xor_sync(0xFFFFFFFFu, key, o);
        key = other > key ? other : key;
    }
    if ((threadIdx.x & 31) == 0) s_key[threadIdx.x >> 5] = key;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) key = s_key[w] > key ? s_key[w] : key;
        *best = m > 0 ? 0x7FFFFFFF - (int)(key & 0xFFFFFFFFu) : -1;
    }
}

__global__ void mask_of_model_kernel(const double* __restrict__ E, const int* __restrict__ best,
                                     const double* __restrict__ xn, int stride, int n, float thr32,
                                     uint8_t* __restrict__ mask) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int b = *best;
    if (b < 0) { mask[i] = 0; return; }
    double e[9];
    for (int q = 0; q < 9; ++q) e[q] = E[(int64_t)b * 9 + q];
    mask[i] = sampson_inlier(e, xn[i], xn[stride + i], xn[2 * stride + i], xn[3 * stride + i], make_samp_thr(thr32)) ? 1 : 0;
}

// pixel -> K-normalised float64 (five-point.cpp: one scale-and-shift per coordinate)
__global__ void normalize_kernel(const float* __restrict__ p0, const float* __restrict__ p1, int n, int stride,
                                 double ax, double bx, double ay, double by, double* __restrict__ xn) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    xn[i] = __fma_rn((double)p0[2 * i], ax, bx);
    xn[stride + i] = __fma_rn((double)p0[2 * i + 1], ay, by);
    xn[2 * stride + i] = __fma_rn((double)p1[2 * i], ax, bx);
    xn[3 * stride + i] = __fma_rn((double)p1[2 * i + 1], ay, by);
}

}  // namespace

int epv_normalize_launch(epivo_ctx* ctx, const float* d_p0, const float* d_p1, int n, int stride, const double K[9],
                         double* d_xn) {
    if (n <= 0) return EPIVO_OK;
    const double ax = 1.0 / K[0], ay = 1.0 / K[4];
    normalize_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(d_p0, d_p1, n, stride, ax, -K[2] * ax, ay,
                                                               -K[5] * ay, d_xn);
    EPV_LAUNCHED(ctx);
    return EPIVO_OK;
}

size_t epv_essential_work_bytes(int n_pairs) { return ess_work_carve(nullptr, nullptr, std::max(n_pairs, 1)); }

// round sizes: a short first round for RANSAC (on KITTI-like data it stops after ~10 samples), then
// doubling up to ES_RMAX; LMedS has a fixed iteration count and takes it in ES_RMAX pieces
static int ess_round_sizes(int method, double prob, int max_iters, int m_samples, int* R) {
    int total;
    int first;
    if (method == EPIVO_LMEDS) {
        double num = log(fmax(1.0 - prob, DBL_MIN)), den = log(1.0 - pow(1.0 - 0.45, 5.0));
        int ni = (int)rint(num / den);
        total = std::max(std::min(ni, max_iters), 3);
        first = ES_RMAX;
    } else {
        total = std::max(max_iters, 1);
        first = 2 * ES_WARPS;
    }
    if (m_samples > 0) total = std::min(total, m_samples);
    int nr = 0, done = 0, r = first;
    while (done < total && nr < ES_MAX_ROUNDS) {
        const bool last_slot = nr == ES_MAX_ROUNDS - 1;
        R[nr] = last_slot ? std::min(total - done, ES_RMAX) : std::min(r, total - done);
        done += R[nr];
        ++nr;
        r = std::min(2 * r, ES_RMAX);
    }
    return done >= total ? nr : -1;
}

int epv_essential_launch(epivo_ctx* ctx, const EssentialPlan& p) {
    if (p.n_pairs <= 0) return EPIVO_OK;
    if (!p.work || p.work_bytes < epv_essential_work_bytes(p.n_pairs))
        EPV_FAIL(ctx, EPIVO_ERR_INVALID, "essential work buffer too small");
    EssArgs a{};
    a.n_pairs = p.n_pairs;
    a.stride = p.stride;
    a.xn = p.xn;
    a.n = p.n;
    a.method = p.method;
    a.prob = p.prob;
    a.thresh = p.thresh;
    a.max_iters = p.max_iters;
    a.samples = p.samples;
    a.m = p.m;
    a.errbuf = p.errbuf;
    a.E = p.E;
    a.mask = p.mask;
    a.n_inliers = p.n_inliers;
    a.iters = p.iters;
    a.n_models = p.n_models;
    a.status = p.status;
    a.xin = p.xin;
    ess_work_carve(&a.w, reinterpret_cast<char*>(p.work), p.n_pairs);
    int R[ES_MAX_ROUNDS];
    const int nr = ess_round_sizes(p.method, p.prob, p.max_iters, p.samples ? p.m : 0, R);
    if (nr < 0)
        EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "max_iters = %d needs more than %d rounds of %d samples", p.max_iters,
                 ES_MAX_ROUNDS, ES_RMAX);
    if (!ctx->func_attrs_set) {                  // function attributes are per device: once per context
        EPV_CUDA(ctx, cudaFuncSetAttribute(solve_a_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SA_SMEM));
        EPV_CUDA(ctx, cudaFuncSetAttribute(five_point_a_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SA_SMEM));
        EPV_CUDA(ctx, cudaFuncSetAttribute(ess_round_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        ctx->func_attrs_set = true;
    }
    // correspondences staged in shared memory when two CTAs per SM still fit (<= 100 KB each)
    const size_t pts_bytes = (size_t)p.stride * 4 * sizeof(double);
    const size_t pts_smem = pts_bytes <= 100 * 1024 ? pts_bytes : 0;
    ess_init_kernel<<<(p.n_pairs + 127) / 128, 128, 0, ctx->stream>>>(a);
    EPV_LAUNCHED(ctx);
    // Round 0 runs on every pair; later rounds usually see a short (often empty) work list, so their
    // grids are small and loop (grid-stride) -- an empty round is four near-empty launches.
    const int sms = ctx->sm_count;
    for (int r = 0; r < nr; ++r) {
        const long long pairs_ub = p.n_pairs;
        const long long slots_ub = pairs_ub * R[r];
        const bool full = r == 0;
        const unsigned g_pairs = (unsigned)std::min<long long>(pairs_ub, full ? pairs_ub : 2LL * sms);
        const unsigned g_samp = (unsigned)std::min<long long>((pairs_ub + 127) / 128, full ? (1LL << 30) : sms);
        const unsigned g_a = (unsigned)std::min<long long>((slots_ub + 31) / 32, full ? (1LL << 30) : 4LL * sms);
        const unsigned g_b1 = (unsigned)std::min<long long>((slots_ub + SB1_THREADS - 1) / SB1_THREADS,
                                                            full ? (1LL << 30) : 4LL * sms);
        // stage B2 sees ~4.3 real roots per hypothesis; its grid-stride loop absorbs the rest
        const unsigned g_b2 = (unsigned)std::min<long long>((slots_ub * 5 + SB2_THREADS - 1) / SB2_THREADS,
                                                            full ? (1LL << 30) : 4LL * sms);
        ess_sample_kernel<<<g_samp, 128, 0, ctx->stream>>>(a, r, R[r]);
        EPV_LAUNCHED(ctx);
        solve_a_kernel<<<g_a, 32, SA_SMEM, ctx->stream>>>(a, r, R[r]);
        EPV_LAUNCHED(ctx);
        solve_b1_kernel<<<g_b1, SB1_THREADS, 0, ctx->stream>>>(a, r, R[r]);
        EPV_LAUNCHED(ctx);
        solve_b1_slow_kernel<<<full ? 2 * sms : sms, SB1_THREADS, 0, ctx->stream>>>(a, r);
        EPV_LAUNCHED(ctx);
        solve_b2_kernel<<<g_b2, SB2_THREADS, 0, ctx->stream>>>(a, r);
        EPV_LAUNCHED(ctx);
        if (r == 0 && p.ev_presolved) EPV_CUDA(ctx, cudaEventRecord(p.ev_presolved, ctx->stream));
        ess_round_kernel<<<g_pairs, ES_THREADS, pts_smem, ctx->stream>>>(a, r, R[r], r == nr - 1 ? 1 : 0, pts_smem > 0);
        EPV_LAUNCHED(ctx);
    }
    return EPIVO_OK;
}

size_t epv_essential_errbuf_floats(int n_pairs, int stride) { return (size_t)n_pairs * ES_WARPS * stride; }

// d_rec: m * 96 doubles; d_items: m * 10 u32; d_item_z: m * 10 doubles; d_count: 1 int (scratch).
// d_E: m x 10 x 9 with model j of sample i valid iff bit j of d_flags[i].
int epv_five_point_launch(epivo_ctx* ctx, const double* d_x1, const double* d_x2, int m, double* d_rec,
                          uint32_t* d_items, double* d_item_z, int32_t* d_count, double* d_E, uint32_t* d_flags) {
    if (m <= 0) return EPIVO_OK;
    EPV_CUDA(ctx, cudaFuncSetAttribute(five_point_a_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SA_SMEM));
    EPV_CUDA(ctx, cudaMemsetAsync(d_count, 0, 4, ctx->stream));
    five_point_a_kernel<<<(m + 31) / 32, 32, SA_SMEM, ctx->stream>>>(d_x1, d_x2, m, d_rec);
    EPV_LAUNCHED(ctx);
    five_point_b1_kernel<<<(m + SB1_THREADS - 1) / SB1_THREADS, SB1_THREADS, 0, ctx->stream>>>(d_rec, m, d_flags, d_items,
                                                                                            d_item_z, d_count);
    EPV_LAUNCHED(ctx);
    const long long ub = (long long)m * 5;
    five_point_b2_kernel<<<(unsigned)((ub + SB2_THREADS - 1) / SB2_THREADS), SB2_THREADS, 0, ctx->stream>>>(
        d_rec, m, d_items, d_item_z, d_count, d_E, d_flags);
    EPV_LAUNCHED(ctx);
    return EPIVO_OK;
}

int epv_score_launch(epivo_ctx* ctx, const double* d_E, int m, const double* d_xn, int stride, int n, double thresh,
                     int32_t* d_counts, float* d_medians, float* d_errbuf, int* d_best, uint8_t* d_mask) {
    const float thr32 = (float)(thresh * thresh);
    EPV_CUDA(ctx, cudaMemsetAsync(d_counts, 0, (size_t)std::max(m, 1) * 4, ctx->stream));
    if (m > 0 && n > 0) {
        // model tile: as large as possible (fewer re-loads of the correspondences) while the grid still
        // covers the GPU about four times
        int ppt = 6, best_slots = 0;
        for (int c = 6; c >= 4; --c) {           // fewest point slots; ties go to the larger count
            const int slots = (n + SC_THREADS * c - 1) / (SC_THREADS * c) * c;
            if (c == 6 || slots < best_slots) { ppt = c; best_slots = slots; }
        }
        const int pblocks = (n + SC_THREADS * ppt - 1) / (SC_THREADS * ppt);
        int mtile = SC_MODELS;
        while (mtile > 8 && (long long)pblocks * ((m + mtile - 1) / mtile) < 4LL * ctx->sm_count) mtile /= 2;
        dim3 grid(pblocks, (m + mtile - 1) / mtile);
        if (ppt == 6)
            score_count_kernel<6><<<grid, SC_THREADS, 0, ctx->stream>>>(d_E, m, mtile, d_xn, stride, n, thr32, d_counts);
        else if (ppt == 5)
            score_count_kernel<5><<<grid, SC_THREADS, 0, ctx->stream>>>(d_E, m, mtile, d_xn, stride, n, thr32, d_counts);
        else
            score_count_kernel<4><<<grid, SC_THREADS, 0, ctx->stream>>>(d_E, m, mtile, d_xn, stride, n, thr32, d_counts);
        EPV_LAUNCHED(ctx);
        if (d_medians) {
            score_median_kernel<<<(m * 32 + 255) / 256, 256, 0, ctx->stream>>>(d_E, m, d_xn, stride, n, d_errbuf,
                                                                             d_medians);
            EPV_LAUNCHED(ctx);
        }
    }
    argmax_first_kernel<<<1, 256, 0, ctx->stream>>>(d_counts, m, d_best);
    EPV_LAUNCHED(ctx);
    if (n > 0) {
        mask_of_model_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(d_E, d_best, d_xn, stride, n, thr32, d_mask);
        EPV_LAUNCHED(ctx);
    }
    return EPIVO_OK;
}
