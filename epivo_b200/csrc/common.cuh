// Shared host/device plumbing for libepivo_b200: context, workspace, error handling.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "../../include/epivo_b200.h"

// Stage ranges for profilers (SURVEY section 5, "tracing"): header-only NVTX v3, active only when the context was created
// with EPIVO_NVTX=1 in the environment -- otherwise one predictable branch per stage.
#include <nvtx3/nvToolsExt.h>
struct epivo_ctx;
struct EpvRange {
    bool on;
    inline EpvRange(const epivo_ctx* ctx, const char* name);
    ~EpvRange() { if (on) nvtxRangePop(); }
};

struct epivo_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    std::string err;
    int64_t launches = 0;
    bool func_attrs_set = false;   // per-device opt-in attributes (large dynamic shared memory) applied for this context's device
    // grow-only device workspace, carved by a bump pointer per call
    char* ws = nullptr;
    size_t ws_bytes = 0;
    size_t ws_used = 0;
    // grow-only pinned host staging buffer
    char* pin = nullptr;
    size_t pin_bytes = 0;
    size_t pin_used = 0;
    // events around the kernels of the last stage-wise call that records them (epivo_last_kernel_ms)
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr;
    bool nvtx = false;             // EPIVO_NVTX=1 at epivo_create: NVTX ranges around the stages (nsys / ncu --nvtx)
};

inline EpvRange::EpvRange(const epivo_ctx* ctx, const char* name) : on(ctx && ctx->nvtx) { if (on) nvtxRangePushA(name); }

#define EPV_FAIL(ctx, code, ...)                          \
    do {                                                  \
        char _b[512];                                     \
        snprintf(_b, sizeof(_b), __VA_ARGS__);            \
        (ctx)->err = _b;                                  \
        return (code);                                    \
    } while (0)

#define EPV_CUDA(ctx, expr)                                                                   \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            EPV_FAIL(ctx, EPIVO_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                     __FILE__, __LINE__);                                                     \
        }                                                                                     \
    } while (0)

#define EPV_LAUNCHED(ctx)                      \
    do {                                       \
        (ctx)->launches++;                     \
        EPV_CUDA(ctx, cudaGetLastError());     \
    } while (0)

static inline size_t epv_align(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// Reserve at least `bytes` of device workspace (may reallocate: syncs the stream first).
int epv_ws_reserve(epivo_ctx* ctx, size_t bytes);
int epv_pin_reserve(epivo_ctx* ctx, size_t bytes);

template <typename T>
static inline T* epv_ws_take(epivo_ctx* ctx, size_t count) {
    size_t off = epv_align(ctx->ws_used);
    ctx->ws_used = off + count * sizeof(T);
    return reinterpret_cast<T*>(ctx->ws + off);
}
template <typename T>
static inline T* epv_pin_take(epivo_ctx* ctx, size_t count) {
    size_t off = epv_align(ctx->pin_used);
    ctx->pin_used = off + count * sizeof(T);
    return reinterpret_cast<T*>(ctx->pin + off);
}

// ---- matcher (match.cu) -------------------------------------------------------------
constexpr int EPV_KEY_SHIFT = 22;                       // key = dist << 22 | index
constexpr uint32_t EPV_IDX_MASK = (1u << EPV_KEY_SHIFT) - 1;

struct MatchPlan {
    // descriptor rows are `words` 32-bit words; pair p matches rows [q0 + p*qs, +nq) against
    // rows [t0 + p*ts, +nt) of the same device array.
    const uint32_t* desc;      // raw descriptors
    uint32_t* planes;          // HAMMING2 bit-plane copy (same shape), or nullptr for HAMMING
    int64_t total_rows;        // rows in desc (for the plane pre-pass)
    int words;
    int norm;
    int top2;                  // also keep the second-best key per query
    int n_pairs;
    int64_t q0, qs, t0, ts;
    int nq, nt;
    int tsplits;               // train-set splits (grid.z); row keys are per split
    uint32_t* rowkey;          // [tsplits][n_pairs][stride]
    uint32_t* rowkey2;         // [tsplits][n_pairs][stride] or nullptr
    uint32_t* colkey;          // [n_pairs][stride]
    int stride;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // optional: recorded right around the tile kernel
    // optional general addressing (device arrays; all three or none): pair p matches frame fq[p] against frame
    // ft[p] of a frame array with qs (= ts) rows per slot, counts[frame] of them valid; q0 / t0 are ignored
    const int32_t* fq = nullptr;
    const int32_t* ft = nullptr;
    const int32_t* counts = nullptr;
    int64_t prepass_row0 = 0;  // first row of desc / planes the HAMMING2 plane pre-pass converts (total_rows rows)
};
int epv_match_launch(epivo_ctx* ctx, const MatchPlan& mp, bool run_prepass);
int epv_planes_launch(epivo_ctx* ctx, const uint32_t* desc, uint32_t* planes, int64_t rows, int words, cudaStream_t st);
int epv_match_splits(const epivo_ctx* ctx, int n_pairs, int nq, int nt);   // train splits that fill the GPU
int epv_match_pairs_per_wave(const epivo_ctx* ctx, int nq);                // pairs per full wave of matcher CTAs

struct FinalizePlan {
    int n_pairs, nq, nt, stride, mode, tsplits;
    float ratio;
    const uint32_t* rowkey;
    const uint32_t* rowkey2;
    const uint32_t* colkey;
    // outputs, all [n_pairs][stride] (nullable except n_matches)
    int32_t* mq;
    int32_t* mt;
    int32_t* md;
    int32_t* md2;
    int32_t* n_matches;        // [n_pairs]
    // optional fused gather (M2) + K-normalisation (E stage input)
    const float* kps;          // keypoints, row r -> (x, y); same row indexing as the descriptors
    int64_t q0, qs, t0, ts;
    float* p0;                 // [n_pairs][stride][2] pixel
    float* p1;
    double* xn;                // [n_pairs][4][stride]: x1, y1, x2, y2 normalised
    double ax, bx, ay, by;     // x = u*ax + bx
    const int32_t* fq = nullptr;       // optional general addressing, as in MatchPlan
    const int32_t* ft = nullptr;
    const int32_t* counts = nullptr;
};
int epv_finalize_launch(epivo_ctx* ctx, const FinalizePlan& fp);
