// K1: brute-force Hamming / Hamming2 nearest-neighbour matcher for sm_100a.
//
// Replaces cv::BFMatcher(NORM_HAMMING2, true).match (reference kitti_ba.cpp:602,641).
// One pass over the nq x nt distance matrix yields BOTH the per-query minimum (row key)
// and the per-train minimum (column key) that the mutual-NN cross-check needs, so the
// cross-check costs one evaluation per (query, train) pair, not two.
//
// Layout / mapping
//   * descriptors are rows of WORDS 32-bit words.  For NORM_HAMMING2 a pre-pass rewrites
//     every row as bit planes (L = even bits, H = odd bits, two source words interleaved
//     per output word) so that the 2-bit-group distance is popc((Lq^Lt) | (Hq^Ht)):
//     4 POPC per 256-bit pair instead of 8 XOR/SHF/LOP/POPC groups.
//   * a CTA owns THREADS*RQ = 128*8 query rows (RQ rows per thread, held in registers, loaded with
//     128-bit coalesced loads) and streams ALL train rows through shared memory in tiles of
//     TILE rows, double-buffered by TMA 1-D bulk copies (cp.async.bulk + mbarrier).  Every
//     lane reads the same train row (shared-memory broadcast, LDS.128).
//   * keys are dist << 22 | index, so an unsigned min gives "smallest distance, then
//     lowest index" = OpenCV's first-minimum tie-break.  Row keys stay in registers; column
//     keys are reduced across the warp with REDUX.MIN, across warps through per-warp shared
//     memory slots and across CTAs with one global atomicMin per (CTA, train row).
//   * grid = (query blocks, pairs): a batch of frame pairs is one launch.
#include <algorithm>

#include "common.cuh"

namespace {

constexpr int MT_THREADS = 128;
constexpr int MT_RQ = 8;
constexpr int MT_MINBLOCKS = 4;
constexpr int MT_TILE = 128;
constexpr int MT_UNROLL = 1;

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t phase) {
    uint32_t ok;
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(phase)
        : "memory");
    return ok != 0;
}

// NORM_HAMMING2 pre-pass: words (a0, a1) -> L = a0.even | a1.even << 1, H = a0.odd >> 1 | a1.odd
__global__ void desc_planes_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, int64_t rows,
                                   int words) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // one thread per (row, word pair)
    int half = words / 2;
    if (i >= rows * half) return;
    int64_t r = i / half;
    int w = (int)(i % half);
    uint32_t a0 = in[r * words + 2 * w], a1 = in[r * words + 2 * w + 1];
    out[r * words + w] = (a0 & 0x55555555u) | ((a1 & 0x55555555u) << 1);
    out[r * words + half + w] = ((a0 >> 1) & 0x55555555u) | (a1 & 0xAAAAAAAAu);
}

// 3:2 carry-save compressor: a + b + c = s + 2*carry, bitwise (2 LOP3)
__device__ __forceinline__ void csa(uint32_t a, uint32_t b, uint32_t c, uint32_t& s, uint32_t& carry) {
    s = a ^ b ^ c;
    carry = (a & b) | (a & c) | (b & c);
}

// Distance of one descriptor pair.  POPC runs on the XU pipe at 16 lanes/clk/SM -- a quarter of
// the ALU (LOP3) rate -- so words are first compressed with carry-save adders and only the
// compressed words are counted: 3 POPC instead of 4 per 256-bit Hamming2 pair (4 instead of 8
// for plain Hamming), which balances the XU and ALU pipes.
template <int WORDS, bool NORM2>
__device__ __forceinline__ uint32_t desc_dist(const uint32_t (&q)[WORDS], const uint32_t (&t)[WORDS]) {
    constexpr int NX = NORM2 ? WORDS / 2 : WORDS;
    uint32_t x[NX];
    if (NORM2) {
#pragma unroll
        for (int w = 0; w < NX; ++w) x[w] = (q[w] ^ t[w]) | (q[w + NX] ^ t[w + NX]);
    } else {
#pragma unroll
        for (int w = 0; w < NX; ++w) x[w] = q[w] ^ t[w];
    }
    if (NX == 4) {
        uint32_t s, c;
        csa(x[0], x[1], x[2], s, c);
        return (uint32_t)__popc(s) + (uint32_t)__popc(x[3]) + 2u * (uint32_t)__popc(c);
    } else if (NX == 8) {
        uint32_t s0, c0, s1, c1, s2, c2, s3, c3;
        csa(x[0], x[1], x[2], s0, c0);
        csa(x[3], x[4], x[5], s1, c1);
        csa(s0, s1, x[6], s2, c2);
        csa(c0, c1, c2, s3, c3);
        return (uint32_t)__popc(s2) + (uint32_t)__popc(x[7]) + 2u * (uint32_t)__popc(s3) + 4u * (uint32_t)__popc(c3);
    } else {
        uint32_t d = 0;
#pragma unroll
        for (int w = 0; w < NX; ++w) d += __popc(x[w]);
        return d;
    }
}

// RQ = query rows per thread: 8 (a CTA covers 1024 query rows) or 6 (768), whichever wastes fewer row slots for the
// given set size -- 1500 EuRoC keypoints are two CTAs either way, but 2 x 768 instead of 2 x 1024 slots (mt_pick_rq).
template <int WORDS, int RQ, bool NORM2, bool TOP2, bool COUNTS>
__global__ void __launch_bounds__(MT_THREADS, WORDS <= 8 ? MT_MINBLOCKS : 1)   // 64-byte descriptors need the registers
match_tile_kernel(const uint32_t* __restrict__ desc, int64_t q0, int64_t qs, int64_t t0, int64_t ts, int nq,
                  int nt, uint32_t* __restrict__ rowkey, uint32_t* __restrict__ rowkey2,
                  uint32_t* __restrict__ colkey, int stride, int tiles_per_split, int64_t part_stride,
                  const int32_t* __restrict__ fq, const int32_t* __restrict__ ft, const int32_t* __restrict__ counts) {
    extern __shared__ uint32_t s_occupancy_pad[];   // unused: sized by the host to cap CTAs per SM (co-scheduling)
    __shared__ __align__(128) uint32_t s_tile[2][MT_TILE * WORDS];
    __shared__ uint32_t s_col[2][MT_THREADS / 32][MT_TILE];   // per-warp column minima of the tile in flight
    __shared__ __align__(8) uint64_t s_bar[2];

    const int pair = blockIdx.y;
    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int qbase = blockIdx.x * (MT_THREADS * RQ);
    // GENERAL variant (template flag COUNTS): pair p matches frame fq[p] (query) against frame ft[p] (train) of a
    // frame array with qs rows per frame slot, of which counts[frame] are valid
    int64_t qrow0 = q0 + (int64_t)pair * qs, trow0 = t0 + (int64_t)pair * ts;
    if (COUNTS) {
        const int f0 = fq[pair], f1 = ft[pair];
        nq = counts[f0];
        nt = counts[f1];
        qrow0 = (int64_t)f0 * qs;
        trow0 = (int64_t)f1 * ts;
    }
    if (qbase >= nq) return;
    const uint32_t* qrows = desc + qrow0 * WORDS;
    const uint32_t* trows = desc + trow0 * WORDS;
    // this CTA's share of the train tiles (blockIdx.z splits the train set so that a single
    // small pair still fills the GPU; a batch of pairs uses one split)
    const int tile0 = blockIdx.z * tiles_per_split;
    const int n_tiles = min((nt + MT_TILE - 1) / MT_TILE - tile0, tiles_per_split);
    if (n_tiles <= 0) return;
    trows += (int64_t)tile0 * MT_TILE * WORDS;
    nt -= tile0 * MT_TILE;
    colkey += tile0 * MT_TILE;
    rowkey += blockIdx.z * part_stride;
    if (TOP2) rowkey2 += blockIdx.z * part_stride;
    const uint32_t jglob0 = (uint32_t)(tile0 * MT_TILE);

    if (tid == 0) {
        mbar_init(&s_bar[0], 1);
        mbar_init(&s_bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        for (int b = 0; b < 2 && b < n_tiles; ++b) {
            int rows = min(MT_TILE, nt - b * MT_TILE);
            uint32_t bytes = (uint32_t)rows * WORDS * 4;
            mbar_expect_tx(&s_bar[b], bytes);
            tma_load_1d(s_tile[b], trows + (int64_t)b * MT_TILE * WORDS, bytes, &s_bar[b]);
        }
    }

    // query rows -> registers (rows past nq are clamped to the last valid row: a duplicate
    // produces the same keys as the genuine row, so it never changes a minimum)
    uint32_t q[RQ][WORDS];
    uint32_t qidx[RQ];
    uint32_t best[RQ], best2[RQ];
#pragma unroll
    for (int r = 0; r < RQ; ++r) {
        int qi = min(qbase + r * MT_THREADS + tid, nq - 1);
        qidx[r] = (uint32_t)qi;
        const uint4* src = reinterpret_cast<const uint4*>(qrows + (int64_t)qi * WORDS);
#pragma unroll
        for (int w = 0; w < WORDS / 4; ++w) {
            uint4 v = __ldg(src + w);
            q[r][4 * w + 0] = v.x;
            q[r][4 * w + 1] = v.y;
            q[r][4 * w + 2] = v.z;
            q[r][4 * w + 3] = v.w;
        }
        best[r] = 0xFFFFFFFFu;
        best2[r] = 0xFFFFFFFFu;
    }

    for (int tile = 0; tile < n_tiles; ++tile) {
        const int buf = tile & 1;
        const uint32_t phase = (tile >> 1) & 1;
        while (!mbar_try_wait(&s_bar[buf], phase)) {
        }
        const int rows = min(MT_TILE, nt - tile * MT_TILE);
        const uint32_t jbase = (uint32_t)(tile * MT_TILE);
        const uint4* trow4 = reinterpret_cast<const uint4*>(s_tile[buf]);
#pragma unroll MT_UNROLL
        for (int j = 0; j < rows; ++j) {
            uint32_t t[WORDS];
#pragma unroll
            for (int w = 0; w < WORDS / 4; ++w) {
                uint4 v = trow4[j * (WORDS / 4) + w];          // same address in every lane: broadcast
                t[4 * w + 0] = v.x;
                t[4 * w + 1] = v.y;
                t[4 * w + 2] = v.z;
                t[4 * w + 3] = v.w;
            }
            uint32_t cmin = 0xFFFFFFFFu;
            const uint32_t jj = jglob0 + jbase + j;
#pragma unroll
            for (int r = 0; r < RQ; ++r) {
                const uint32_t d = desc_dist<WORDS, NORM2>(q[r], t);
                // keys as multiply-add so that they issue on the FMA pipe (IMAD), not the ALU
                const uint32_t rk = d * (1u << EPV_KEY_SHIFT) + jj;
                if (TOP2) {
                    best2[r] = min(best2[r], max(best[r], rk));
                }
                best[r] = min(best[r], rk);
                if (!TOP2) cmin = min(cmin, d * (1u << EPV_KEY_SHIFT) + qidx[r]);
            }
            if (!TOP2) {     // column minima feed the cross-check only; the top-2 (ratio / knn) modes never read them
                cmin = __reduce_min_sync(0xFFFFFFFFu, cmin);
                if (lane == 0) s_col[buf][warp][j] = cmin;      // plain store: one slot per (warp, train row)
            }
        }
        __syncthreads();                                       // tile + its column keys are complete
        if (tid == 0 && tile + 2 < n_tiles) {
            int nrows = min(MT_TILE, nt - (tile + 2) * MT_TILE);
            uint32_t bytes = (uint32_t)nrows * WORDS * 4;
            mbar_expect_tx(&s_bar[buf], bytes);
            tma_load_1d(s_tile[buf], trows + (int64_t)(tile + 2) * MT_TILE * WORDS, bytes, &s_bar[buf]);
        }
        for (int j = tid; j < rows && !TOP2; j += MT_THREADS) {
            uint32_t m = s_col[buf][0][j];
#pragma unroll
            for (int w = 1; w < MT_THREADS / 32; ++w) m = min(m, s_col[buf][w][j]);
            atomicMin(&colkey[(int64_t)pair * stride + jbase + j], m);
        }
        // s_col[buf] is next written two tiles later, after at least one more __syncthreads
    }

#pragma unroll
    for (int r = 0; r < RQ; ++r) {
        int qi = qbase + r * MT_THREADS + tid;
        if (qi < nq) {
            rowkey[(int64_t)pair * stride + qi] = best[r];
            if (TOP2) rowkey2[(int64_t)pair * stride + qi] = best2[r];
        }
    }
}

__global__ void fill_u32_kernel(uint32_t* p, int64_t n, uint32_t v) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// Per pair: apply the match mode, compact in query order (BFMatcher output order), and
// optionally gather the matched keypoints (reference kitti_ba.cpp:684-693) and
// K-normalise them for the essential-matrix stage.
__global__ void __launch_bounds__(256) match_finalize_kernel(FinalizePlan fp) {
    __shared__ int s_warp[8];
    __shared__ int s_base;
    const int pair = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t o = (int64_t)pair * fp.stride;
    int64_t qrow0 = fp.q0 + (int64_t)pair * fp.qs, trow0 = fp.t0 + (int64_t)pair * fp.ts;   // keypoint rows of the pair
    if (fp.fq) {
        const int f0 = fp.fq[pair], f1 = fp.ft[pair];
        fp.nq = fp.counts[f0];
        fp.nt = fp.counts[f1];
        qrow0 = (int64_t)f0 * fp.qs;
        trow0 = (int64_t)f1 * fp.ts;
    }
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int start = 0; start < fp.nq; start += 256) {
        int qi = start + tid;
        bool keep = false;
        uint32_t rk = 0xFFFFFFFFu, rk2 = 0xFFFFFFFFu;
        if (qi < fp.nq && fp.nt > 0) {
            const int64_t part = (int64_t)fp.n_pairs * fp.stride;
            const bool top2 = fp.mode == EPIVO_MATCH_RATIO;
            for (int s = 0; s < fp.tsplits; ++s) {           // merge the train-split partial minima
                uint32_t a = fp.rowkey[s * part + o + qi];
                rk2 = min(rk2, max(rk, a));
                rk = min(rk, a);
                if (top2) rk2 = min(rk2, fp.rowkey2[s * part + o + qi]);
            }
            uint32_t t = rk & EPV_IDX_MASK;
            if (fp.mode == EPIVO_MATCH_NN) {
                keep = true;
            } else if (fp.mode == EPIVO_MATCH_CROSSCHECK) {
                keep = (fp.colkey[o + t] & EPV_IDX_MASK) == (uint32_t)qi;
            } else {
                keep = fp.nt >= 2 &&
                       (float)(rk >> EPV_KEY_SHIFT) < fp.ratio * (float)(rk2 >> EPV_KEY_SHIFT);
            }
        }
        unsigned bal = __ballot_sync(0xFFFFFFFFu, keep);
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        int off = s_base;
        for (int w = 0; w < warp; ++w) off += s_warp[w];
        int k = off + __popc(bal & ((1u << lane) - 1));
        if (keep) {
            int t = (int)(rk & EPV_IDX_MASK);
            if (fp.mq) fp.mq[o + k] = qi;
            if (fp.mt) fp.mt[o + k] = t;
            if (fp.md) fp.md[o + k] = (int)(rk >> EPV_KEY_SHIFT);
            if (fp.md2 && fp.mode == EPIVO_MATCH_RATIO) fp.md2[o + k] = (int)(rk2 >> EPV_KEY_SHIFT);
            if (fp.kps) {
                const float2 a = reinterpret_cast<const float2*>(fp.kps)[qrow0 + qi];
                const float2 b = reinterpret_cast<const float2*>(fp.kps)[trow0 + t];
                if (fp.p0) {
                    reinterpret_cast<float2*>(fp.p0)[o + k] = a;
                    reinterpret_cast<float2*>(fp.p1)[o + k] = b;
                }
                if (fp.xn) {
                    double* x = fp.xn + (int64_t)pair * 4 * fp.stride;
                    x[k] = __fma_rn((double)a.x, fp.ax, fp.bx);
                    x[fp.stride + k] = __fma_rn((double)a.y, fp.ay, fp.by);
                    x[2 * fp.stride + k] = __fma_rn((double)b.x, fp.ax, fp.bx);
                    x[3 * fp.stride + k] = __fma_rn((double)b.y, fp.ay, fp.by);
                }
            }
        }
        __syncthreads();
        if (tid == 0) {
            int tot = 0;
            for (int w = 0; w < 8; ++w) tot += s_warp[w];
            s_base += tot;
        }
        __syncthreads();
    }
    if (tid == 0) fp.n_matches[pair] = s_base;
}

// query rows per thread for a set of nq descriptors: fewest row slots over the CTAs, ties to the larger block
inline int mt_pick_rq(int nq, int words) {
    if (words != 8) return MT_RQ;                       // the smaller block is instantiated for 32-byte descriptors only
    auto slots = [nq](int rq) { return (nq + MT_THREADS * rq - 1) / (MT_THREADS * rq) * rq; };
    return slots(6) < slots(MT_RQ) ? 6 : MT_RQ;
}

template <int WORDS, int RQ>
int launch_words(epivo_ctx* ctx, const MatchPlan& mp, const uint32_t* src) {
    const int n_tiles = std::max(1, (mp.nt + MT_TILE - 1) / MT_TILE);
    const int tps = (n_tiles + mp.tsplits - 1) / mp.tsplits;
    dim3 grid((mp.nq + MT_THREADS * RQ - 1) / (MT_THREADS * RQ), mp.n_pairs, (n_tiles + tps - 1) / tps);
    const int64_t part = (int64_t)mp.n_pairs * mp.stride;
    dim3 block(MT_THREADS);
    const bool n2 = mp.norm == EPIVO_NORM_HAMMING2;
#define EPV_MT(N2, T2, CN)                                                                                 \
    do {                                                                                                   \
        match_tile_kernel<WORDS, RQ, N2, T2, CN><<<grid, block, 0, ctx->stream>>>(                         \
            src, mp.q0, mp.qs, mp.t0, mp.ts, mp.nq, mp.nt, mp.rowkey, mp.rowkey2, mp.colkey, mp.stride, tps, part, \
            mp.fq, mp.ft, mp.counts);                                                                      \
    } while (0)
#define EPV_MT2(N2, T2)                     \
    do {                                    \
        if (mp.fq) EPV_MT(N2, T2, true);    \
        else EPV_MT(N2, T2, false);         \
    } while (0)
    if (n2 && mp.top2) EPV_MT2(true, true);
    else if (n2) EPV_MT2(true, false);
    else if (mp.top2) EPV_MT2(false, true);
    else EPV_MT2(false, false);
#undef EPV_MT2
#undef EPV_MT
    EPV_LAUNCHED(ctx);
    return EPIVO_OK;
}

}  // namespace

int epv_match_splits(const epivo_ctx* ctx, int n_pairs, int nq, int nt) {
    const int rq = mt_pick_rq(nq, 8);
    const int64_t qblocks = (nq + MT_THREADS * rq - 1) / (MT_THREADS * rq);
    const int n_tiles = (nt + MT_TILE - 1) / MT_TILE;
    if (n_tiles <= 1) return 1;
    const int64_t ctas = std::max<int64_t>(1, qblocks * n_pairs);
    const int64_t want = 4LL * ctx->sm_count;             // ~4 CTAs per SM
    int64_t s = (want + ctas - 1) / ctas;
    s = std::max<int64_t>(1, std::min<int64_t>(s, std::max(1, n_tiles / 2)));
    const int64_t tps = (n_tiles + s - 1) / s;            // tiles per split
    return (int)std::max<int64_t>(1, (n_tiles + tps - 1) / tps);   // splits actually launched (no empty part)
}

// frame pairs whose matcher CTAs fill the GPU exactly once (one "wave"): launches sized in whole
// waves lose nothing to a partially filled last wave
int epv_match_pairs_per_wave(const epivo_ctx* ctx, int nq) {
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, match_tile_kernel<8, MT_RQ, true, false, false>, MT_THREADS, 0) != cudaSuccess ||
        occ < 1)
        occ = 2;
    const int rq = mt_pick_rq(nq, 8);
    const int qblocks = std::max(1, (nq + MT_THREADS * rq - 1) / (MT_THREADS * rq));
    return std::max(1, ctx->sm_count * occ / qblocks);
}

int epv_match_launch(epivo_ctx* ctx, const MatchPlan& mp, bool run_prepass) {
    if (mp.tsplits < 1) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "tsplits < 1");
    if (mp.words != 4 && mp.words != 8 && mp.words != 16)
        EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "descriptor size %d bytes unsupported (16, 32 or 64)", mp.words * 4);
    if (mp.norm != EPIVO_NORM_HAMMING && mp.norm != EPIVO_NORM_HAMMING2)
        EPV_FAIL(ctx, EPIVO_ERR_INVALID, "norm %d is not NORM_HAMMING(6) / NORM_HAMMING2(7)", mp.norm);
    if (mp.nq > (int)EPV_IDX_MASK || mp.nt > (int)EPV_IDX_MASK)
        EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "more than %u descriptors per set", EPV_IDX_MASK);
    if (mp.n_pairs <= 0 || mp.nq <= 0) return EPIVO_OK;
    const uint32_t* src = mp.desc;
    if (mp.norm == EPIVO_NORM_HAMMING2) {
        if (run_prepass) {
            int64_t n = mp.total_rows * (mp.words / 2);
            const int64_t off = mp.prepass_row0 * mp.words;
            desc_planes_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(mp.desc + off, mp.planes + off,
                                                                                     mp.total_rows, mp.words);
            EPV_LAUNCHED(ctx);
        }
        src = mp.planes;
    }
    int64_t nkeys = (int64_t)mp.n_pairs * mp.stride;
    fill_u32_kernel<<<(unsigned)((nkeys + 255) / 256), 256, 0, ctx->stream>>>(mp.colkey, nkeys, 0xFFFFFFFFu);
    EPV_LAUNCHED(ctx);
    if (mp.nt <= 0) return EPIVO_OK;
    if (mp.ev0) EPV_CUDA(ctx, cudaEventRecord(mp.ev0, ctx->stream));
    int rc;
    switch (mp.words) {
        case 4: rc = launch_words<4, MT_RQ>(ctx, mp, src); break;
        case 8: rc = mt_pick_rq(mp.nq, 8) == 6 ? launch_words<8, 6>(ctx, mp, src) : launch_words<8, MT_RQ>(ctx, mp, src); break;
        default: rc = launch_words<16, MT_RQ>(ctx, mp, src); break;
    }
    if (rc) return rc;
    if (mp.ev1) EPV_CUDA(ctx, cudaEventRecord(mp.ev1, ctx->stream));
    return EPIVO_OK;
}

// The NORM_HAMMING2 plane pre-pass alone, on a stream of the caller's choice (the host-buffer path converts every
// upload piece on the copy stream, right behind its cudaMemcpyAsync).
int epv_planes_launch(epivo_ctx* ctx, const uint32_t* desc, uint32_t* planes, int64_t rows, int words, cudaStream_t st) {
    if (rows <= 0) return EPIVO_OK;
    const int64_t n = rows * (words / 2);
    desc_planes_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(desc, planes, rows, words);
    EPV_LAUNCHED(ctx);
    return EPIVO_OK;
}

int epv_finalize_launch(epivo_ctx* ctx, const FinalizePlan& fp) {
    if (fp.n_pairs <= 0) return EPIVO_OK;
    match_finalize_kernel<<<fp.n_pairs, 256, 0, ctx->stream>>>(fp);
    EPV_LAUNCHED(ctx);
    return EPIVO_OK;
}
