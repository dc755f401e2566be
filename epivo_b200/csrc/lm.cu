// K5: the reference's SE(3)-chain Levenberg-Marquardt (jac_Rt_gen_.cpp:287-478), one CTA per
// problem, every iteration on the device (no host round trips).
//
// Per iteration (reference line numbers in brackets):
//   chain memo  mem[a][b] = T[b] ... T[a]  and its inverses                     [:328-335]
//   weighted residuals r = w * res(T_rep, p, p')                                 [:338-360, :212-259]
//   Jacobian rows wrt every zeta in each rep's span, Dr_Deps as written          [:363-399, :23-209]
//     (closed form: the 6 generator columns are constant; only non-zero blocks are formed)
//   H = J'J, b = J'r accumulated tile by tile in shared memory                   [:401-402]
//   H += lambda diag(H);  delta = -H^-1 b  by LU with partial pivoting           [:403-405]
//   stop on NaN or |delta| < eps                                                 [:407-414]
//   T'_k = T_k exp(delta_k)  (Sophus SE3::exp, right-multiplied)                 [:416-422]
//   candidate chains by explicit products, UNWEIGHTED candidate residual norm    [:425-456]
//   accept if smaller: lambda /= 2, else lambda *= 5                             [:457-467]
// Reference quirks kept on purpose: the Jacobian's Huber branch switches on e'e <= delta
// while res switches on e'e/2 > delta (sqrt(2) mismatch at delta = 1e-5); reverse reps
// differentiate a LEFT perturbation of the zeta although the update is right-multiplied.
#include <cooperative_groups.h>

#include "common.cuh"
#include "stages.cuh"

namespace cg = cooperative_groups;

namespace {

// The window kernel is instantiated for six CTA shapes <threads, points per Jacobian tile, cluster>; the launcher picks
// one by problem size (measured on B200: small windows want many small CTAs, large ones wider CTAs).
// Chain length: the reference's bound is rep_max = 128 (jac_Rt_gen_.cpp:18, the size of its memo array); its drivers
// and demo use 4..10 zetas.  Here a window lives in shared memory -- chain memo and inverses 2 nz^2 x 96 B, H | b
// (6 nz)(6 nz + 1) x 8 B, one Jacobian tile -- which fits for n_zeta <= 18 (the smallest tile shape is chosen
// automatically when the preferred one does not fit); longer chains are refused with EPIVO_ERR_UNSUPPORTED.
constexpr int LM_MAX_ZETA = 128;
constexpr size_t LM_SMEM_LIMIT = 220 * 1024;

struct Rt { double R[9]; double t[3]; };

__device__ __forceinline__ void rt_identity(Rt& o) {
#pragma unroll
    for (int i = 0; i < 9; ++i) o.R[i] = (i % 4 == 0) ? 1.0 : 0.0;
    o.t[0] = o.t[1] = o.t[2] = 0.0;
}
// o = a * b   (4x4 with last row 0 0 0 1)
__device__ __forceinline__ void rt_mul(const Rt& a, const Rt& b, Rt& o) {
    Rt r;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j) r.R[i * 3 + j] = a.R[i * 3] * b.R[j] + a.R[i * 3 + 1] * b.R[3 + j] + a.R[i * 3 + 2] * b.R[6 + j];
        r.t[i] = a.R[i * 3] * b.t[0] + a.R[i * 3 + 1] * b.t[1] + a.R[i * 3 + 2] * b.t[2] + a.t[i];
    }
    o = r;
}
// general inverse of [A t; 0 1] (the reference calls MatrixXd::inverse(), not a rigid inverse)
__device__ __forceinline__ void rt_inv(const Rt& a, Rt& o) {
    const double* m = a.R;
    const double c00 = m[4] * m[8] - m[5] * m[7], c01 = m[5] * m[6] - m[3] * m[8], c02 = m[3] * m[7] - m[4] * m[6];
    const double det = m[0] * c00 + m[1] * c01 + m[2] * c02;
    const double id = 1.0 / det;
    Rt r;
    r.R[0] = c00 * id; r.R[1] = (m[2] * m[7] - m[1] * m[8]) * id; r.R[2] = (m[1] * m[5] - m[2] * m[4]) * id;
    r.R[3] = c01 * id; r.R[4] = (m[0] * m[8] - m[2] * m[6]) * id; r.R[5] = (m[2] * m[3] - m[0] * m[5]) * id;
    r.R[6] = c02 * id; r.R[7] = (m[1] * m[6] - m[0] * m[7]) * id; r.R[8] = (m[0] * m[4] - m[1] * m[3]) * id;
#pragma unroll
    for (int i = 0; i < 3; ++i) r.t[i] = -(r.R[i * 3] * a.t[0] + r.R[i * 3 + 1] * a.t[1] + r.R[i * 3 + 2] * a.t[2]);
    o = r;
}

// Arithmetic note.  FP64 division and square root cost ~20 dependent instructions each on the
// GPU and the reference's formulas are full of them (||A||/||B||, X/X_z, .../||B||^2 per Jacobian
// column).  The functions below compute the same quantities from one reciprocal square root per
// norm and one reciprocal per depth; results differ from the literal formulas in the last bits
// only (the parity tolerance for the LM is relative 1e-5, tests/test_gpu_pose_lm.py).

// Sophus::SE3<double>::exp(delta), delta = (upsilon, omega)                         [:419]
__device__ __forceinline__ void se3_exp(const double* d, Rt& o) {
    const double wx = d[3], wy = d[4], wz = d[5];
    const double th2 = wx * wx + wy * wy + wz * wz;
    const double th = sqrt(th2);
    double a, b, c;   // R = I + a Om + b Om^2 ; V = I + b Om + c Om^2
    if (th < 1e-10) {
        a = 1.0; b = 0.5; c = 1.0 / 6.0;
    } else {
        double sn, cs;
        sincos(th, &sn, &cs);
        const double ith = 1.0 / th, ith2 = ith * ith;
        a = sn * ith;
        b = (1.0 - cs) * ith2;
        c = (th - sn) * (ith2 * ith);
    }
    const double Om[9] = {0, -wz, wy, wz, 0, -wx, -wy, wx, 0};
    double Om2[9];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) Om2[i * 3 + j] = Om[i * 3] * Om[j] + Om[i * 3 + 1] * Om[3 + j] + Om[i * 3 + 2] * Om[6 + j];
    double V[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) {
        const double I = (i % 4 == 0) ? 1.0 : 0.0;
        o.R[i] = I + a * Om[i] + b * Om2[i];
        V[i] = (th < 1e-10) ? o.R[i] : I + b * Om[i] + c * Om2[i];    // Sophus: V = so3.matrix() below epsilon
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) o.t[i] = V[i * 3] * d[0] + V[i * 3 + 1] * d[1] + V[i * 3 + 2] * d[2];
}

// res() for one correspondence                                                     [:230-258]
__device__ __forceinline__ double res_one(const Rt& T, const double* p, const double* p_, double hd) {
    const double px = -p_[0], py = -p_[1];
    const double A0 = T.t[0] + px * T.t[2], A1 = T.t[1] + py * T.t[2];
    const double q0 = T.R[0] * p[0] + T.R[1] * p[1] + T.R[2] * p[2];
    const double q1 = T.R[3] * p[0] + T.R[4] * p[1] + T.R[5] * p[2];
    const double q2 = T.R[6] * p[0] + T.R[7] * p[1] + T.R[8] * p[2];
    const double B0 = q0 + px * q2, B1 = q1 + py * q2;
    const double ATA = A0 * A0 + A1 * A1, BTB = B0 * B0 + B1 * B1;
    double d = 0.0;                                                                  // ||A|| / ||B||, 0 if ||B|| = 0
    if (BTB > 0) d = (ATA > 0) ? (ATA * rsqrt(ATA)) * rsqrt(BTB) : 0.0;
    const double X0 = q0 * d + T.t[0], X1 = q1 * d + T.t[1], X2 = q2 * d + T.t[2];
    const double iz = 1.0 / X2;
    const double e0 = p_[0] - X0 * iz, e1 = p_[1] - X1 * iz, e2 = p_[2] - X2 * iz;
    double r = (e0 * e0 + e1 * e1 + e2 * e2) * 0.5;
    if (r > hd) r = hd * (sqrt(r) - hd * 0.5);
    return r;
}

// Dr_Deps [:109-208] in two parts.  With M_j = s Tl G_j Tr (G_j the se(3) generators, translations first) the
// reference forms, per correspondence and per column j,
//     dA_j = P M_j[:3,3],  dB_j = P M_j[:3,:3] p,  jd_j = (|B|/|A| A.dA_j - |A|/|B| B.dB_j) / |B|^2            [:162]
//     dX_j = M_j [p d0; 1] + R0 p jd_j,   row_j = g' J_pi dX_j                                                 [:171-207]
// (g = e or delta e/|e|, the Huber switch of [:203-207]).  Everything is linear in M_j, and
//     M_j[:3,3] = Tl.R e_j (j < 3),   Tl.R (e_k x h) (j = 3 + k),      M_j[:3,:3] p = 0,   Tl.R (e_k x u)
// with u = Tr.R p, h = Tr.t.  Writing w' = g' J_pi (1 x 3), a3 = P'A, b3 = P'B (so that A.dA = a3.M[:3,3] and
// B.dB = b3.(M[:3,:3] p)), cq = w.q with q = R0 p, the row collapses to
//     z1 = w + cq (|B|/|A|)/|B|^2 a3,      z2 = d0 w - cq (|A|/|B|)/|B|^2 b3          (per correspondence, rep-wide)
//     t1 = Tl.R' z1,  t2 = Tl.R' z2,       row = s [ t1 | u x t2 + h x t1 ]             (per zeta: 39 multiply-adds)
// -- the same numbers as the literal formulas up to rounding (1e-12 relative, checked against the restatement of
// the reference over forward and reverse reps), for a fifth of the arithmetic.  Everything that depends only on
// the correspondence and on the rep's full transform T0 = Tl Tr (the same for every zeta of the span) is computed
// once per point:
struct JacCommon {
    double z1[3], z2[3];
    double res;          // res() of the same correspondence under T0 [:230-258]
    bool degenerate;     // |A| == 0 or |B| == 0: the row stays zero [:152-154]
};

__device__ __forceinline__ void jac_common(const Rt& T0, const double* p, const double* p_, double hd, JacCommon& c) {
    const double px = -p_[0], py = -p_[1];
    const double A0 = T0.t[0] + px * T0.t[2], A1 = T0.t[1] + py * T0.t[2];
    const double q0 = T0.R[0] * p[0] + T0.R[1] * p[1] + T0.R[2] * p[2];
    const double q1 = T0.R[3] * p[0] + T0.R[4] * p[1] + T0.R[5] * p[2];
    const double q2 = T0.R[6] * p[0] + T0.R[7] * p[1] + T0.R[8] * p[2];
    const double B0 = q0 + px * q2, B1 = q1 + py * q2;
    const double ATA = A0 * A0 + A1 * A1, BTB = B0 * B0 + B1 * B1;
    c.degenerate = (ATA == 0 || BTB == 0);
    const double isa = c.degenerate ? 0.0 : rsqrt(ATA), isb = c.degenerate ? 0.0 : rsqrt(BTB);
    const double sa = ATA * isa, sb = BTB * isb;                                     // ||A||, ||B||
    const double d0 = (BTB > 0) ? sa * isb : 0.0;                                    // res(): d = 0 when ||B|| = 0
    const double iBTB = isb * isb;
    const double X0 = q0 * d0 + T0.t[0], X1 = q1 * d0 + T0.t[1], X2 = q2 * d0 + T0.t[2];
    const double iz = 1.0 / X2;
    {
        const double f0 = p_[0] - X0 * iz, f1 = p_[1] - X1 * iz, f2 = p_[2] - X2 * iz;
        double r = (f0 * f0 + f1 * f1 + f2 * f2) * 0.5;
        if (r > hd) r = hd * (sqrt(r) - hd * 0.5);
        c.res = r;
    }
    const double e0 = X0 * iz - p_[0];
    const double e1 = X1 * iz - p_[1];
    const double e2 = 1.0 - p_[2];
    const double ee = e0 * e0 + e1 * e1 + e2 * e2;
    double g0 = e0, g1 = e1;                                                        // [:203-207]
    if (!(ee <= hd)) {
        const double k = hd * rsqrt(ee);
        g0 *= k;
        g1 *= k;
    }
    // w' = g' J_pi, J_pi = [[1/z, 0, -x/z^2], [0, 1/z, -y/z^2], [0, 0, 0]] (all zero when z = 0) [:184-186]
    const double jz = (X2 != 0) ? iz : 0.0;
    const double w0 = g0 * jz, w1 = g1 * jz, w2 = -(g0 * X0 + g1 * X1) * (jz * jz);
    const double cq = w0 * q0 + w1 * q1 + w2 * q2;
    const double ca = cq * (isa * sb) * iBTB, cb = cq * (isb * sa) * iBTB;           // cq |B|/|A| / |B|^2, cq |A|/|B| / |B|^2
    c.z1[0] = w0 + ca * A0;
    c.z1[1] = w1 + ca * A1;
    c.z1[2] = w2 + ca * (px * A0 + py * A1);
    c.z2[0] = d0 * w0 - cb * B0;
    c.z2[1] = d0 * w1 - cb * B1;
    c.z2[2] = d0 * w2 - cb * (px * B0 + py * B1);
}

// ... and the six columns of one zeta: d r / d eps for T = Tl exp(eps) Tr (sign s for reverse reps)
__device__ __forceinline__ void jac_zeta(const JacCommon& c, const Rt& Tl, const Rt& Tr, double s, const double* p,
                                         double* row) {
    if (c.degenerate) {
#pragma unroll
        for (int j = 0; j < 6; ++j) row[j] = 0.0;
        return;
    }
    const double u0 = Tr.R[0] * p[0] + Tr.R[1] * p[1] + Tr.R[2] * p[2];
    const double u1 = Tr.R[3] * p[0] + Tr.R[4] * p[1] + Tr.R[5] * p[2];
    const double u2 = Tr.R[6] * p[0] + Tr.R[7] * p[1] + Tr.R[8] * p[2];
    double t1[3], t2[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {                                                   // Tl.R' z
        t1[k] = s * (Tl.R[k] * c.z1[0] + Tl.R[3 + k] * c.z1[1] + Tl.R[6 + k] * c.z1[2]);
        t2[k] = s * (Tl.R[k] * c.z2[0] + Tl.R[3 + k] * c.z2[1] + Tl.R[6 + k] * c.z2[2]);
    }
    const double h0 = Tr.t[0], h1 = Tr.t[1], h2 = Tr.t[2];
    row[0] = t1[0];
    row[1] = t1[1];
    row[2] = t1[2];
    row[3] = (u1 * t2[2] - u2 * t2[1]) + (h1 * t1[2] - h2 * t1[1]);
    row[4] = (u2 * t2[0] - u0 * t2[2]) + (h2 * t1[0] - h0 * t1[2]);
    row[5] = (u0 * t2[1] - u1 * t2[0]) + (h0 * t1[1] - h1 * t1[0]);
}

// One row of Dr_Deps plus (optionally) the residual at the same transform: the single-pair kernel's form.
__device__ __forceinline__ void jac_row(const Rt& Tl, const Rt& Tr, const Rt& T0, double s, const double* p,
                                        const double* p_, double hd, double* row, double* res = nullptr) {
    JacCommon c;
    jac_common(T0, p, p_, hd, c);
    if (res) *res = c.res;
    jac_zeta(c, Tl, Tr, s, p, row);
}

struct LmArgs {
    LmPlan p;
    int D;
    size_t smem_doubles;
};

__device__ __forceinline__ double lm_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

// Damped normal equations H delta = -b on the augmented D x (D + 1) matrix in shared memory: LU with partial
// pivoting [:405] and back substitution by NW warps (one per SM sub-partition) that meet at a NAMED barrier, not at
// the block barrier.  A pivot step on 60..96 unknowns is a few thousand multiply-adds behind a chain of dependent
// latencies (pivot -> reciprocal -> row factor -> update -> next pivot); the block-wide version paid three block
// barriers and a separate pivot search for it (3600 cycles per step).  Here
//  * warp w updates the rows k + 1 + w, k + 1 + w + NW, ...; lane l owns columns k + 1 + l + 32 i (i < NC) and keeps
//    the pivot row in registers; rows are updated RB at a time, every load of a batch issued before its first store
//    (row by row the compiler must assume that a store aliases the next row's loads and serialises them);
//  * lane 0 of a warp owns column k + 1, i.e. it produces that warp's candidates for the NEXT pivot: it keeps the
//    first largest |value| as it goes (compared as integers: for non-negative doubles the bit patterns order like
//    the values; NaN never wins, as in a sequential `>` search) and posts it; after the barrier every warp picks
//    the winner of the NW posts itself (largest, then lowest row), so the separate search disappears;
//  * two named barriers per step (after the row swap, after the update); warps outside the solve wait at the
//    block barrier that follows.
// Returns through sDelta; *stop is set on NaN or |delta| < eps [:407-414].
template <int NW>
__device__ __forceinline__ void lm_solve_bar() {
    if (NW > 1) asm volatile("bar.sync 1, %0;" ::"n"(NW * 32) : "memory");
    else __syncwarp();
}

template <int NC, int RB, int NW>
__device__ __noinline__ void lm_warp_solve(double* sH, double* sDelta, int D, int tid, double epsilon, int* stop,
                                           long long* sKey, int* sRow) {
    const int lane = tid & 31, w = tid >> 5, W1 = D + 1;
    // pivot of column 0: every warp searches the whole column itself (first row with the largest |value|)
    double best = -1.0;
    int pv = 0;
    for (int r = lane; r < D; r += 32) {
        const double v = fabs(sH[(size_t)r * W1]);
        if (v > best) { best = v; pv = r; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ob = __shfl_xor_sync(0xFFFFFFFFu, best, o);
        const int op = __shfl_xor_sync(0xFFFFFFFFu, pv, o);
        if (ob > best || (ob == best && op < pv)) { best = ob; pv = op; }
    }
    lm_solve_bar<NW>();                              // nobody swaps before everybody has searched
    for (int k = 0; k < D; ++k) {
        if (pv != k) {                               // row swap: one column per thread (D + 1 <= 32 NC <= 32 NW NC)
            for (int c = k + tid; c <= D; c += 32 * NW) {
                const double t = sH[(size_t)k * W1 + c];
                sH[(size_t)k * W1 + c] = sH[(size_t)pv * W1 + c];
                sH[(size_t)pv * W1 + c] = t;
            }
        }
        lm_solve_bar<NW>();
        const double* prw = sH + (size_t)k * W1;
        const double ipiv = 1.0 / prw[k];
        double prow[NC];
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            const int c = k + 1 + lane + 32 * i;
            prow[i] = (c <= D) ? prw[c] : 0.0;
        }
        long long nkey = -1;                         // lane 0: bit pattern of the largest |value| of column k + 1 so far
        int npv = D;
        for (int r0 = k + 1 + w; r0 < D; r0 += RB * NW) {
            double f[RB], v[RB][NC];
#pragma unroll
            for (int j = 0; j < RB; ++j) {
                const double* row = sH + (size_t)min(r0 + j * NW, D - 1) * W1;     // clamped rows are loaded, never stored
                f[j] = row[k];
#pragma unroll
                for (int i = 0; i < NC; ++i) {
                    const int c = k + 1 + lane + 32 * i;
                    v[j][i] = (c <= D) ? row[c] : 0.0;
                }
            }
#pragma unroll
            for (int j = 0; j < RB; ++j) {
                f[j] *= ipiv;
#pragma unroll
                for (int i = 0; i < NC; ++i) v[j][i] -= f[j] * prow[i];
            }
#pragma unroll
            for (int j = 0; j < RB; ++j) {
                const int r = r0 + j * NW;
                if (r < D) {
                    double* row = sH + (size_t)r * W1;
#pragma unroll
                    for (int i = 0; i < NC; ++i) {
                        const int c = k + 1 + lane + 32 * i;
                        if (c <= D) row[c] = v[j][i];
                    }
                    long long key = __double_as_longlong(v[j][0]) & 0x7FFFFFFFFFFFFFFFLL;
                    if (key > 0x7FF0000000000000LL) key = -1;          // NaN
                    if (key > nkey) { nkey = key; npv = r; }           // rows ascend within a warp: first maximum
                }
            }
        }
        if (lane == 0) { sKey[w] = nkey; sRow[w] = npv; }
        lm_solve_bar<NW>();
        long long bk = sKey[0];
        pv = sRow[0];
#pragma unroll
        for (int q = 1; q < NW; ++q) {
            const long long kq = sKey[q];
            const int rq = sRow[q];
            if (kq > bk || (kq == bk && rq < pv)) { bk = kq; pv = rq; }
        }
        if (bk < 0) pv = k + 1;                       // nothing comparable (all NaN, or no rows left): keep the diagonal
    }
    if (w != 0) return;
    // back substitution, column oriented, by warp 0: lane l keeps y_r of rows r = l + 32 i in registers; for
    // c = D-1 .. 0 the owner forms delta_c = y_c / U_cc, broadcasts it, and every lane updates its rows above c
    double y[NC], dgl[NC];
#pragma unroll
    for (int i = 0; i < NC; ++i) {
        const int r = lane + 32 * i;
        y[i] = (r < D) ? sH[(size_t)r * W1 + D] : 0.0;
        dgl[i] = (r < D) ? sH[(size_t)r * W1 + r] : 1.0;
    }
    bool nan = false;
    double nrm = 0.0;
    for (int c = D - 1; c >= 0; --c) {
        double yc = 0.0, dg = 1.0;
#pragma unroll
        for (int i = 0; i < NC; ++i)
            if ((c >> 5) == i) { yc = y[i]; dg = dgl[i]; }
        double col[NC];                              // column c above the diagonal: loaded while the division runs
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            const int r = lane + 32 * i;
            col[i] = (r < c) ? sH[(size_t)r * W1 + c] : 0.0;
        }
        double dc = yc / dg;                         // every lane divides its own candidate; the owner's is taken
        dc = __shfl_sync(0xFFFFFFFFu, dc, c & 31);
        if (lane == 0) sDelta[c] = dc;
        nan |= !(dc == dc);                          // hasNaN(): NaN only, an inf passes (as in the reference)
        nrm += dc * dc;
#pragma unroll
        for (int i = 0; i < NC; ++i) y[i] -= col[i] * dc;
    }
    if (lane == 0 && (nan || sqrt(nrm) < epsilon)) *stop = 1;                      // [:407-414]
}

// ---- Gram tiles on the FP64 tensor cores -------------------------------------------------------------------------
// H = J'J is the one dense contraction of this path (a SYRK: per rep and tile, (W+1) x np times np x (W+1), W = 6 x span
// columns plus the residual column, which yields b = J'r for free).  As scalar FMAs on a shared-memory tile it is
// bound by shared-memory bandwidth, not by the FP64 pipe: a 4 x 4 register block issues 8 LDS.64 per 16 DFMA.  The
// warp-wide mma.sync.m8n8k4.f64 (DMMA; measured on B200 at the same 18.5 T FMA/s as scalar DFMA, epivo_microbench 5)
// takes ONE double per lane for each operand and does 256 multiply-adds: an 8 x 8 block of the Gram matrix over 4
// correspondences.  The tile is stored TRANSPOSED, sJ[column][point]: consecutive lanes own consecutive points when
// the Jacobian is written (conflict-free stores), and a fragment load reads 8 columns x 4 points; with a column
// stride of 4 mod 16 doubles the 16 lanes of a half-warp hit 16 different bank pairs.
__host__ __device__ inline int lm_tile_stride(int tp) {      // doubles between the columns of a tile of tp points
    int ts = (tp + 3) & ~3;
    while (ts % 16 != 4) ts += 4;
    return ts;
}
__host__ __device__ inline int lm_tile_cols(int D) { return (D + 1 + 7) / 8 * 8; }   // columns incl. residual, padded to 8

__device__ __forceinline__ void dmma_m8n8k4(double (&c)[2], double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}
// block index of the upper triangle (row-major: row bi holds NB - bi blocks) -> (bi, bj)
__device__ __forceinline__ void lm_block_of(int blk, int NB, int& bi, int& bj) {
    int r = 0;
    while (blk >= NB - r) { blk -= NB - r; ++r; }
    bi = r;
    bj = r + blk;
}
// element e (0 / 1) of this lane's accumulator fragment of block (bi, bj) -> H | b of the window
__device__ __forceinline__ void lm_gram_store(double* sAcc, int D, int lo, int W, int bi, int bj, int lane, int e, double v) {
    const int u = 8 * bi + (lane >> 2), c = 8 * bj + 2 * (lane & 3) + e;
    if (u < W && c >= u && c <= W) {                // upper triangle of H; column W is the residual: b = J'r
        const int gr = 6 * lo + u;
        sAcc[(size_t)gr * (D + 1) + (c == W ? D : 6 * lo + c)] += v;
    }
}

// CL > 1: a window is shared by a thread-block CLUSTER of CL CTAs (launched with a cluster dimension of CL).  Each
// CTA builds the Jacobian / Gram tiles t with t % CL == rank into its own partial H | b; after one cluster barrier
// every CTA sums the CL partials straight out of the peers' shared memory (DSMEM) in rank order, so all of them hold
// the same H | b bit for bit and run the (cheap, latency-bound) damped solve redundantly -- no broadcast of delta is
// needed and every CTA takes the same stop / accept decisions.  The candidate residual is split the same way.  Used
// when the batch is too small to fill the GPU with one CTA per window (a multi-GPU shard of cfg5).
template <int LM_THREADS, int LM_TP, int CL>
__global__ void __launch_bounds__(LM_THREADS) lm_kernel(LmArgs a) {
    extern __shared__ __align__(16) double sm[];
    const LmPlan& p = a.p;
    const int nz = p.n_zeta, nr = p.n_rep, N = p.N, D = a.D;
    const int tid = threadIdx.x, prob = blockIdx.x / CL;
    int crank = 0;
    if (CL > 1) crank = (int)cg::this_cluster().block_rank();
    if (p.active && !p.active[prob]) return;          // the whole cluster leaves together
    // shared layout
    Rt* sT = reinterpret_cast<Rt*>(sm);            // [nz] current
    Rt* sTn = sT + nz;                             // [nz] candidate
    Rt* sMem = sTn + nz;                           // [nz*nz] chain memo
    Rt* sInv = sMem + nz * nz;                     // [nz*nz] inverses
    Rt* sRep = sInv + nz * nz;                     // [nr] per-rep transform
    double* sH = reinterpret_cast<double*>(sRep + nr);   // [D][D+1] augmented
    const int TS = lm_tile_stride(LM_TP);          // tile column stride (see "Gram tiles" above)
    double* sJ = sH + (size_t)D * (D + 1);         // [lm_tile_cols(D)][TS] transposed tile: J columns of the span + residual
    double* sDelta = sJ + (size_t)lm_tile_cols(D) * TS;   // [D]
    double* sRed = sDelta + D;                     // [LM_THREADS]
    double* sScr = sRed + LM_THREADS;              // [LM_THREADS / 32][64] partial Gram fragments of a k-split
    double* sHp = sScr + 2 * LM_THREADS;           // [D][D+1] this CTA's partial H | b (CL > 1 only)
    double* sAcc = (CL > 1) ? sHp : sH;            // where the Gram blocks are accumulated
    __shared__ double s_part[2];                   // this CTA's partial sums of squares (r0, candidate)
    __shared__ long long s_key[4];                 // solver warps: next-pivot candidates
    __shared__ int s_row[4];
    __shared__ double s_lambda, s_prevE, s_Hnorm, s_rnorm;
    __shared__ int s_stop, s_iters, s_piv;
    __shared__ Rt s_identity;

    double* gT = p.T0s + (size_t)prob * nz * 16;
    const double* gpr = p.pr + (size_t)prob * nr * N * 3;
    const double* gp_r = p.p_r + (size_t)prob * nr * N * 3;
    const double* w = p.wreps + (size_t)prob * nr;
    const double hd = p.huber_delta;

    for (int k = tid; k < nz; k += LM_THREADS) {
        for (int i = 0; i < 3; ++i) {
            for (int j = 0; j < 3; ++j) sT[k].R[i * 3 + j] = gT[k * 16 + i * 4 + j];
            sT[k].t[i] = gT[k * 16 + i * 4 + 3];
        }
    }
    if (tid == 0) {
        rt_identity(s_identity);
        s_lambda = p.lambda0;
        s_prevE = 1e10;                                                            // [:322]
        s_stop = 0;
        s_iters = 0;
        s_Hnorm = 0.0;
        s_rnorm = 0.0;
    }
    __syncthreads();

    for (int iter = 0; iter < p.max_iters; ++iter) {
        if (tid == 0) s_iters = iter + 1;
        // ---- chain memo + inverses                                              [:328-335]
        for (int j = tid; j < nz; j += LM_THREADS) {
            Rt acc = sT[j];
            sMem[j * nz + j] = acc;
            rt_inv(acc, sInv[j * nz + j]);
            for (int k = j + 1; k < nz; ++k) {
                rt_mul(sT[k], acc, acc);
                sMem[j * nz + k] = acc;
                rt_inv(acc, sInv[j * nz + k]);
            }
        }
        for (int i = tid; i < D * (D + 1); i += LM_THREADS) sAcc[i] = 0.0;
        __syncthreads();
        for (int j = tid; j < nr; j += LM_THREADS) {                                // [:338-348]
            const int z0 = p.reps[2 * j], z1 = p.reps[2 * j + 1];
            sRep[j] = (z0 <= z1) ? sMem[z0 * nz + z1] : sInv[z1 * nz + z0];
        }
        __syncthreads();
        // ---- residuals, Jacobian tiles, H = J'J, b = J'r
        double rsq = 0.0;
        int tile_id = 0;                            // running tile counter over all reps: tile t belongs to rank t % CL
        for (int j = 0; j < nr; ++j) {
            const int z0 = p.reps[2 * j], z1 = p.reps[2 * j + 1];
            const int lo = min(z0, z1), hi = max(z0, z1);
            const int span = hi - lo + 1, W = 6 * span;
            const bool fwd = z0 <= z1;
            const double wj = w[j];
            for (int base = 0; base < N; base += LM_TP) {
                if (CL > 1 && (tile_id++ % CL) != crank) continue;
                const int np = min(LM_TP, N - base);
                // work item = (point, lane group g): the per-point part of Dr_Deps (everything that depends only on
                // the rep's full transform) is computed once and reused for the zetas g, g + LM_G, ... of the span;
                // point fastest, so the lanes of a warp share g and the chain transforms are broadcast reads.
                // The reference forms T0 = Tl * Tr per zeta [:96]; here every zeta of a rep uses the rep's own
                // product sRep[j], which is the same matrix up to the association order of the chain.
                constexpr int LM_G = 2;
                for (int it = tid; it < np * LM_G; it += LM_THREADS) {
                    const int pt = it % np, g = it / np;
                    const double* pp = gpr + ((size_t)j * N + base + pt) * 3;
                    const double* pq = gp_r + ((size_t)j * N + base + pt) * 3;
                    double* dst = sJ + pt;                                          // column c of this point: dst[c * TS]
                    JacCommon cm;
                    jac_common(sRep[j], pp, pq, hd, cm);
                    if (g == 0) dst[(size_t)W * TS] = wj * cm.res;                   // [:356-359]
                    for (int zi = g; zi < span; zi += LM_G) {
                        const int k = lo + zi;
                        double row[6];
                        if (fwd) {                                                  // [:271-275]
                            if (z0 < k) jac_zeta(cm, sMem[k * nz + z1], sMem[z0 * nz + (k - 1)], 1.0, pp, row);
                            else jac_zeta(cm, sMem[k * nz + z1], s_identity, 1.0, pp, row);
                        } else {                                                    // [:276-281]
                            if (z0 > k) jac_zeta(cm, sInv[z1 * nz + k], sInv[(k + 1) * nz + z0], -1.0, pp, row);
                            else jac_zeta(cm, sInv[z1 * nz + k], s_identity, -1.0, pp, row);
                        }
#pragma unroll
                        for (int c = 0; c < 6; ++c) dst[(size_t)(6 * zi + c) * TS] = wj * row[c];  // [:381,397]
                    }
                }
                // zero padding the MMA reads: columns W+1 .. 8 NB - 1, and the points np .. np4 - 1 of every column
                const int NB = (W + 1 + 7) >> 3, np4 = (np + 3) & ~3;
                for (int it = tid; it < (8 * NB - W - 1) * np4; it += LM_THREADS)
                    sJ[(size_t)(W + 1 + it / np4) * TS + it % np4] = 0.0;
                for (int it = tid; it < (W + 1) * (np4 - np); it += LM_THREADS)
                    sJ[(size_t)(it / (np4 - np)) * TS + np + it % (np4 - np)] = 0.0;
                __syncthreads();
                // Upper triangle of the (W+1) x (W+1) Gram matrix of the tile in 8 x 8 blocks on the tensor cores:
                // columns 0..W-1 -> H, column W (the residual) -> b.  A block belongs to one warp, which adds its
                // fragment into H | b afterwards: no atomics, a fixed summation order.  When there are fewer blocks
                // than warps (short spans) the correspondences of a block are split over several warps and the
                // partial fragments are summed in a fixed order through shared memory.
                {
                    constexpr int NWARP = LM_THREADS / 32, MAXB = 6;
                    const int nblk = NB * (NB + 1) / 2, ksteps = np4 >> 2;
                    const int warp = tid >> 5, lane = tid & 31;
                    const double* frag = sJ + (size_t)(lane >> 2) * TS + (lane & 3);   // + 8 b TS + 4 ks
                    if (nblk >= NWARP) {
                        for (int b0 = warp; b0 < nblk; b0 += NWARP * MAXB) {
                            double acc[MAXB][2];
                            int bi[MAXB], bj[MAXB];
                            bool ok[MAXB];
#pragma unroll
                            for (int q = 0; q < MAXB; ++q) {
                                const int blk = b0 + q * NWARP;
                                ok[q] = blk < nblk;
                                lm_block_of(ok[q] ? blk : 0, NB, bi[q], bj[q]);
                                acc[q][0] = acc[q][1] = 0.0;
                            }
                            for (int ks = 0; ks < ksteps; ++ks) {
#pragma unroll
                                for (int q = 0; q < MAXB; ++q)
                                    if (ok[q])
                                        dmma_m8n8k4(acc[q], frag[(size_t)8 * bi[q] * TS + 4 * ks], frag[(size_t)8 * bj[q] * TS + 4 * ks]);
                            }
#pragma unroll
                            for (int q = 0; q < MAXB; ++q)
                                if (ok[q]) {
                                    lm_gram_store(sAcc, D, lo, W, bi[q], bj[q], lane, 0, acc[q][0]);
                                    lm_gram_store(sAcc, D, lo, W, bi[q], bj[q], lane, 1, acc[q][1]);
                                }
                        }
                    } else {
                        const int KS = NWARP / nblk;                                 // warps per block (>= 1)
                        const int blk = warp / KS, sl = warp % KS;
                        if (blk < nblk) {
                            int bi, bj;
                            lm_block_of(blk, NB, bi, bj);
                            double acc[2] = {0.0, 0.0};
                            for (int ks = sl; ks < ksteps; ks += KS)
                                dmma_m8n8k4(acc, frag[(size_t)8 * bi * TS + 4 * ks], frag[(size_t)8 * bj * TS + 4 * ks]);
                            sScr[warp * 64 + 2 * lane] = acc[0];
                            sScr[warp * 64 + 2 * lane + 1] = acc[1];
                        }
                        __syncthreads();
                        for (int it = tid; it < nblk * 64; it += LM_THREADS) {
                            const int bq = it >> 6, el = it & 63;
                            double v = 0.0;
                            for (int q = 0; q < KS; ++q) v += sScr[(bq * KS + q) * 64 + el];   // fixed order
                            int bi, bj;
                            lm_block_of(bq, NB, bi, bj);
                            lm_gram_store(sAcc, D, lo, W, bi, bj, el >> 1, el & 1, v);
                        }
                    }
                }
                for (int pt = tid; pt < np; pt += LM_THREADS) {
                    const double r = sJ[(size_t)W * TS + pt];
                    rsq += r * r;
                }
                __syncthreads();
            }
        }
        if (CL > 1) {                               // cluster reduction of the partial H | b and of |r0|^2
            rsq = lm_warp_sum(rsq);
            if ((tid & 31) == 0) sRed[tid >> 5] = rsq;
            __syncthreads();
            if (tid == 0) {
                double s = 0.0;
                for (int i = 0; i < LM_THREADS / 32; ++i) s += sRed[i];
                s_part[0] = s;
            }
            cg::cluster_group cluster = cg::this_cluster();
            cluster.sync();                         // every rank's partial sums are complete and visible
            for (int e = tid; e < D * (D + 1); e += LM_THREADS) {
                double s = 0.0;
#pragma unroll
                for (int r = 0; r < CL; ++r) s += cluster.map_shared_rank(sHp, r)[e];     // rank order: identical in every CTA
                sH[e] = s;
            }
            if (tid == 0) {
                double s = 0.0;
#pragma unroll
                for (int r = 0; r < CL; ++r) s += *cluster.map_shared_rank(&s_part[0], r);
                s_rnorm = sqrt(s);
            }
            __syncthreads();
        }
        // symmetrise, damp, Frobenius norm, negate b                                [:403,473]
        for (int e = tid; e < D * D; e += LM_THREADS) {
            const int r = e / D, c = e % D;
            if (c < r) sH[(size_t)r * (D + 1) + c] = sH[(size_t)c * (D + 1) + r];
        }
        if (CL == 1) {
            rsq = lm_warp_sum(rsq);                  // per-warp partials: thread 0 adds LM_THREADS / 32 values, not LM_THREADS
            if ((tid & 31) == 0) sRed[tid >> 5] = rsq;
        }
        __syncthreads();
        const double lam = s_lambda;
        for (int r = tid; r < D; r += LM_THREADS) {
            sH[(size_t)r * (D + 1) + r] += lam * sH[(size_t)r * (D + 1) + r];
            sH[(size_t)r * (D + 1) + D] = -sH[(size_t)r * (D + 1) + D];
        }
        if (CL == 1 && tid == 0) {
            double s = 0.0;
            for (int i = 0; i < LM_THREADS / 32; ++i) s += sRed[i];
            s_rnorm = sqrt(s);
        }
        __syncthreads();
        {
            double hs = 0.0;
            for (int e = tid; e < D * D; e += LM_THREADS) {
                const double v = sH[(size_t)(e / D) * (D + 1) + e % D];
                hs += v * v;
            }
            __syncthreads();
            hs = lm_warp_sum(hs);
            if ((tid & 31) == 0) sRed[tid >> 5] = hs;
            __syncthreads();
            if (tid == 0) {
                double s = 0.0;
                for (int i = 0; i < LM_THREADS / 32; ++i) s += sRed[i];
                s_Hnorm = sqrt(s);
            }
        }
        // ---- solve H delta = -b: LU with partial pivoting on the augmented matrix  [:405]
        __syncthreads();
        {
            constexpr int NW = LM_THREADS >= 128 ? 4 : LM_THREADS / 32;     // solver warps: one per SM sub-partition
            if (tid < 32 * NW) {
                if (D + 1 <= 64) lm_warp_solve<2, 4, NW>(sH, sDelta, D, tid, p.epsilon, &s_stop, s_key, s_row);
                else lm_warp_solve<4, 4, NW>(sH, sDelta, D, tid, p.epsilon, &s_stop, s_key, s_row);
            }
        }
        __syncthreads();
        if (s_stop) break;
        // ---- candidate update T' = T exp(delta_k)                                  [:416-422]
        for (int k = tid; k < nz; k += LM_THREADS) {
            Rt ex;
            se3_exp(sDelta + 6 * k, ex);
            rt_mul(sT[k], ex, sTn[k]);
        }
        __syncthreads();
        for (int j = tid; j < nr; j += LM_THREADS) {                                 // [:425-442]
            const int z0 = p.reps[2 * j], z1 = p.reps[2 * j + 1];
            Rt acc;
            rt_identity(acc);
            if (z0 <= z1) {
                for (int k = z0; k <= z1; ++k) rt_mul(sTn[k], acc, acc);
            } else {
                for (int k = z0; k >= z1; --k) {
                    Rt inv;
                    rt_inv(sTn[k], inv);
                    rt_mul(inv, acc, acc);
                }
            }
            sRep[j] = acc;
        }
        __syncthreads();
        double csq = 0.0;                                                            // [:445-456]
        for (int it = crank * LM_THREADS + tid; it < nr * N; it += CL * LM_THREADS) {
            const int j = it / N;
            const double r = res_one(sRep[j], gpr + (size_t)it * 3, gp_r + (size_t)it * 3, hd);
            csq += r * r;
        }
        csq = lm_warp_sum(csq);
        if ((tid & 31) == 0) sRed[tid >> 5] = csq;
        __syncthreads();
        if (CL > 1) {
            if (tid == 0) {
                double s = 0.0;
                for (int i = 0; i < LM_THREADS / 32; ++i) s += sRed[i];
                s_part[1] = s;
            }
            cg::this_cluster().sync();
        }
        if (tid == 0) {
            double s = 0.0;
            if (CL > 1) {
#pragma unroll
                for (int r = 0; r < CL; ++r) s += *cg::this_cluster().map_shared_rank(&s_part[1], r);
            } else {
                for (int i = 0; i < LM_THREADS / 32; ++i) s += sRed[i];
            }
            const double currE = sqrt(s);
            s_rnorm = currE;                                                         // r0 now holds the candidate residuals
            if (currE < s_prevE) {                                                   // [:457-467]
                s_prevE = currE;
                s_piv = 1;
                s_lambda /= 2.0;
            } else {
                s_piv = 0;
                s_lambda *= 5.0;
            }
        }
        __syncthreads();
        if (s_piv) {
            for (int k = tid; k < nz; k += LM_THREADS) sT[k] = sTn[k];
        }
        __syncthreads();
    }
    __syncthreads();
    if (CL > 1) {
        cg::this_cluster().sync();                  // no CTA may exit while a peer can still read its shared memory
        if (crank != 0) return;                     // rank 0 reports (every rank holds the same result)
    }
    for (int k = tid; k < nz; k += LM_THREADS) {
        for (int i = 0; i < 3; ++i) {
            for (int j = 0; j < 3; ++j) gT[k * 16 + i * 4 + j] = sT[k].R[i * 3 + j];
            gT[k * 16 + i * 4 + 3] = sT[k].t[i];
        }
        gT[k * 16 + 12] = 0.0; gT[k * 16 + 13] = 0.0; gT[k * 16 + 14] = 0.0; gT[k * 16 + 15] = 1.0;
    }
    if (tid == 0) {
        p.out[prob].H_norm = s_Hnorm;                                                // [:473-475]
        p.out[prob].r_norm = s_rnorm;
        p.out[prob].lambda = s_lambda;
        if (p.iters) p.iters[prob] = s_iters;
    }
}

// ---- single-pair specialisation: n_zeta = 1, reps = {(0,0)} (the kitti_E.cpp:196 call) --------
// One WARP per problem, everything in registers: each lane owns up to two correspondences,
// the 6x6 normal equations are reduced with warp shuffles and solved redundantly by every lane,
// so the 30 dependent iterations need no shared memory and no block barrier.
constexpr int LMP_WARPS = 4;
constexpr int LMP_MINBLOCKS = 1;

// lanes per problem: 32 = one warp per problem (two correspondences per lane); 16 / 8 pack two /
// four problems into a warp (four / eight correspondences per lane), trading per-problem latency
// for fewer, fuller warps -- the 30 dependent iterations make this kernel latency bound.
constexpr int LM_LPP = 8;
constexpr int LM_PPL = 64 / LM_LPP;                 // correspondences per lane (N <= 64)

__device__ __forceinline__ double group_sum_d(double v) {
#pragma unroll
    for (int o = LM_LPP / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

__global__ void __launch_bounds__(LMP_WARPS * 32, LMP_MINBLOCKS) lm_pair_kernel(LmPlan p) {
    const int gl = threadIdx.x & (LM_LPP - 1);                                  // lane within the problem's group
    const int prob_raw = (blockIdx.x * LMP_WARPS * 32 + threadIdx.x) / LM_LPP;
    const bool exists = prob_raw < p.B;
    const int prob = exists ? prob_raw : p.B - 1;                               // clamp: shuffles need every lane
    bool done = !exists || (p.active && !p.active[prob]);
    const bool skip = done;                                                      // nothing is written for this problem
    if (__all_sync(0xFFFFFFFFu, done)) return;
    const int N = p.N;
    double* gT = p.T0s + (size_t)prob * 16;
    const double* gpr = p.pr + (size_t)prob * N * 3;
    const double* gp_r = p.p_r + (size_t)prob * N * 3;
    const double w = p.wreps[prob];
    const double hd = p.huber_delta;
    Rt T, I;
    rt_identity(I);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j) T.R[i * 3 + j] = gT[i * 4 + j];
        T.t[i] = gT[i * 4 + 3];
    }
    // this lane's correspondences
    double pa[LM_PPL][3], pb[LM_PPL][3];
    bool have[LM_PPL];
#pragma unroll
    for (int k = 0; k < LM_PPL; ++k) {
        const int i = gl + LM_LPP * k;
        have[k] = i < N;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            pa[k][c] = have[k] ? gpr[i * 3 + c] : 1.0;
            pb[k][c] = have[k] ? gp_r[i * 3 + c] : 1.0;
        }
    }
    // the accept test compares NORMS as the reference does [:456-457]: on a converged plateau two sums of squares
    // that differ by an ulp can have equal square roots, and `<` must then reject
    double lambda = p.lambda0, prevE = 1e10, hs_out = 0.0, rsq_out = 0.0;
    int iters = 0;
    for (int iter = 0; iter < p.max_iters; ++iter) {
        if (__all_sync(0xFFFFFFFFu, done)) break;
        if (!done) iters = iter + 1;
        double H[21], b[6], rsq = 0.0;
#pragma unroll
        for (int i = 0; i < 21; ++i) H[i] = 0.0;
#pragma unroll
        for (int i = 0; i < 6; ++i) b[i] = 0.0;
#pragma unroll
        for (int k = 0; k < LM_PPL; ++k) {
            if (!have[k]) continue;
            double row[6], r;
            jac_row(T, I, T, 1.0, pa[k], pb[k], hd, row, &r);                       // [:356-359, :372-381]
            r *= w;
#pragma unroll
            for (int c = 0; c < 6; ++c) row[c] *= w;
            int e = 0;
#pragma unroll
            for (int a = 0; a < 6; ++a) {
#pragma unroll
                for (int c = a; c < 6; ++c) H[e++] += row[a] * row[c];
                b[a] += row[a] * r;
            }
            rsq += r * r;
        }
#pragma unroll
        for (int i = 0; i < 21; ++i) H[i] = group_sum_d(H[i]);
#pragma unroll
        for (int i = 0; i < 6; ++i) b[i] = group_sum_d(b[i]);
        rsq = group_sum_d(rsq);
        // augmented, damped system  [H + lambda diag(H) | -b]                      [:403-405]
        double A[6][7];
        {
            int e = 0;
#pragma unroll
            for (int a = 0; a < 6; ++a)
#pragma unroll
                for (int c = a; c < 6; ++c) { A[a][c] = H[e]; A[c][a] = H[e]; ++e; }
        }
        double hs = 0.0;
#pragma unroll
        for (int a = 0; a < 6; ++a) {
            A[a][a] += lambda * A[a][a];
            A[a][6] = -b[a];
        }
#pragma unroll
        for (int a = 0; a < 6; ++a)
#pragma unroll
            for (int c = 0; c < 6; ++c) hs += A[a][c] * A[a][c];
        double ip[6];                                       // reciprocal pivots
#pragma unroll
        for (int k = 0; k < 6; ++k) {                       // LU, partial pivoting (uniform across the group)
            int pv = k;
            double best = fabs(A[k][k]);
#pragma unroll
            for (int r = k + 1; r < 6; ++r)
                if (fabs(A[r][k]) > best) { best = fabs(A[r][k]); pv = r; }
#pragma unroll
            for (int r = k + 1; r < 6; ++r)
                if (r == pv) {
#pragma unroll
                    for (int c = 0; c < 7; ++c) { const double t = A[k][c]; A[k][c] = A[r][c]; A[r][c] = t; }
                }
            ip[k] = 1.0 / A[k][k];
#pragma unroll
            for (int r = k + 1; r < 6; ++r) {
                const double f = A[r][k] * ip[k];
#pragma unroll
                for (int c = k + 1; c < 7; ++c) A[r][c] -= f * A[k][c];
            }
        }
        double d[6], dn = 0.0;
        bool bad = false;
#pragma unroll
        for (int r = 5; r >= 0; --r) {
            double s = A[r][6];
#pragma unroll
            for (int c = r + 1; c < 6; ++c) s -= A[r][c] * d[c];
            d[r] = s * ip[r];
            bad |= !(d[r] == d[r]);                                                 // hasNaN(): NaN only
            dn += d[r] * d[r];
        }
        if (!done) { rsq_out = rsq; hs_out = hs; }
        if (bad || sqrt(dn) < p.epsilon) done = true;                               // [:407-414]
        Rt ex, Tn;
        se3_exp(d, ex);                                                             // [:416-422]
        rt_mul(T, ex, Tn);
        double csq = 0.0;                                                           // [:445-456]
#pragma unroll
        for (int k = 0; k < LM_PPL; ++k) {
            if (!have[k]) continue;
            const double r = res_one(Tn, pa[k], pb[k], hd);
            csq += r * r;
        }
        csq = group_sum_d(csq);
        if (!done) {
            rsq_out = csq;                                                          // r0 now holds the candidate residuals
            const double currE = sqrt(csq);
            if (currE < prevE) {                                                    // [:457-467]
                prevE = currE;
                T = Tn;
                lambda /= 2.0;
            } else {
                lambda *= 5.0;
            }
        }
    }
    const double Hnorm = sqrt(hs_out), rnorm = sqrt(rsq_out);
    if (gl == 0 && !skip) {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
#pragma unroll
            for (int j = 0; j < 3; ++j) gT[i * 4 + j] = T.R[i * 3 + j];
            gT[i * 4 + 3] = T.t[i];
        }
        gT[12] = 0.0; gT[13] = 0.0; gT[14] = 0.0; gT[15] = 1.0;
        p.out[prob].H_norm = Hnorm;
        p.out[prob].r_norm = rnorm;
        p.out[prob].lambda = lambda;
        if (p.iters) p.iters[prob] = iters;
    }
}

size_t lm_smem_doubles(int nz, int nr, int D, int threads, int tp, int cl) {
    size_t rt = sizeof(Rt) / sizeof(double);
    return rt * (2 * (size_t)nz + 2 * (size_t)nz * nz + nr) + (size_t)D * (D + 1) * (cl > 1 ? 2 : 1) +
           (size_t)lm_tile_cols(D) * lm_tile_stride(tp) + D + 3 * (size_t)threads;
}

// the shared-memory test of one CTA shape: a window of n_zeta zetas and n_rep reps must fit
template <int THREADS, int TP, int CL = 1>
int lm_shape_fits(epivo_ctx* ctx, int n_zeta, int n_rep) {
    const size_t bytes = lm_smem_doubles(n_zeta, n_rep, 6 * n_zeta, THREADS, TP, CL) * sizeof(double);
    if (bytes > LM_SMEM_LIMIT)
        EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "LM problem needs %zu bytes of shared memory (n_zeta=%d, n_rep=%d)", bytes,
                 n_zeta, n_rep);
    return EPIVO_OK;
}

template <int THREADS, int TP, int CL = 1>
int lm_launch_shape(epivo_ctx* ctx, LmArgs& a) {
    const int rc = lm_shape_fits<THREADS, TP, CL>(ctx, a.p.n_zeta, a.p.n_rep);
    if (rc) return rc;
    a.smem_doubles = lm_smem_doubles(a.p.n_zeta, a.p.n_rep, a.D, THREADS, TP, CL);
    const size_t bytes = a.smem_doubles * sizeof(double);
    EPV_CUDA(ctx, cudaFuncSetAttribute(lm_kernel<THREADS, TP, CL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    if (CL == 1) {
        lm_kernel<THREADS, TP, CL><<<a.p.B, THREADS, bytes, ctx->stream>>>(a);
    } else {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)a.p.B * CL);
        cfg.blockDim = dim3(THREADS);
        cfg.dynamicSmemBytes = bytes;
        cfg.stream = ctx->stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = CL;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        EPV_CUDA(ctx, cudaLaunchKernelEx(&cfg, lm_kernel<THREADS, TP, CL>, a));
    }
    EPV_LAUNCHED(ctx);
    return EPIVO_OK;
}

}  // namespace

int epv_lm_check_n32(epivo_ctx* ctx, int n_zeta, int n_rep) {
    if (n_zeta < 1 || n_zeta > LM_MAX_ZETA)
        EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "n_zeta = %d outside [1, %d]", n_zeta, LM_MAX_ZETA);
    if (n_rep < 1) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "n_rep = %d", n_rep);
    return lm_shape_fits<64, 32>(ctx, n_zeta, n_rep);
}

int epv_lm_launch(epivo_ctx* ctx, const LmPlan& p) {
    if (p.B <= 0) return EPIVO_OK;
    if (p.n_zeta < 1 || p.n_zeta > LM_MAX_ZETA)
        EPV_FAIL(ctx, EPIVO_ERR_UNSUPPORTED, "n_zeta = %d outside [1, %d]", p.n_zeta, LM_MAX_ZETA);
    if (p.n_rep < 1 || p.N < 1) EPV_FAIL(ctx, EPIVO_ERR_INVALID, "n_rep = %d, N = %d", p.n_rep, p.N);
    if (p.single_pair && p.n_zeta == 1 && p.n_rep == 1 && p.N <= 64) {
        const int per_block = LMP_WARPS * 32 / LM_LPP;       // problems per CTA
        lm_pair_kernel<<<(p.B + per_block - 1) / per_block, LMP_WARPS * 32, 0, ctx->stream>>>(p);
        EPV_LAUNCHED(ctx);
        return EPIVO_OK;
    }
    LmArgs a;
    a.p = p;
    a.D = 6 * p.n_zeta;
    // long chains: only the smallest tile leaves room for H | b and the memo
    if (lm_smem_doubles(p.n_zeta, p.n_rep, a.D, 128, 64, 1) * sizeof(double) > LM_SMEM_LIMIT)
        return lm_launch_shape<64, 32>(ctx, a);
    // The shapes differ in summation order (tile boundaries, cluster partials), so the last bits of H | b -- and, on a
    // converged plateau, the accept / reject sequence -- depend on the shape, which follows from the batch size: the
    // same window can take a different (equally valid) trajectory in a 504-window batch and in a 63-window shard.
    // tests/test_gpu_lm_ref.py holds every shape below to the reference's result within north_star's tolerance.
    if (p.N <= 32) return lm_launch_shape<64, 32>(ctx, a);          // e.g. the shipped kitti_ba shape: 9 reps x 32 points
    // few large windows (a multi-GPU shard of cfg5: 63 windows per GPU): every CTA has an SM to itself, so the
    // wider CTA wins (63 cfg5 windows: 11.3 ms against 14.0 ms); with several CTAs per SM the narrower one does
    // and when even that leaves SMs idle, a window is shared by a cluster of 2 or 4 CTAs (63 windows: 6.65 ms on
    // pairs of CTAs; 30 windows: 6.05 ms on clusters of four, 9.9 ms on single CTAs)
    if (p.N >= 96 && p.B * 4 <= ctx->sm_count) return lm_launch_shape<384, 64, 4>(ctx, a);
    if (p.N >= 96 && p.B * 2 <= ctx->sm_count) return lm_launch_shape<384, 128, 2>(ctx, a);
    if (p.N >= 96 && p.B <= ctx->sm_count) return lm_launch_shape<384, 128>(ctx, a);
    if (p.N >= 96) return lm_launch_shape<192, 96>(ctx, a);         // e.g. cfg5: 20 reps x 250 points
    return lm_launch_shape<128, 64>(ctx, a);
}
