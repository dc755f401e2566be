// K2: Nister 5-point minimal solver, FP64, in three stages (A, B1: one hypothesis per lane; B2: one real root per lane).
//
// Restates the algorithm of cv::findEssentialMat's EMEstimatorCallback::runKernel
// (OpenCV modules/calib3d/src/five-point.cpp; called from kitti.cpp:98, kitti_E.cpp:98,
// euroc_E.cpp:202, kitti_ba.cpp:232,308,702):
//   1. 5x9 epipolar system (row-major E, x2' E x1 = 0) -> 4-D null space
//      (OpenCV: full SVD; here: Householder QR of the transpose -- any orthonormal basis of
//      the same null space yields the same set of essential matrices),
//   2. the ten cubic constraints -> Nister's 10x20 matrix (fivept_gen.cuh),
//   3. elimination with partial pivoting on the left 10x10 block (OpenCV: inv() * right); only
//      rows 4..9 of inv(left) * right are needed, so the back substitution stops there,
//   4. B(z) = {rows 4,6,8} - z {rows 5,7,9}, det B(z) = degree-10 polynomial,
//   5. all complex roots by the Durand-Kerner iteration of cv::solvePoly (same start
//      values (1+i)^k, same Gauss-Seidel sweep, 300 sweeps at most; stops early once every
//      update of a sweep is below 1e-13 of its root -- OpenCV keeps sweeping at round-off level),
//   6. per root with |imag| <= 1e-10: (x, y) from the null vector of B(z) (skipped if its
//      third component is < 1e-10 in magnitude), E = x E0 + y E1 + z E2 + E3, normalised,
//   7. (not in OpenCV) each solution is refined by Gauss-Newton on the ten constraints inside the
//      null space (refine_essential below), which removes the basis-dependent loss of accuracy.
//
// Stage A (steps 1-3) needs the 10x20 matrix, which only fits on chip in shared memory: one warp
// = 32 hypotheses, the matrix lane-strided (element (r,c) of lane l at [(r*20+c)*32 + l], bank =
// lane, conflict free even though every lane pivots on a different row).  Its product is 96
// doubles per hypothesis (null-space basis + six reduced rows).  A thread-private 10x20 array
// would live in local memory, and with tens of thousands of hypotheses in flight that traffic
// goes to HBM.  Stage B1 (steps 4-5) is one lane per hypothesis, registers only.  Stage B2
// (steps 6-7) is one lane per REAL ROOT: hypotheses have 0..10 real roots (4.3 on average), so
// the roots are compacted into a work list first instead of idling the lanes of a warp.
#pragma once
#include "fivept_gen.cuh"

namespace fivept {

constexpr int EB_DOUBLES = 96;     // stage A -> stage B record: e[4][9] then rows 4..9 x 10 right-hand columns

// this lane's 10x20 matrix inside a warp-wide, lane-strided shared-memory block
struct SmemMat {
    double* base;       // already offset by the lane
    __device__ __forceinline__ double& operator()(int r, int c) const { return base[(r * 20 + c) * 32]; }
};

__device__ __forceinline__ void null_space_5x9(const double (&x1)[5][2], const double (&x2)[5][2],
                                               double (&e)[4][9]) {
    // A = Q' (9 x 5), column c = epipolar row of correspondence c
    double A[9][5];
#pragma unroll
    for (int c = 0; c < 5; ++c) {
        const double a1 = x1[c][0], b1 = x1[c][1], a2 = x2[c][0], b2 = x2[c][1];
        A[0][c] = a2 * a1; A[1][c] = a2 * b1; A[2][c] = a2;
        A[3][c] = b2 * a1; A[4][c] = b2 * b1; A[5][c] = b2;
        A[6][c] = a1;      A[7][c] = b1;      A[8][c] = 1.0;
    }
    double beta[5];
    // Householder QR: reflector k zeroes A[k+1.., k]; v_k is stored in A[k.., k] (v_k[k] = 1 implied)
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        double s = 0.0;
#pragma unroll
        for (int r = k; r < 9; ++r) s += A[r][k] * A[r][k];
        const double nrm = sqrt(s);
        const double alpha = A[k][k] > 0 ? -nrm : nrm;
        const double v0 = A[k][k] - alpha;
        // beta = 2 / (v'v), with v = (v0, A[k+1..][k]);  v'v = s - A[k][k]^2 + v0^2
        const double vtv = s - A[k][k] * A[k][k] + v0 * v0;
        beta[k] = vtv > 0 ? 2.0 / vtv : 0.0;
        A[k][k] = v0;
#pragma unroll
        for (int c = k + 1; c < 5; ++c) {
            double d = 0.0;
#pragma unroll
            for (int r = k; r < 9; ++r) d += A[r][k] * A[r][c];
            d *= beta[k];
#pragma unroll
            for (int r = k; r < 9; ++r) A[r][c] -= d * A[r][k];
        }
    }
    // null space = last four columns of Q_full = H_0 ... H_4 applied to e_5 .. e_8
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        double v[9];
#pragma unroll
        for (int r = 0; r < 9; ++r) v[r] = (r == 5 + b) ? 1.0 : 0.0;
#pragma unroll
        for (int k = 4; k >= 0; --k) {
            double d = 0.0;
#pragma unroll
            for (int r = k; r < 9; ++r) d += A[r][k] * v[r];
            d *= beta[k];
#pragma unroll
            for (int r = k; r < 9; ++r) v[r] -= d * A[r][k];
        }
#pragma unroll
        for (int r = 0; r < 9; ++r) e[b][r] = v[r];
    }
}

// Rows 4..9 of inv(left 10x10) * (right 10x10): forward elimination with partial pivoting to a
// unit upper-triangular left block, then back substitution of rows 9..4 only.  The result
// overwrites A(4..9, 10..19).  Returns false if the left block is singular.
template <class Mat>
__device__ __forceinline__ bool reduce_rows_4_9(Mat& A) {
    for (int k = 0; k < 10; ++k) {
        int p = k;
        double best = fabs(A(k, k));
        for (int r = k + 1; r < 10; ++r) {
            const double v = fabs(A(r, k));
            if (v > best) { best = v; p = r; }
        }
        if (!(best > 1e-300)) return false;
        // pivot row -> registers, scaled; the old row k goes where the pivot row was
        double row[20];
        const double inv = 1.0 / A(p, k);
        if (p != k) A(p, k) = A(k, k);                 // multiplier column of the displaced row
#pragma unroll
        for (int c = 0; c < 20; ++c) {
            if (c > k) {                               // columns <= k of the pivot row are never read again
                const double v = A(p, c);
                if (p != k) A(p, c) = A(k, c);
                row[c] = v * inv;
                A(k, c) = row[c];
            }
        }
        for (int r = k + 1; r < 10; ++r) {
            const double f = A(r, k);
            if (f == 0.0) continue;
#pragma unroll
            for (int c = 0; c < 20; ++c)
                if (c > k) A(r, c) -= f * row[c];
        }
    }
    // X_i = Y_i - sum_{j > i} U_ij X_j, rows 9 (already final) down to 4
    for (int i = 8; i >= 4; --i) {
        double acc[10];
#pragma unroll
        for (int c = 0; c < 10; ++c) acc[c] = A(i, 10 + c);
        for (int j = i + 1; j < 10; ++j) {
            const double u = A(i, j);
#pragma unroll
            for (int c = 0; c < 10; ++c) acc[c] -= u * A(j, 10 + c);
        }
#pragma unroll
        for (int c = 0; c < 10; ++c) A(i, 10 + c) = acc[c];
    }
    return true;
}

// ---- stage A: correspondences -> null-space basis + reduced rows ------------------------------
// out[k * out_stride], k < EB_DOUBLES.  A singular system is flagged by a NaN in out[36].
__device__ __forceinline__ void stage_a(const double (&x1)[5][2], const double (&x2)[5][2], SmemMat A, double* out,
                                        size_t out_stride) {
    double e[4][9];
    null_space_5x9(x1, x2, e);
    fivept_constraints(e, A);
#pragma unroll
    for (int b = 0; b < 4; ++b)
#pragma unroll
        for (int r = 0; r < 9; ++r) out[(size_t)(b * 9 + r) * out_stride] = e[b][r];
    const bool ok = reduce_rows_4_9(A);
    for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int c = 0; c < 10; ++c)
            out[(size_t)(36 + i * 10 + c) * out_stride] = ok ? A(4 + i, 10 + c) : __longlong_as_double(0x7FF8000000000000LL);
}

// ascending-power polynomial product: out[0..na+nb] = a[0..na] * b[0..nb]
template <int NA, int NB>
__device__ __forceinline__ void pmul(const double (&a)[NA + 1], const double (&b)[NB + 1], double (&out)[NA + NB + 1]) {
#pragma unroll
    for (int i = 0; i <= NA + NB; ++i) out[i] = 0.0;
#pragma unroll
    for (int i = 0; i <= NA; ++i)
#pragma unroll
        for (int j = 0; j <= NB; ++j) out[i + j] += a[i] * b[j];
}

// cv::solvePoly's Durand-Kerner on real coefficients c[0..n] (ascending), n <= 10.
// dk_sweeps<N>: degree known at compile time, so the roots live in registers and both loops are
// fully unrolled.  Same start values and Gauss-Seidel sweep order as cv::solvePoly.
// cv::solvePoly only stops when a sweep's update is exactly zero, which practically never
// happens: it runs all 300 sweeps while the roots jitter at round-off level.  Stopping once
// every update is below 1e-13 of the root leaves the roots equal to OpenCV's up to that jitter.
// Some polynomials never get there: clustered roots sit on a noise floor of 1e-12 .. 1e-9, where the update
// stops shrinking and merely fluctuates -- more sweeps only re-draw the noise, so the iteration ends there
// (small update, not smaller than the sweep before).  Close pairs of real roots, on the other hand, converge
// LINEARLY for dozens of sweeps before the quadratic phase sets in, their update shrinking a little every
// sweep; these must be followed to the end, because whether the pair comes out real (|imag| <= 1e-10) decides
// which models the sample contributes.  (Round 1 stopped as soon as the update shrank by less than 10x per
// sweep: on low-parallax EuRoC-shaped pairs that lost close pairs of real roots and, now and then, the winning
// model.)  A lane that is still shrinking after DK_FAST_SWEEPS sweeps returns false and the caller queues the
// hypothesis for the slow pass (the same iteration, continued up to OpenCV's 300 sweeps), so that it does not
// stall its warp.
// The relative update of a sweep is tracked as a fraction (numerator, denominator) compared by
// cross-multiplication, so a sweep costs one division per root, not two.
constexpr int DK_FAST_SWEEPS = 32;   // sweeps the fast path spends before handing a hypothesis over
constexpr int DK_STATE = 21;         // doubles saved for the slow pass: re[10], im[10], prev2

// Sweeps [first, last) of the iteration; first == 0 sets the start values, otherwise re / im / prev2 continue a
// previous call.  Returns true when the iteration is settled (converged, on the noise floor, or 300 sweeps done).
template <int N>
__device__ __forceinline__ bool dk_sweeps(const double (&c)[11], double (&re)[10], double (&im)[10], double& prev2,
                                          int first, int last) {
    if (first == 0) {
        double pr = 1.0, pi = 0.0;
#pragma unroll
        for (int i = 0; i < N; ++i) {                        // roots[i] = (1 + 1i)^i
            re[i] = pr; im[i] = pi;
            const double t = pr - pi;
            pi = pr + pi; pr = t;
        }
        prev2 = 1e300;
    }
#pragma unroll 1
    for (int iter = first; iter < last; ++iter) {
        double mnum = 0.0, mden = 1.0;                       // max over roots of |update|^2 / max(1, |root|^2)
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const double xr = re[i], xi = im[i];
            double nr = c[N], ni = 0.0, dr = c[N], di = 0.0;
#pragma unroll
            for (int j = 0; j < N; ++j) {
                const double t = nr * xr - ni * xi + c[N - j - 1];     // num = num * x + c[N-j-1]
                ni = nr * xi + ni * xr;
                nr = t;
                if (j != i) {
                    const double er = xr - re[j], ei = xi - im[j];
                    const bool nz = (er != 0.0 || ei != 0.0);
                    const double u = dr * er - di * ei;
                    const double v = dr * ei + di * er;
                    di = nz ? v : di;
                    dr = nz ? u : dr;
                }
            }
            const double s = 1.0 / (dr * dr + di * di);
            const double qr = (nr * dr + ni * di) * s;
            const double qi = (ni * dr - nr * di) * s;
            re[i] = xr - qr; im[i] = xi - qi;
            const double q2 = qr * qr + qi * qi, m = fmax(1.0, xr * xr + xi * xi);
            if (q2 * mden > mnum * m || !(q2 == q2)) { mnum = q2; mden = m; }
        }
        const double maxrel2 = mnum / mden;
        if (!(maxrel2 > 1e-26)) return true;                 // converged (or NaN: nothing more to do either way)
        // On the noise floor the update stops shrinking and fluctuates; while a close pair is still converging
        // linearly it keeps shrinking, sweep after sweep.  So: small AND not smaller than last sweep's = floor.
        if (maxrel2 < 1e-12 && !(maxrel2 < prev2)) return true;
        prev2 = maxrel2;
    }
    return last >= 300;                                      // false: still shrinking slowly -> the slow pass continues
}

// Generic degree, all sweeps: cv::solvePoly as written (stops only when a sweep changes nothing).  Used for the rare
// polynomials whose leading coefficients vanished; kept out of line.
__device__ __noinline__ void dk_sweeps_full(const double (&c)[11], int n, double (&re)[10], double (&im)[10]) {
    double pr = 1.0, pi = 0.0;
    for (int i = 0; i < n; ++i) {
        re[i] = pr; im[i] = pi;
        const double t = pr - pi;
        pi = pr + pi; pr = t;
    }
    for (int iter = 0; iter < 300; ++iter) {
        double maxdiff2 = 0.0;
        for (int i = 0; i < n; ++i) {
            const double xr = re[i], xi = im[i];
            double nr = c[n], ni = 0.0, dr = c[n], di = 0.0;
            for (int j = 0; j < n; ++j) {
                const double t = nr * xr - ni * xi + c[n - j - 1];
                ni = nr * xi + ni * xr;
                nr = t;
                if (j != i) {
                    const double er = xr - re[j], ei = xi - im[j];
                    if (er != 0.0 || ei != 0.0) {
                        const double u = dr * er - di * ei;
                        di = dr * ei + di * er;
                        dr = u;
                    }
                }
            }
            const double s = 1.0 / (dr * dr + di * di);
            const double qr = (nr * dr + ni * di) * s;
            const double qi = (ni * dr - nr * di) * s;
            re[i] = xr - qr; im[i] = xi - qi;
            maxdiff2 = fmax(maxdiff2, qr * qr + qi * qi);
        }
        if (!(maxdiff2 > 0.0)) break;                        // `if (maxDiff <= 0) break;`
    }
}

// Unit null vector of a (near) rank-2 3x3 matrix: the largest of the row cross products.
__device__ __forceinline__ void null_vec3(const double (&M)[3][3], double (&v)[3]) {
    double best = -1.0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const int r0 = a, r1 = (a + 1) % 3;
        const double cx = M[r0][1] * M[r1][2] - M[r0][2] * M[r1][1];
        const double cy = M[r0][2] * M[r1][0] - M[r0][0] * M[r1][2];
        const double cz = M[r0][0] * M[r1][1] - M[r0][1] * M[r1][0];
        const double n2 = cx * cx + cy * cy + cz * cz;
        if (n2 > best) { best = n2; v[0] = cx; v[1] = cy; v[2] = cz; }
    }
    const double inv = best > 0 ? rsqrt(best) : 0.0;
    v[0] *= inv; v[1] *= inv; v[2] *= inv;
}

// ---- refinement (not in OpenCV) -----------------------------------------------------------
// Nister's elimination works in the chart "coefficient of e[3] = 1" of an ARBITRARY null-space
// basis (OpenCV: LAPACK SVD; here: Householder QR).  When a solution has a small e[3]
// component, or the sample is near-degenerate (low parallax), the expanded degree-10
// polynomial loses digits by an amount that differs from basis to basis.  A few Gauss-Newton
// steps on the ten cubic constraints themselves, on the unit sphere of the four basis
// coefficients, make every implementation converge (quadratically) to the same exact
// solutions.  A step is kept only if it lowers the constraint residual.
__device__ __forceinline__ void mat3_mul(const double* A, const double* B, double* C) {          // C = A B
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) C[i * 3 + j] = A[i * 3] * B[j] + A[i * 3 + 1] * B[3 + j] + A[i * 3 + 2] * B[6 + j];
}
__device__ __forceinline__ void mat3_mul_nt(const double* A, const double* B, double* C) {       // C = A B'
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) C[i * 3 + j] = A[i * 3] * B[j * 3] + A[i * 3 + 1] * B[j * 3 + 1] + A[i * 3 + 2] * B[j * 3 + 2];
}
__device__ __forceinline__ void mat3_mul_tn(const double* A, const double* B, double* C) {       // C = A' B
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) C[i * 3 + j] = A[i] * B[j] + A[3 + i] * B[3 + j] + A[6 + i] * B[6 + j];
}

constexpr int REFINE_ITERS = 10;
// A refined model must satisfy the ten constraints to this (max-abs, unit Frobenius norm).  On a near-degenerate sample
// the Gauss-Newton iteration can stall far from any solution (residual 1e-5 .. 1e-3): what it holds then is not an
// essential matrix, and it is dropped -- OpenCV would carry its own, equally meaningless, un-refined root instead.
constexpr double REFINE_ACCEPT = 1e-9;

__device__ __forceinline__ double constraints10(const double* E, double* F) {
    double G[9], T[9];
    mat3_mul_nt(E, E, G);                      // E E'
    mat3_mul(G, E, T);
    const double tr = G[0] + G[4] + G[8];
    double m = 0.0;
#pragma unroll
    for (int i = 0; i < 9; ++i) { F[i] = 2.0 * T[i] - tr * E[i]; m = fmax(m, fabs(F[i])); }
    F[9] = E[0] * (E[4] * E[8] - E[5] * E[7]) - E[1] * (E[3] * E[8] - E[5] * E[6]) + E[2] * (E[3] * E[7] - E[4] * E[6]);
    return fmax(m, fabs(F[9]));
}

// e: the null-space basis, element i of basis matrix k at e[(k * 9 + i) * es] (es = element stride,
// so the basis can stay in a thread-strided shared-memory block)
__device__ __noinline__ double refine_essential(const double* e, int es, double (&E)[9]) {
    double c[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        double s = 0.0;
#pragma unroll
        for (int i = 0; i < 9; ++i) s += E[i] * e[(k * 9 + i) * es];
        c[k] = s;
    }
    {
        const double n2 = c[0] * c[0] + c[1] * c[1] + c[2] * c[2] + c[3] * c[3];
        if (!(n2 > 0)) return 1e300;
        const double in = rsqrt(n2);
#pragma unroll
        for (int k = 0; k < 4; ++k) c[k] *= in;
    }
    double Ec[9], F[10];
#pragma unroll
    for (int i = 0; i < 9; ++i)
        Ec[i] = c[0] * e[i * es] + c[1] * e[(9 + i) * es] + c[2] * e[(18 + i) * es] + c[3] * e[(27 + i) * es];
    double fmaxv = constraints10(Ec, F);
    for (int it = 0; it < REFINE_ITERS; ++it) {
        // J column k = dF along basis matrix k
        double J[10][4];
        double G[9], EtE[9], cof[9];
        mat3_mul_nt(Ec, Ec, G);                 // E E'
        mat3_mul_tn(Ec, Ec, EtE);               // E'E
        const double tr = G[0] + G[4] + G[8];
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
                cof[i * 3 + j] = Ec[i1 * 3 + j1] * Ec[i2 * 3 + j2] - Ec[i1 * 3 + j2] * Ec[i2 * 3 + j1];
            }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            double D[9];
#pragma unroll
            for (int i = 0; i < 9; ++i) D[i] = e[(k * 9 + i) * es];
            double A1[9], A2[9], A3[9], T[9];
            mat3_mul(D, EtE, A1);               // D E'E
            mat3_mul_nt(Ec, D, T);              // E D'
            mat3_mul(T, Ec, A2);                // E D' E
            mat3_mul(G, D, A3);                 // E E' D
            const double trED = T[0] + T[4] + T[8];
            double dd = 0.0;
#pragma unroll
            for (int i = 0; i < 9; ++i) {
                J[i][k] = 2.0 * (A1[i] + A2[i] + A3[i]) - 2.0 * trED * Ec[i] - tr * D[i];
                dd += cof[i] * D[i];
            }
            J[9][k] = dd;
        }
        double N[4][5];
        double trN = 0.0;
#pragma unroll
        for (int a = 0; a < 4; ++a) {
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                double s = 0.0;
#pragma unroll
                for (int r = 0; r < 10; ++r) s += J[r][a] * J[r][b];
                N[a][b] = s;
            }
            double s = 0.0;
#pragma unroll
            for (int r = 0; r < 10; ++r) s += J[r][a] * F[r];
            N[a][4] = -s;
            trN += N[a][a];
        }
        const double mu = 1e3 * trN;             // pins the radial (scale) direction
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) N[a][b] += mu * c[a] * c[b];
        // 4x4 Gaussian elimination with partial pivoting (reciprocal pivots)
        bool ok = true;
        double ip[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            int p = k;
            double best = fabs(N[k][k]);
#pragma unroll
            for (int r = k + 1; r < 4; ++r)
                if (fabs(N[r][k]) > best) { best = fabs(N[r][k]); p = r; }
            if (!(best > 0)) { ok = false; break; }
#pragma unroll
            for (int r = k + 1; r < 4; ++r)
                if (r == p) {
#pragma unroll
                    for (int q = 0; q < 5; ++q) { const double t = N[k][q]; N[k][q] = N[r][q]; N[r][q] = t; }
                }
            ip[k] = 1.0 / N[k][k];
#pragma unroll
            for (int r = k + 1; r < 4; ++r) {
                const double f = N[r][k] * ip[k];
#pragma unroll
                for (int q = k; q < 5; ++q) N[r][q] -= f * N[k][q];
            }
        }
        if (!ok) break;
        double d[4];
#pragma unroll
        for (int r = 3; r >= 0; --r) {
            double s = N[r][4];
#pragma unroll
            for (int q = r + 1; q < 4; ++q) s -= N[r][q] * d[q];
            d[r] = s * ip[r];
        }
        double c2[4], n2 = 0.0, dn = 0.0;
#pragma unroll
        for (int k = 0; k < 4; ++k) { c2[k] = c[k] + d[k]; n2 += c2[k] * c2[k]; dn += d[k] * d[k]; }
        const double in2 = rsqrt(n2);
        double E2[9], F2[10];
#pragma unroll
        for (int k = 0; k < 4; ++k) c2[k] *= in2;
#pragma unroll
        for (int i = 0; i < 9; ++i)
            E2[i] = c2[0] * e[i * es] + c2[1] * e[(9 + i) * es] + c2[2] * e[(18 + i) * es] + c2[3] * e[(27 + i) * es];
        const double f2 = constraints10(E2, F2);
        if (!(f2 < fmaxv)) break;                // NaN or no improvement: keep the current iterate
        fmaxv = f2;
#pragma unroll
        for (int k = 0; k < 4; ++k) c[k] = c2[k];
#pragma unroll
        for (int i = 0; i < 9; ++i) Ec[i] = E2[i];
#pragma unroll
        for (int i = 0; i < 10; ++i) F[i] = F2[i];
        if (dn < 1e-28) break;                   // |step| < 1e-14
    }
#pragma unroll
    for (int i = 0; i < 9; ++i) E[i] = Ec[i];
    return fmaxv;
}

// ---- stage B1: reduced rows -> degree-10 polynomial -> roots -----------------------------------
// rec[k * rs]: the stage-A record.  zs[0..count): the real roots (|imag| <= 1e-10) in cv::solvePoly's
// root order.  Returns their number (0 if stage A flagged a singular system; -1: see the template parameter).
// Row j of B(z) comes from reduced rows 4+2j ("e - z f"): the coefficient layout of the right block per
// row is [xz^2 xz x | yz^2 yz y | z^3 z^2 z 1] (descending in z inside each group); entries (j,0),(j,1)
// are cubic, (j,2) quartic, ascending powers.
__device__ __forceinline__ void build_B_row(const double* rec, size_t rs, int j, double (&B)[3][5]) {
    double r1[10], r2[10];
#pragma unroll
    for (int c = 0; c < 10; ++c) {
        r1[c] = rec[(size_t)(36 + (2 * j) * 10 + c) * rs];
        r2[c] = rec[(size_t)(36 + (2 * j + 1) * 10 + c) * rs];
    }
    // group g (x: 0..2, y: 3..5) -> cubic: r1 contributes z^2..z^0, -z*r2 contributes z^3..z^1
#pragma unroll
    for (int g = 0; g < 2; ++g) {
        B[g][0] = r1[3 * g + 2];
        B[g][1] = r1[3 * g + 1] - r2[3 * g + 2];
        B[g][2] = r1[3 * g + 0] - r2[3 * g + 1];
        B[g][3] = -r2[3 * g + 0];
        B[g][4] = 0.0;
    }
    B[2][0] = r1[9];
    B[2][1] = r1[8] - r2[9];
    B[2][2] = r1[7] - r2[8];
    B[2][3] = r1[6] - r2[7];
    B[2][4] = -r2[6];
}

// SLOW = false: the fast path; returns -1 when the roots are not settled (the caller queues the hypothesis for a
// SLOW = true pass, which continues the iteration up to the 300 sweeps OpenCV runs).
// state (DK_STATE doubles, stride ss): written by the fast path when it returns -1, read by the slow pass.
template <bool SLOW>
__device__ __forceinline__ int stage_b1(const double* rec, size_t rs, double (&zs)[10], double* state = nullptr,
                                        size_t ss = 1) {
    if (!(rec[36 * rs] == rec[36 * rs])) return 0;            // stage A flagged a singular system
    double B[3][3][5];
#pragma unroll
    for (int j = 0; j < 3; ++j) build_B_row(rec, rs, j, B[j]);
    double c[11];
    {
        double c3a[4], c3b[4], q4[5], m7a[8], m7b[8], m6a[7], m6b[7], t10[11];
#pragma unroll
        for (int i = 0; i < 11; ++i) c[i] = 0.0;
        // + B00 * (B11*B22 - B12*B21)
#pragma unroll
        for (int i = 0; i < 4; ++i) { c3a[i] = B[1][1][i]; c3b[i] = B[2][1][i]; }
#pragma unroll
        for (int i = 0; i < 5; ++i) q4[i] = B[2][2][i];
        pmul<3, 4>(c3a, q4, m7a);
#pragma unroll
        for (int i = 0; i < 5; ++i) q4[i] = B[1][2][i];
        pmul<3, 4>(c3b, q4, m7b);
#pragma unroll
        for (int i = 0; i < 8; ++i) m7a[i] -= m7b[i];
#pragma unroll
        for (int i = 0; i < 4; ++i) c3a[i] = B[0][0][i];
        pmul<3, 7>(c3a, m7a, t10);
#pragma unroll
        for (int i = 0; i < 11; ++i) c[i] += t10[i];
        // - B01 * (B10*B22 - B12*B20)
#pragma unroll
        for (int i = 0; i < 4; ++i) { c3a[i] = B[1][0][i]; c3b[i] = B[2][0][i]; }
#pragma unroll
        for (int i = 0; i < 5; ++i) q4[i] = B[2][2][i];
        pmul<3, 4>(c3a, q4, m7a);
#pragma unroll
        for (int i = 0; i < 5; ++i) q4[i] = B[1][2][i];
        pmul<3, 4>(c3b, q4, m7b);
#pragma unroll
        for (int i = 0; i < 8; ++i) m7a[i] -= m7b[i];
#pragma unroll
        for (int i = 0; i < 4; ++i) c3a[i] = B[0][1][i];
        pmul<3, 7>(c3a, m7a, t10);
#pragma unroll
        for (int i = 0; i < 11; ++i) c[i] -= t10[i];
        // + B02 * (B10*B21 - B11*B20)
#pragma unroll
        for (int i = 0; i < 4; ++i) { c3a[i] = B[1][0][i]; c3b[i] = B[2][1][i]; }
        pmul<3, 3>(c3a, c3b, m6a);
#pragma unroll
        for (int i = 0; i < 4; ++i) { c3a[i] = B[1][1][i]; c3b[i] = B[2][0][i]; }
        pmul<3, 3>(c3a, c3b, m6b);
#pragma unroll
        for (int i = 0; i < 7; ++i) m6a[i] -= m6b[i];
#pragma unroll
        for (int i = 0; i < 5; ++i) q4[i] = B[0][2][i];
        pmul<4, 6>(q4, m6a, t10);
#pragma unroll
        for (int i = 0; i < 11; ++i) c[i] += t10[i];
    }
    double re[10], im[10];
    int n = 10;
    for (; n > 1; --n)
        if (fabs(c[n]) > 2.220446049250313e-16) break;      // DBL_EPSILON, as cv::solvePoly
    if (n != 10) {
        dk_sweeps_full(c, n, re, im);
    } else if (!SLOW) {
        double prev2;
        if (!dk_sweeps<10>(c, re, im, prev2, 0, state ? DK_FAST_SWEEPS : 300)) {
#pragma unroll
            for (int i = 0; i < 10; ++i) { state[i * ss] = re[i]; state[(10 + i) * ss] = im[i]; }
            state[20 * ss] = prev2;
            return -1;
        }
    } else {
        double prev2 = state[20 * ss];
#pragma unroll
        for (int i = 0; i < 10; ++i) { re[i] = state[i * ss]; im[i] = state[(10 + i) * ss]; }
        dk_sweeps<10>(c, re, im, prev2, DK_FAST_SWEEPS, 300);
    }
    int count = 0;
#pragma unroll
    for (int i = 0; i < 10; ++i) {                           // unrolled: re/im stay in registers
        const bool real = i < n && !(fabs(im[i]) > 1e-10);
#pragma unroll
        for (int k = 0; k < 10; ++k)
            if (k <= i && real && k == count) zs[k] = re[i];  // zs[count] = re[i] with static indices
        count += real ? 1 : 0;
    }
    return count;
}

// ---- stage B2: one real root -> one essential matrix ------------------------------------------
// sh: this thread's scratch in shared memory for the null-space basis (36 doubles, element i at sh[i * ss]).
// E: row-major, unit Frobenius norm, refined.  Returns false if OpenCV would skip this root (the null
// vector of B(z) has a third component below 1e-10) or the refinement did not reach a solution (REFINE_ACCEPT).
__device__ __forceinline__ bool stage_b2(const double* rec, size_t rs, double z, double* sh, int ss, double (&E)[9]) {
    double Bz[3][3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        double B[3][5];
        build_B_row(rec, rs, j, B);
        Bz[j][0] = ((B[0][3] * z + B[0][2]) * z + B[0][1]) * z + B[0][0];
        Bz[j][1] = ((B[1][3] * z + B[1][2]) * z + B[1][1]) * z + B[1][0];
        Bz[j][2] = (((B[2][4] * z + B[2][3]) * z + B[2][2]) * z + B[2][1]) * z + B[2][0];
    }
    double v[3];
    null_vec3(Bz, v);
    if (!(fabs(v[2]) >= 1e-10)) return false;
#pragma unroll
    for (int i = 0; i < 36; ++i) sh[i * ss] = rec[(size_t)i * rs];
    const double iv = 1.0 / v[2];
    const double x = v[0] * iv, y = v[1] * iv;
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
        E[k] = sh[k * ss] * x + sh[(9 + k) * ss] * y + sh[(18 + k) * ss] * z + sh[(27 + k) * ss];
        s += E[k] * E[k];
    }
    const double inv = rsqrt(s);
#pragma unroll
    for (int k = 0; k < 9; ++k) E[k] *= inv;
    return refine_essential(sh, ss, E) <= REFINE_ACCEPT;
}

}  // namespace fivept
