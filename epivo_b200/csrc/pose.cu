// K4: fused cv::recoverPose -- decomposeEssentialMat + 4x DLT triangulation of every
// correspondence + cheirality/distance tests + candidate selection, one CTA per pair.
//
// Replaces kitti_E.cpp:120, euroc_E.cpp:251, kitti_ba.cpp:245,322,715.  OpenCV
// (modules/calib3d/src/five-point.cpp recoverPose, triangulate.cpp) runs four passes of a
// per-point 4x4 SVD; here each thread triangulates its correspondences against the four
// (R, t) candidates in registers and only a 4-bit flag per point leaves the thread.
//   E = U diag(s) V'  (V from the Jacobi eigen-decomposition of E'E, U = E V / s,
//                      third columns by cross product so det U = det V = +1)
//   R1 = U W V', R2 = U W' V', t = U[:,2];  candidates (R1,t) (R2,t) (R1,-t) (R2,-t)
//   Q = smallest right singular vector of the DLT matrix (inverse iteration on A'A from the
//       first camera's exact ray; cyclic Jacobi only if that does not converge)
//   good = Qz*Qw > 0 && Qz/Qw < d && 0 < ([R|t] Q/Qw)_z < d   [&& input mask]
//   winner = first candidate whose count is >= all the others; mask values {0,255}.
#include "common.cuh"
#include "stages.cuh"

namespace {

constexpr int PS_THREADS = 128;
constexpr int PS_MINBLOCKS = 4;

// Cyclic Jacobi eigen-decomposition of a symmetric NxN matrix (N = 3, 4): A -> diag, V = eigenvectors (columns)
template <int N>
__device__ __forceinline__ void jacobi_eig(double (&A)[N][N], double (&V)[N][N]) {
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) V[i][j] = (i == j) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 30; ++sweep) {
        double off = 0.0, diag = 0.0;
#pragma unroll
        for (int i = 0; i < N; ++i) {
            diag += A[i][i] * A[i][i];
#pragma unroll
            for (int j = i + 1; j < N; ++j) off += A[i][j] * A[i][j];
        }
        if (off <= 1e-34 * diag || off == 0.0) break;
#pragma unroll
        for (int p = 0; p < N - 1; ++p) {
#pragma unroll
            for (int q = p + 1; q < N; ++q) {
                const double apq = A[p][q];
                if (apq == 0.0) continue;
                const double theta = (A[q][q] - A[p][p]) / (2.0 * apq);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
#pragma unroll
                for (int k = 0; k < N; ++k) {                 // A <- A J
                    const double akp = A[k][p], akq = A[k][q];
                    A[k][p] = c * akp - s * akq;
                    A[k][q] = s * akp + c * akq;
                }
#pragma unroll
                for (int k = 0; k < N; ++k) {                 // A <- J' A
                    const double apk = A[p][k], aqk = A[q][k];
                    A[p][k] = c * apk - s * aqk;
                    A[q][k] = s * apk + c * aqk;
                }
#pragma unroll
                for (int k = 0; k < N; ++k) {
                    const double vkp = V[k][p], vkq = V[k][q];
                    V[k][p] = c * vkp - s * vkq;
                    V[k][q] = s * vkp + c * vkq;
                }
            }
        }
    }
}

__device__ void decompose_essential(const double* E, double (&R1)[9], double (&R2)[9], double (&t)[3]) {
    double M[3][3], V[3][3];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) M[i][j] = E[0 * 3 + i] * E[0 * 3 + j] + E[1 * 3 + i] * E[1 * 3 + j] + E[2 * 3 + i] * E[2 * 3 + j];
    jacobi_eig<3>(M, V);
    // order eigenvalues descending
    int o[3] = {0, 1, 2};
    double ev[3] = {M[0][0], M[1][1], M[2][2]};
    for (int i = 0; i < 2; ++i)
        for (int j = 0; j < 2 - i; ++j)
            if (ev[o[j]] < ev[o[j + 1]]) { int tmp = o[j]; o[j] = o[j + 1]; o[j + 1] = tmp; }
    double v[3][3], u[3][3];   // v[k] = k-th right singular vector, u[k] = k-th left
    for (int k = 0; k < 2; ++k) {
        for (int i = 0; i < 3; ++i) v[k][i] = V[i][o[k]];
    }
    v[2][0] = v[0][1] * v[1][2] - v[0][2] * v[1][1];
    v[2][1] = v[0][2] * v[1][0] - v[0][0] * v[1][2];
    v[2][2] = v[0][0] * v[1][1] - v[0][1] * v[1][0];
    for (int k = 0; k < 2; ++k) {
        double w[3], nn = 0.0;
        for (int i = 0; i < 3; ++i) {
            w[i] = E[i * 3 + 0] * v[k][0] + E[i * 3 + 1] * v[k][1] + E[i * 3 + 2] * v[k][2];
            nn += w[i] * w[i];
        }
        const double inv = nn > 0 ? 1.0 / sqrt(nn) : 0.0;
        for (int i = 0; i < 3; ++i) u[k][i] = w[i] * inv;
    }
    {   // re-orthogonalise u1 against u0 (exact for a true essential matrix, a guard otherwise)
        const double d = u[0][0] * u[1][0] + u[0][1] * u[1][1] + u[0][2] * u[1][2];
        double nn = 0.0;
        for (int i = 0; i < 3; ++i) { u[1][i] -= d * u[0][i]; nn += u[1][i] * u[1][i]; }
        const double inv = nn > 0 ? 1.0 / sqrt(nn) : 0.0;
        for (int i = 0; i < 3; ++i) u[1][i] *= inv;
    }
    u[2][0] = u[0][1] * u[1][2] - u[0][2] * u[1][1];
    u[2][1] = u[0][2] * u[1][0] - u[0][0] * u[1][2];
    u[2][2] = u[0][0] * u[1][1] - u[0][1] * u[1][0];
    // U W = [-u1, u0, u2], U W' = [u1, -u0, u2]
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            const double a = u[0][i] * v[1][j] - u[1][i] * v[0][j];
            const double b = u[2][i] * v[2][j];
            R1[i * 3 + j] = a + b;
            R2[i * 3 + j] = -a + b;
        }
    for (int i = 0; i < 3; ++i) t[i] = u[2][i];
}

// Slow, always-convergent path: cyclic Jacobi on the full 4x4 normal matrix.
__device__ __noinline__ void smallest_eigvec4_jacobi(const double* m10, double* Q) {
    double M[4][4], V[4][4];
    int e = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = i; j < 4; ++j) {
            M[i][j] = m10[e];
            M[j][i] = m10[e];
            ++e;
        }
    jacobi_eig<4>(M, V);
    int k = 0;
    double best = M[0][0];
#pragma unroll
    for (int i = 1; i < 4; ++i)
        if (M[i][i] < best) { best = M[i][i]; k = i; }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        double v = V[i][0];
        if (k == 1) v = V[i][1];
        if (k == 2) v = V[i][2];
        if (k == 3) v = V[i][3];
        Q[i] = v;
    }
}

// Cheirality / distance tests of one correspondence against the candidates [R | t] AND [R | -t].
// The DLT matrix of -t is that of +t with its fourth column negated, so its smallest right
// singular vector is the same vector with W negated (exactly, IEEE arithmetic being
// sign-symmetric): one eigenvector solve serves both candidates.  Returns bit 0 = (R,t), bit 1 = (R,-t).
__device__ __forceinline__ unsigned triangulate_good2(const double* R, const double* t, double a1, double b1,
                                                      double a2, double b2, double dist) {
    // DLT rows (triangulate.cpp): x*P[2] - P[0], y*P[2] - P[1] for P0 = [I|0], P1 = [R|t]:
    //   (-1, 0, a1, 0), (0, -1, b1, 0), r2 = a2*P1[2] - P1[0], r3 = b2*P1[2] - P1[1]
    const double r2[4] = {a2 * R[6] - R[0], a2 * R[7] - R[1], a2 * R[8] - R[2], a2 * t[2] - t[0]};
    const double r3[4] = {b2 * R[6] - R[3], b2 * R[7] - R[4], b2 * R[8] - R[5], b2 * t[2] - t[1]};
    // M = A'A, upper triangle in row order: 00 01 02 03 11 12 13 22 23 33
    double m[10];
    m[0] = 1.0 + (r2[0] * r2[0] + r3[0] * r3[0]);
    m[1] = r2[0] * r2[1] + r3[0] * r3[1];
    m[2] = (r2[0] * r2[2] + r3[0] * r3[2]) - a1;
    m[3] = r2[0] * r2[3] + r3[0] * r3[3];
    m[4] = 1.0 + (r2[1] * r2[1] + r3[1] * r3[1]);
    m[5] = (r2[1] * r2[2] + r3[1] * r3[2]) - b1;
    m[6] = r2[1] * r2[3] + r3[1] * r3[3];
    m[7] = (a1 * a1 + b1 * b1) + (r2[2] * r2[2] + r3[2] * r3[2]);
    m[8] = r2[2] * r2[3] + r3[2] * r3[3];
    m[9] = r2[3] * r2[3] + r3[3] * r3[3];
    // The smallest right singular vector of A = eigenvector of M for its smallest eigenvalue, by
    // inverse iteration on M + mu I = L D L' (same eigenvectors; the shift only keeps the
    // factorisation finite when the point is noise-free and M is singular to working precision).
    // Start: the least-squares solution inside the subspace X = a1 Z, Y = b1 Z that the first
    // camera's two rows span exactly; it is within the pixel noise of the answer, so the
    // iteration contracts by lambda1/lambda2 (~1e-3 .. 1e-6) per step from ~1e-3.
    const double mu = 1e-15 * ((m[0] + m[4]) + (m[7] + m[9]));
    const double d0 = m[0] + mu, i0 = 1.0 / d0;
    const double l10 = m[1] * i0, l20 = m[2] * i0, l30 = m[3] * i0;
    const double d1 = (m[4] + mu) - l10 * m[1], i1 = 1.0 / d1;
    const double u21 = m[5] - l20 * m[1], u31 = m[6] - l30 * m[1];
    const double l21 = u21 * i1, l31 = u31 * i1;
    const double d2 = ((m[7] + mu) - l20 * m[2]) - l21 * u21, i2 = 1.0 / d2;
    const double u32 = (m[8] - l30 * m[2]) - l31 * u21;
    const double l32 = u32 * i2;
    double d3 = (((m[9] + mu) - l30 * m[3]) - l31 * u31) - l32 * u32;
    if (d3 == 0.0) d3 = 1e-300;
    const double i3 = 1.0 / d3;
    const double c2 = (r2[0] * a1 + r2[1] * b1) + r2[2], c3 = (r3[0] * a1 + r3[1] * b1) + r3[2];
    double Q[4];
    {
        const double z = -(c2 * r2[3] + c3 * r3[3]), w = c2 * c2 + c3 * c3;
        Q[0] = a1 * z; Q[1] = b1 * z; Q[2] = z; Q[3] = w;
    }
    bool converged = false;
#pragma unroll 1
    for (int it = 0; it < 12; ++it) {
        // y = (L D L')^-1 Q
        const double f0 = Q[0];
        const double f1 = Q[1] - l10 * f0;
        const double f2 = (Q[2] - l20 * f0) - l21 * f1;
        const double f3 = ((Q[3] - l30 * f0) - l31 * f1) - l32 * f2;
        const double y3 = f3 * i3;
        const double y2 = f2 * i2 - l32 * y3;
        const double y1 = (f1 * i1 - l21 * y2) - l31 * y3;
        const double y0 = ((f0 * i0 - l10 * y1) - l20 * y2) - l30 * y3;
        // y parallel to Q?  component-wise y (Q.Q) - Q (Q.y): no cancellation below round-off
        const double qq = (Q[0] * Q[0] + Q[1] * Q[1]) + (Q[2] * Q[2] + Q[3] * Q[3]);
        const double qy = (Q[0] * y0 + Q[1] * y1) + (Q[2] * y2 + Q[3] * y3);
        const double yy = (y0 * y0 + y1 * y1) + (y2 * y2 + y3 * y3);
        const double e0 = y0 * qq - Q[0] * qy, e1 = y1 * qq - Q[1] * qy, e2 = y2 * qq - Q[2] * qy,
                     e3 = y3 * qq - Q[3] * qy;
        const double err2 = (e0 * e0 + e1 * e1) + (e2 * e2 + e3 * e3);
        // rescale by a power of two near 1/|y|_inf to stay in range (exact, direction unchanged)
        const double big = fmax(fmax(fabs(y0), fabs(y1)), fmax(fabs(y2), fabs(y3)));
        // sc = 2^-floor(log2 big), assembled from the exponent field (big = 0 gives a harmless 2^1023)
        const double sc = __hiloint2double(0x7FE00000 - (__double2hiint(big) & 0x7FF00000), 0);
        Q[0] = y0 * sc; Q[1] = y1 * sc; Q[2] = y2 * sc; Q[3] = y3 * sc;
        // |sin angle(y, Q)|^2 = err2 / (qq^2 yy): converged once a step moves the direction by
        // < 2e-15 (the new iterate is then better than that by the contraction factor)
        if (err2 <= 4e-30 * (qq * qq) * yy) { converged = true; break; }
        if (!(big == big) || big > 1e300) break;
    }
    if (!converged) smallest_eigvec4_jacobi(m, Q);
    const double zw = Q[2] * Q[3];
    const double X = Q[0] / Q[3], Y = Q[1] / Q[3], Z = Q[2] / Q[3];
    const double rz = (R[6] * X + R[7] * Y) + R[8] * Z;
    // +t: point (X, Y, Z), second-camera depth rz + t2
    const double z2p = rz + t[2];
    const bool gp = (zw > 0) && (Z < dist) && (z2p > 0) && (z2p < dist);
    // -t: W -> -W, i.e. point (-X, -Y, -Z), second-camera depth -rz - t2
    const double z2n = (-rz) + (-t[2]);
    const bool gn = (-zw > 0) && (-Z < dist) && (z2n > 0) && (z2n < dist);
    return (gp ? 1u : 0u) | (gn ? 2u : 0u);
}

__global__ void __launch_bounds__(PS_THREADS, PS_MINBLOCKS) pose_kernel(PosePlan p) {
    __shared__ double s_R[2][9];
    __shared__ double s_t[3];
    __shared__ int s_cnt[4];
    __shared__ int s_choice;
    const int pair = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const int n = p.n[pair];
    const bool skip = p.skip && p.skip[pair] != 0;
    uint8_t* mask = p.mask + (int64_t)pair * p.stride;
    if (skip) {
        if (tid < 9) p.R[(int64_t)pair * 9 + tid] = 0.0;
        if (tid < 3) p.t[(int64_t)pair * 3 + tid] = 0.0;
        if (tid == 0) p.n_good[pair] = 0;
        for (int i = tid; i < n; i += PS_THREADS) mask[i] = 0;
        return;
    }
    if (tid == 0) {
        double R1[9], R2[9], t[3];
        decompose_essential(p.E + (int64_t)pair * 9, R1, R2, t);
        for (int i = 0; i < 9; ++i) { s_R[0][i] = R1[i]; s_R[1][i] = R2[i]; }
        for (int i = 0; i < 3; ++i) s_t[i] = t[i];
    }
    if (tid < 4) s_cnt[tid] = 0;
    __syncthreads();
    const double* X1 = p.xn + (int64_t)pair * 4 * p.stride;
    const double* Y1 = X1 + p.stride;
    const double* X2 = Y1 + p.stride;
    const double* Y2 = X2 + p.stride;
    const uint8_t* im = p.in_mask ? p.in_mask + (int64_t)pair * p.stride : nullptr;
    const double tp[3] = {s_t[0], s_t[1], s_t[2]};
    int c0 = 0, c1 = 0, c2 = 0, c3 = 0;
    for (int i = tid; i < n; i += PS_THREADS) {
        const double a1 = X1[i], b1 = Y1[i], a2 = X2[i], b2 = Y2[i];
        unsigned f = 0;
        if (!im || im[i]) {
            const unsigned g1 = triangulate_good2(s_R[0], tp, a1, b1, a2, b2, p.dist_thresh);   // (R1, +-t)
            const unsigned g2 = triangulate_good2(s_R[1], tp, a1, b1, a2, b2, p.dist_thresh);   // (R2, +-t)
            f = (g1 & 1u) | ((g2 & 1u) << 1) | ((g1 & 2u) << 1) | ((g2 & 2u) << 2);
        }
        mask[i] = (uint8_t)f;
        c0 += f & 1; c1 += (f >> 1) & 1; c2 += (f >> 2) & 1; c3 += (f >> 3) & 1;
    }
    c0 = __reduce_add_sync(0xFFFFFFFFu, c0);
    c1 = __reduce_add_sync(0xFFFFFFFFu, c1);
    c2 = __reduce_add_sync(0xFFFFFFFFu, c2);
    c3 = __reduce_add_sync(0xFFFFFFFFu, c3);
    if (lane == 0) {
        atomicAdd(&s_cnt[0], c0); atomicAdd(&s_cnt[1], c1); atomicAdd(&s_cnt[2], c2); atomicAdd(&s_cnt[3], c3);
    }
    __syncthreads();
    if (tid == 0) {
        const int g1 = s_cnt[0], g2 = s_cnt[1], g3 = s_cnt[2], g4 = s_cnt[3];
        int k;
        if (g1 >= g2 && g1 >= g3 && g1 >= g4) k = 0;
        else if (g2 >= g1 && g2 >= g3 && g2 >= g4) k = 1;
        else if (g3 >= g1 && g3 >= g2 && g3 >= g4) k = 2;
        else k = 3;
        s_choice = k;
        p.n_good[pair] = s_cnt[k];
    }
    __syncthreads();
    const int k = s_choice;
    if (tid < 9) p.R[(int64_t)pair * 9 + tid] = s_R[k & 1][tid];
    if (tid < 3) p.t[(int64_t)pair * 3 + tid] = (k & 2) ? -s_t[tid] : s_t[tid];
    for (int i = tid; i < n; i += PS_THREADS) mask[i] = ((mask[i] >> k) & 1) ? 255 : 0;   // own writes only
}

// ---- 8-point hypotheses (north_star: "each warp solves one minimal 5-point (and 8-point) hypothesis") ----------------
// The reference never calls an 8-point solver (every findEssentialMat call site runs OpenCV's 5-point estimator,
// SURVEY section 0 M6), so this is the textbook algorithm, offered next to epivo_five_point for hypothesis generation
// and scored by the same K3 (epivo_score_sampson):
//   A (8 x 9), row = (x2 x1, x2 y1, x2, y2 x1, y2 y1, y2, x1, y1, 1) on K-normalised points  ->  null vector
//   (Householder QR of A': the last column of Q)  ->  E0 (row-major)  ->  nearest essential matrix
//   E = U diag(1, 1, 0) V' (V from the Jacobi eigen-decomposition of E0'E0, U = E0 V / s), unit Frobenius norm.
// One LANE per hypothesis, everything in registers (a warp-per-hypothesis split would idle 24 of 32 lanes on
// 8 x 9 work); ok = 0 when the eight points are degenerate (second singular value of E0 below 1e-12 of the first).
__global__ void __launch_bounds__(128) eight_point_kernel(const double* __restrict__ x1, const double* __restrict__ x2,
                                                          int m, double* __restrict__ E_out, int32_t* __restrict__ ok) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    double A[9][8];                                  // A' : column c = row of correspondence c
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const double a1 = x1[((size_t)i * 8 + c) * 2], b1 = x1[((size_t)i * 8 + c) * 2 + 1];
        const double a2 = x2[((size_t)i * 8 + c) * 2], b2 = x2[((size_t)i * 8 + c) * 2 + 1];
        A[0][c] = a2 * a1; A[1][c] = a2 * b1; A[2][c] = a2;
        A[3][c] = b2 * a1; A[4][c] = b2 * b1; A[5][c] = b2;
        A[6][c] = a1;      A[7][c] = b1;      A[8][c] = 1.0;
    }
    double beta[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {                    // Householder QR; v_k in A[k.., k]
        double s = 0.0;
#pragma unroll
        for (int r = k; r < 9; ++r) s += A[r][k] * A[r][k];
        const double nrm = sqrt(s);
        const double alpha = A[k][k] > 0 ? -nrm : nrm;
        const double v0 = A[k][k] - alpha;
        const double vtv = s - A[k][k] * A[k][k] + v0 * v0;
        beta[k] = vtv > 0 ? 2.0 / vtv : 0.0;
        A[k][k] = v0;
#pragma unroll
        for (int c = k + 1; c < 8; ++c) {
            double d = 0.0;
#pragma unroll
            for (int r = k; r < 9; ++r) d += A[r][k] * A[r][c];
            d *= beta[k];
#pragma unroll
            for (int r = k; r < 9; ++r) A[r][c] -= d * A[r][k];
        }
    }
    double e[9];                                     // Q e_8: the null vector
#pragma unroll
    for (int r = 0; r < 9; ++r) e[r] = (r == 8) ? 1.0 : 0.0;
#pragma unroll
    for (int k = 7; k >= 0; --k) {
        double d = 0.0;
#pragma unroll
        for (int r = k; r < 9; ++r) d += A[r][k] * e[r];
        d *= beta[k];
#pragma unroll
        for (int r = k; r < 9; ++r) e[r] -= d * A[r][k];
    }
    // nearest essential matrix
    double M[3][3], V[3][3];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 3; ++b) M[a][b] = e[a] * e[b] + e[3 + a] * e[3 + b] + e[6 + a] * e[6 + b];   // E0'E0
    jacobi_eig<3>(M, V);
    int o0 = 0, o1 = 1, o2 = 2;                      // eigenvalues in descending order
    if (M[o0][o0] < M[o1][o1]) { const int t = o0; o0 = o1; o1 = t; }
    if (M[o1][o1] < M[o2][o2]) { const int t = o1; o1 = o2; o2 = t; }
    if (M[o0][o0] < M[o1][o1]) { const int t = o0; o0 = o1; o1 = t; }
    const double s0 = sqrt(fmax(M[o0][o0], 0.0)), s1 = sqrt(fmax(M[o1][o1], 0.0));
    const bool good = s1 > 1e-12 * s0 && s0 > 0.0;
    double E[9];
#pragma unroll
    for (int q = 0; q < 9; ++q) E[q] = 0.0;
    if (good) {
#pragma unroll
        for (int which = 0; which < 2; ++which) {
            const int col = which ? o1 : o0;
            const double is = 1.0 / (which ? s1 : s0);
            double v[3], u[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) v[a] = (col == 0) ? V[a][0] : (col == 1 ? V[a][1] : V[a][2]);
#pragma unroll
            for (int a = 0; a < 3; ++a) u[a] = (e[3 * a] * v[0] + e[3 * a + 1] * v[1] + e[3 * a + 2] * v[2]) * is;
#pragma unroll
            for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int b = 0; b < 3; ++b) E[3 * a + b] += u[a] * v[b];
        }
#pragma unroll
        for (int q = 0; q < 9; ++q) E[q] *= 0.70710678118654752440;    // |U diag(1,1,0) V'|_F = sqrt(2)
    }
#pragma unroll
    for (int q = 0; q < 9; ++q) E_out[(size_t)i * 9 + q] = E[q];
    ok[i] = good ? 1 : 0;
}

}  // namespace

int epv_eight_point_launch(epivo_ctx* ctx, const double* d_x1, const double* d_x2, int m, double* d_E, int32_t* d_ok) {
    if (m <= 0) return EPIVO_OK;
    eight_point_kernel<<<(m + 127) / 128, 128, 0, ctx->stream>>>(d_x1, d_x2, m, d_E, d_ok);
    EPV_LAUNCHED(ctx);
    return EPIVO_OK;
}

int epv_pose_launch(epivo_ctx* ctx, const PosePlan& p) {
    if (p.n_pairs <= 0) return EPIVO_OK;
    pose_kernel<<<p.n_pairs, PS_THREADS, 0, ctx->stream>>>(p);
    EPV_LAUNCHED(ctx);
    return EPIVO_OK;
}
