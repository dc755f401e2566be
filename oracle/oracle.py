"""CPU ORACLE -- TEST INFRASTRUCTURE ONLY.

A plain numpy restatement of the per-frame-pair geometric core of Ronnypetson/epivo.  Only
`tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference` leg
may import this package; nothing under `epivo_b200/` does, and the product path fails
loudly if its CUDA library is missing.

What is restated and where parity is pinned
-------------------------------------------
* `Dr_Deps`, `res`, `RepJacobian::compute`, `Levenberg_Marquardt`  -- restated line by line
  from /root/reference/jac_Rt_gen_.cpp (citations on every function).  The reference binary
  cannot be built here (Eigen and Sophus are absent, and the drivers reference an undefined
  `LM_res`), and the reference ships no golden vectors (its demos seed with `time(0)`), so
  the LM restatement is pinned by (i) central finite differences of `res` and (ii) the
  independent single-pair closed form in deprecated/test_jac_Rt.cpp -- see
  tests/test_oracle_lm.py.  PARITY UNPINNED against a running reference binary.
* `BFMatcher::match`, `findEssentialMat`, `recoverPose` are calls into OpenCV, an
  un-vendored dependency with no pinned version (compile_cv:1 `pkg-config opencv`).  They
  are restated from OpenCV's published algorithm (modules/features2d/src/matchers.cpp,
  modules/calib3d/src/{five-point,ptsetreg,triangulate}.cpp, modules/core/src/{rand,
  mathfuncs}.cpp as of 4.x) and pinned against `cv2 4.13.0` in the build container: golden
  vectors under tests/golden/ made by tests/golden/make_golden.py.

Everything is float64 / integer numpy; float32 appears only where OpenCV itself rounds
(the Sampson error and its threshold).
"""
from __future__ import annotations

import math

import numpy as np

NORM_HAMMING = 6      # cv::NORM_HAMMING
NORM_HAMMING2 = 7     # cv::NORM_HAMMING2
RANSAC = 8            # cv::RANSAC
LMEDS = 4             # cv::LMEDS

_POP8 = np.array([bin(i).count("1") for i in range(256)], dtype=np.uint8)
_POP8_H2 = np.array([bin((i | (i >> 1)) & 0x55).count("1") for i in range(256)], dtype=np.uint8)


# ======================================================================================
# M1: BFMatcher(NORM_HAMMING2, crossCheck=true).match          kitti_ba.cpp:602,641
# ======================================================================================

def hamming_matrix(q: np.ndarray, t: np.ndarray, norm: int = NORM_HAMMING2) -> np.ndarray:
    """D[i, j] between uint8 rows; HAMMING2 counts differing 2-bit groups (SURVEY A1)."""
    q = np.ascontiguousarray(q, dtype=np.uint8)
    t = np.ascontiguousarray(t, dtype=np.uint8)
    lut = _POP8 if norm == NORM_HAMMING else _POP8_H2
    D = np.zeros((q.shape[0], t.shape[0]), dtype=np.int32)
    for b in range(q.shape[1]):                     # byte-plane loop keeps memory at nq*nt
        D += lut[q[:, b][:, None] ^ t[:, b][None, :]]
    return D


def bf_match(q, t, norm=NORM_HAMMING2, cross_check=True):
    """`BFMatcher(norm, cross_check).match(q, t)` -> (queryIdx, trainIdx, distance) int32.

    Nearest neighbour = lowest train index among ties; cross-check keeps (i, j) iff j is
    i's NN and i is the NN of j over all queries (first-min on both sides); output sorted by
    queryIdx.
    """
    D = hamming_matrix(q, t, norm)
    if D.shape[0] == 0 or D.shape[1] == 0:
        z = np.zeros(0, dtype=np.int32)
        return z, z.copy(), z.copy()
    nn_q = D.argmin(axis=1)
    qi = np.arange(D.shape[0])
    if cross_check:
        nn_t = D.argmin(axis=0)
        keep = nn_t[nn_q] == qi
        qi, nn_q = qi[keep], nn_q[keep]
    return qi.astype(np.int32), nn_q.astype(np.int32), D[qi, nn_q].astype(np.int32)


def knn2(q, t, norm=NORM_HAMMING):
    """`knnMatch(k=2)`: per query the two smallest by (distance, trainIdx)."""
    D = hamming_matrix(q, t, norm)
    order = np.argsort(D, axis=1, kind="stable")[:, :2]
    d = np.take_along_axis(D, order, axis=1)
    return order.astype(np.int32), d.astype(np.int32)


def ratio_match(q, t, ratio=0.8, norm=NORM_HAMMING):
    """north_star's mode: Lowe ratio on the top-2 (`d1 < ratio * d2`, float32 compare)."""
    idx, d = knn2(q, t, norm)
    if idx.shape[1] < 2:
        z = np.zeros(0, dtype=np.int32)
        return z, z.copy(), z.copy(), z.copy()
    keep = d[:, 0].astype(np.float32) < np.float32(ratio) * d[:, 1].astype(np.float32)
    qi = np.nonzero(keep)[0].astype(np.int32)
    return qi, idx[keep, 0], d[keep, 0], d[keep, 1]


# ======================================================================================
# E1/E2: findEssentialMat                       kitti.cpp:98-104, kitti_E.cpp:98-104
# ======================================================================================

def _two_sum(a, b):
    """Knuth's TwoSum: s = RN(a + b) and the exact error e = a + b - s."""
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def fma_f32_scalar(p: np.ndarray, a: float, b: float) -> np.ndarray:
    """RN(p * a + b) with a single rounding (a fused multiply-add), elementwise, for float64 arrays p whose
    values are float32-representable and float64 scalars a, b (no underflow / overflow).

    Boldo & Melquiond, "Emulation of FMA and correctly rounded sums: proved algorithms using rounding to
    odd" (IEEE TC 2008): with uh + ul = p a exactly and th + tl = b + uh exactly, RN(th + RO(tl + ul)) is
    RN(p a + b).  p a is exact as two products: a = a1 + a2 with a1 the top 29 significant bits of a, so
    p a1 (24 x 29 bits) and p a2 (24 x 24 bits) are both exact doubles."""
    p = np.asarray(p, dtype=np.float64)
    a1 = float((np.array([a], dtype=np.float64).view(np.int64) & ~np.int64((1 << 24) - 1)).view(np.float64)[0])
    a2 = a - a1
    uh, ul = _two_sum(p * a1, p * a2)
    th, tl = _two_sum(np.full_like(p, b), uh)
    v, e = _two_sum(tl, ul)
    # round to odd: where v is inexact and its significand is even, step one ulp towards the exact sum
    even = (v.view(np.int64) & 1) == 0
    fix = (e != 0) & even
    v = np.where(fix, np.nextafter(v, np.where(e > 0, np.inf, -np.inf)), v)
    return th + v


def normalize_points(p: np.ndarray, K: np.ndarray) -> np.ndarray:
    """five-point.cpp findEssentialMat: `points.col(0) = (points.col(0) - cx) / fx`.

    The MatExpr is folded by OpenCV into one scale-and-shift `u * (1/fx) + (-cx * (1/fx))`
    (MatOp_AddEx::multiply) and assigned with `convertTo(col, CV_64F, 1/fx, -cx/fx)`, evaluated in
    float64 on the float32 pixels.  The per-element step of that conversion is FUSED: one rounding of
    `u * (1/fx) + (-cx/fx)`.  Pinned against cv2 4.13.0 (x86-64; its dispatched conversion code is built
    with FMA) by tests/test_oracle_sampson_boundary.py: a strided CV_64F column through `cv2.normalize`'s
    NORM_MINMAX conversion, which is the same `convertTo(alpha, beta)` loop, matches the fused result on
    every pixel where fused and un-fused differ (about half of them with the KITTI K).
    """
    p = np.asarray(p, dtype=np.float32).astype(np.float64).reshape(-1, 2)
    K = np.asarray(K, dtype=np.float64)
    ax, ay = 1.0 / K[0, 0], 1.0 / K[1, 1]
    bx, by = -K[0, 2] * ax, -K[1, 2] * ay
    out = np.empty_like(p)
    out[:, 0] = fma_f32_scalar(p[:, 0], ax, bx)
    out[:, 1] = fma_f32_scalar(p[:, 1], ay, by)
    return out


def sampson_err_f32(E: np.ndarray, x1: np.ndarray, x2: np.ndarray) -> np.ndarray:
    """EMEstimatorCallback::computeError, operation order kept (no FMA contraction).

    err = (float)((x2' E x1)^2 / ((E x1)_0^2 + (E x1)_1^2 + (E' x2)_0^2 + (E' x2)_1^2))
    """
    E = np.asarray(E, dtype=np.float64).reshape(3, 3)
    a1, b1 = x1[:, 0], x1[:, 1]
    a2, b2 = x2[:, 0], x2[:, 1]
    ex0 = (E[0, 0] * a1 + E[0, 1] * b1) + E[0, 2]
    ex1 = (E[1, 0] * a1 + E[1, 1] * b1) + E[1, 2]
    ex2 = (E[2, 0] * a1 + E[2, 1] * b1) + E[2, 2]
    et0 = (E[0, 0] * a2 + E[1, 0] * b2) + E[2, 0]
    et1 = (E[0, 1] * a2 + E[1, 1] * b2) + E[2, 1]
    x2tEx1 = (a2 * ex0 + b2 * ex1) + ex2
    den = ((ex0 * ex0 + ex1 * ex1) + et0 * et0) + et1 * et1
    with np.errstate(divide="ignore", invalid="ignore"):
        return ((x2tEx1 * x2tEx1) / den).astype(np.float32)


def ransac_threshold(thr: float, K: np.ndarray) -> float:
    """`threshold /= (fx + fy) / 2` (five-point.cpp)."""
    K = np.asarray(K, dtype=np.float64)
    return float(thr) / ((K[0, 0] + K[1, 1]) / 2.0)


def find_inliers(err_f32: np.ndarray, thresh: float) -> np.ndarray:
    """ptsetreg.cpp findInliers: `err <= (float)(thresh*thresh)`; mask values {0,1}."""
    return (err_f32 <= np.float32(thresh * thresh)).astype(np.uint8)


def lmeds_median(err_f32: np.ndarray) -> float:
    """ptsetreg.cpp LMeDS: `nth_element(err, err + count/2, err + count); median = err[count/2]`
    -- the upper-middle order statistic for even N (probed against cv2 4.13.0 at small even
    N: the mean-of-two-middle rule of older OpenCV 3.x mis-predicts the mask)."""
    s = np.sort(err_f32)
    return float(s[s.shape[0] // 2])


def lmeds_sigma(median: float, n: int, model_points: int = 5) -> float:
    sigma = 2.5 * 1.4826 * (1 + 5.0 / (n - model_points)) * math.sqrt(median)
    return max(sigma, 0.001)


def ransac_update_num_iters(p: float, ep: float, model_points: int, max_iters: int) -> int:
    """ptsetreg.cpp RANSACUpdateNumIters."""
    p = min(max(p, 0.0), 1.0)
    ep = min(max(ep, 0.0), 1.0)
    dbl_min = 2.2250738585072014e-308
    num = max(1.0 - p, dbl_min)
    denom = 1.0 - (1.0 - ep) ** model_points
    if denom < dbl_min:
        return 0
    num = math.log(num)
    denom = math.log(denom)
    if denom >= 0 or -num >= max_iters * (-denom):
        return max_iters
    return int(np.rint(num / denom))      # cvRound = round-half-even


class CvRNG:
    """cv::RNG (multiply-with-carry), modules/core/include/opencv2/core/operations.hpp."""

    def __init__(self, state: int = 0xFFFFFFFFFFFFFFFF):
        self.state = state & 0xFFFFFFFFFFFFFFFF

    def next(self) -> int:
        self.state = ((self.state & 0xFFFFFFFF) * 4164903690 + (self.state >> 32)) & 0xFFFFFFFFFFFFFFFF
        return self.state & 0xFFFFFFFF

    def uniform(self, a: int, b: int) -> int:
        return a if a == b else self.next() % (b - a) + a


def get_subset(rng: CvRNG, count: int, model_points: int = 5):
    """ptsetreg.cpp getSubset: draw distinct indices, redraw on duplicates."""
    idx = []
    for _ in range(model_points):
        v = rng.uniform(0, count)
        while v in idx:
            v = rng.uniform(0, count)
        idx.append(v)
    return idx


def generate_samples(count: int, m: int, model_points: int = 5) -> np.ndarray:
    """The first m minimal samples OpenCV's RANSAC/LMedS draw for `count` correspondences
    (`RNG rng((uint64)-1)`; the draw sequence does not depend on the data)."""
    rng = CvRNG()
    return np.array([get_subset(rng, count, model_points) for _ in range(m)], dtype=np.int32)


# ---- 5-point minimal solver (five-point.cpp EMEstimatorCallback::runKernel) ----------

# monomials of degree <= 3 in (x, y, z), in the column order of Nister's 10x20 system that
# getCoeffMat fills: x^3 y^3 x^2y xy^2 x^2z x^2 y^2z y^2 xyz xy | xz^2 xz x yz^2 yz y z^3 z^2 z 1
_MONO20 = [(3, 0, 0), (0, 3, 0), (2, 1, 0), (1, 2, 0), (2, 0, 1), (2, 0, 0), (0, 2, 1), (0, 2, 0),
           (1, 1, 1), (1, 1, 0), (1, 0, 2), (1, 0, 1), (1, 0, 0), (0, 1, 2), (0, 1, 1), (0, 1, 0),
           (0, 0, 3), (0, 0, 2), (0, 0, 1), (0, 0, 0)]


def _pmul(a: dict, b: dict) -> dict:
    out: dict = {}
    for ka, va in a.items():
        for kb, vb in b.items():
            k = (ka[0] + kb[0], ka[1] + kb[1], ka[2] + kb[2])
            out[k] = out.get(k, 0.0) + va * vb
    return out


def _padd(a: dict, b: dict, sb: float = 1.0) -> dict:
    out = dict(a)
    for k, v in b.items():
        out[k] = out.get(k, 0.0) + sb * v
    return out


def five_point_constraints(EE: np.ndarray) -> np.ndarray:
    """10x20 coefficient matrix of det(E)=0 and 2 E E'E - tr(E E')E = 0 for
    E = x*EE[0] + y*EE[1] + z*EE[2] + EE[3] (what five-point.cpp getCoeffMat expands)."""
    lin = [(1, 0, 0), (0, 1, 0), (0, 0, 1), (0, 0, 0)]
    Ep = [[{lin[k]: float(EE[k, 3 * i + j]) for k in range(4)} for j in range(3)] for i in range(3)]
    EEt = [[None] * 3 for _ in range(3)]
    for i in range(3):
        for j in range(3):
            acc: dict = {}
            for k in range(3):
                acc = _padd(acc, _pmul(Ep[i][k], Ep[j][k]))
            EEt[i][j] = acc
    tr = _padd(_padd(EEt[0][0], EEt[1][1]), EEt[2][2])
    rows = []
    for i in range(3):
        for j in range(3):
            acc = {}
            for k in range(3):
                lam = EEt[i][k] if i != k else _padd(EEt[i][k], tr, -0.5)
                acc = _padd(acc, _pmul(lam, Ep[k][j]))
            rows.append(acc)
    det = {}
    det = _padd(det, _pmul(Ep[0][0], _padd(_pmul(Ep[1][1], Ep[2][2]), _pmul(Ep[1][2], Ep[2][1]), -1.0)))
    det = _padd(det, _pmul(Ep[0][1], _padd(_pmul(Ep[1][0], Ep[2][2]), _pmul(Ep[1][2], Ep[2][0]), -1.0)), -1.0)
    det = _padd(det, _pmul(Ep[0][2], _padd(_pmul(Ep[1][0], Ep[2][1]), _pmul(Ep[1][1], Ep[2][0]), -1.0)))
    rows.append(det)
    A = np.zeros((10, 20))
    for r, poly in enumerate(rows):
        for c, mono in enumerate(_MONO20):
            A[r, c] = poly.get(mono, 0.0)
    return A



def _eval_B(B, z):
    """B(z) and dB/dz (3x3 each) from the 3x13 coefficient rows (descending powers)."""
    Bz = np.array([[np.polyval(B[j, 0:4], z), np.polyval(B[j, 4:8], z), np.polyval(B[j, 8:13], z)]
                   for j in range(3)])
    dB = np.array([[np.polyval(np.polyder(B[j, 0:4]), z), np.polyval(np.polyder(B[j, 4:8]), z),
                    np.polyval(np.polyder(B[j, 8:13]), z)] for j in range(3)])
    return Bz, dB


def _det3(M):
    return (M[0, 0] * (M[1, 1] * M[2, 2] - M[1, 2] * M[2, 1]) - M[0, 1] * (M[1, 0] * M[2, 2] - M[1, 2] * M[2, 0])
            + M[0, 2] * (M[1, 0] * M[2, 1] - M[1, 1] * M[2, 0]))


def _essential_constraints(E):
    """the ten cubic constraints: 2 E E'E - tr(E E')E (9) and det E (1)"""
    return np.append((2.0 * E @ E.T @ E - np.trace(E @ E.T) * E).ravel(), _det3(E))


def _essential_constraints_dir(E, D):
    """directional derivative of the ten constraints along D"""
    cof = np.array([[E[(i + 1) % 3, (j + 1) % 3] * E[(i + 2) % 3, (j + 2) % 3]
                     - E[(i + 1) % 3, (j + 2) % 3] * E[(i + 2) % 3, (j + 1) % 3] for j in range(3)] for i in range(3)])
    d = 2.0 * (D @ E.T @ E + E @ D.T @ E + E @ E.T @ D) - 2.0 * np.trace(E @ D.T) * E - np.trace(E @ E.T) * D
    return np.append(d.ravel(), float((cof * D).sum()))


REFINE_ACCEPT = 1e-9      # max-abs constraint residual a refined model must reach (unit Frobenius norm)


def refine_essential(E, EE, iters=10):
    """Gauss-Newton refinement of one 5-point solution inside the 4-D null space.

    NOT part of OpenCV's runKernel.  Nister's elimination works in the chart "coefficient of
    EE[3] = 1" of an ARBITRARY null-space basis (OpenCV's comes from LAPACK's SVD, this
    restatement's from numpy's, the CUDA solver's from Householder QR); when a solution has a
    small EE[3] component, or the sample is close to degenerate (low parallax), the expanded
    degree-10 polynomial loses many digits, by an amount that differs from basis to basis.
    A few Newton steps on the constraints themselves, on the unit sphere of coefficients,
    make every implementation converge to the same exact solutions (quadratically: 2-5 steps).
    A step is kept only if it lowers the constraint residual.  Returns (E, final max-abs residual): on a
    near-degenerate sample the iteration can stall far from any solution (1e-5 .. 1e-3); the caller drops
    such a "model" -- it is not an essential matrix."""
    B = EE.reshape(4, 3, 3)
    c = np.array([float((E * B[k]).sum()) for k in range(4)])
    c /= np.linalg.norm(c)
    Ecur = np.tensordot(c, B, 1)
    f = _essential_constraints(Ecur)
    for _ in range(iters):
        J = np.stack([_essential_constraints_dir(Ecur, B[k]) for k in range(4)], axis=1)
        N = J.T @ J
        N = N + 1e3 * np.trace(N) * np.outer(c, c)            # pins the radial (scale) direction
        try:
            d = np.linalg.solve(N, -J.T @ f)
        except np.linalg.LinAlgError:
            break
        c2 = c + d
        c2 /= np.linalg.norm(c2)
        E2 = np.tensordot(c2, B, 1)
        f2 = _essential_constraints(E2)
        if not np.isfinite(f2).all() or np.abs(f2).max() >= np.abs(f).max():
            break
        c, Ecur, f = c2, E2, f2
        if np.linalg.norm(d) < 1e-14:
            break
    return Ecur, float(np.abs(f).max())


def five_point(x1: np.ndarray, x2: np.ndarray, refine: bool = True) -> np.ndarray:
    """EMEstimatorCallback::runKernel on 5 K-normalised correspondences -> (k, 3, 3), k<=10.

    Follows OpenCV's steps: 5x9 epipolar system (row-major E, x2' E x1 = 0), its 4-D null
    space, Nister's 10x20 system reduced by the inverse of its left block, the 3x3
    polynomial matrix B(z) = {rows 4,6,8} - z*{rows 5,7,9}, det B(z) = degree-10 polynomial,
    real roots (|imag| <= 1e-10), (x, y) from the null vector of B(z), skip if its last
    entry is < 1e-10 in magnitude, E normalised to unit Frobenius norm; then, beyond OpenCV,
    each solution is refined on the constraints (refine_essential) unless refine=False.  The null-space
    basis depends on the SVD implementation (OpenCV's comes from LAPACK and is not reproducible
    bit-for-bit); the solutions themselves do not, and they come out in cv::solvePoly's root order.
    """
    x1 = np.asarray(x1, dtype=np.float64)
    x2 = np.asarray(x2, dtype=np.float64)
    Q = np.stack([x2[:, 0] * x1[:, 0], x2[:, 0] * x1[:, 1], x2[:, 0],
                  x2[:, 1] * x1[:, 0], x2[:, 1] * x1[:, 1], x2[:, 1],
                  x1[:, 0], x1[:, 1], np.ones(x1.shape[0])], axis=1)
    _, _, Vt = np.linalg.svd(Q, full_matrices=True)
    EE = Vt[5:9]                                     # 4 x 9 null-space basis
    A = five_point_constraints(EE)
    try:
        A = np.linalg.solve(A[:, :10], A[:, 10:])
    except np.linalg.LinAlgError:
        return np.zeros((0, 3, 3))
    B = np.zeros((3, 13))
    for i in range(3):
        r1, r2 = A[2 * i + 4], A[2 * i + 5]
        row1 = np.zeros(13)
        row2 = np.zeros(13)
        row1[1:4], row1[5:8], row1[9:13] = r1[0:3], r1[3:6], r1[6:10]
        row2[0:3], row2[4:7], row2[8:12] = r2[0:3], r2[3:6], r2[6:10]
        B[i] = row1 - row2
    P = [[np.poly1d(B[i, 0:4]), np.poly1d(B[i, 4:8]), np.poly1d(B[i, 8:13])] for i in range(3)]
    det = (P[0][0] * (P[1][1] * P[2][2] - P[1][2] * P[2][1])
           - P[0][1] * (P[1][0] * P[2][2] - P[1][2] * P[2][0])
           + P[0][2] * (P[1][0] * P[2][1] - P[1][1] * P[2][0]))
    coeffs = np.zeros(11)
    c = det.coeffs
    coeffs[11 - len(c):] = c
    if not (np.abs(coeffs) > np.finfo(float).eps).any():
        return np.zeros((0, 3, 3))
    # cv::solvePoly(coeffs, roots) with its default 300 Durand-Kerner sweeps, restated in C (oracle/poly_c.c):
    # OpenCV's root ORDER fixes the order of a sample's models, and whether a close pair of real roots has
    # settled below |imag| <= 1e-10 after exactly those sweeps fixes which models exist at all
    from . import clib
    roots = clib.solve_poly(coeffs[::-1], 300)
    sols = []
    for r in roots:
        if abs(r.imag) > 1e-10:
            continue
        z = r.real
        Bz = _eval_B(B, z)[0]
        if not np.isfinite(Bz).all():                # degenerate sample (no parallax): no model from this root
            continue
        xy1 = np.linalg.svd(Bz)[2][2]
        if abs(xy1[2]) < 1e-10:
            continue
        x, y = xy1[0] / xy1[2], xy1[1] / xy1[2]
        Ev = EE[0] * x + EE[1] * y + EE[2] * z + EE[3]
        Ev = (Ev / np.linalg.norm(Ev)).reshape(3, 3)
        if refine:
            Ev, resid = refine_essential(Ev, EE)
            if not resid <= REFINE_ACCEPT:
                continue
        sols.append(Ev)
    return np.array(sols).reshape(-1, 3, 3)


def eight_point(x1: np.ndarray, x2: np.ndarray) -> np.ndarray | None:
    """Textbook 8-point on K-normalised points (no reference call site; north_star names it): null vector of the
    8 x 9 epipolar system, projected onto the essential manifold U diag(1,1,0) V', unit Frobenius norm."""
    x1 = np.asarray(x1, dtype=np.float64)
    x2 = np.asarray(x2, dtype=np.float64)
    Q = np.stack([x2[:, 0] * x1[:, 0], x2[:, 0] * x1[:, 1], x2[:, 0],
                  x2[:, 1] * x1[:, 0], x2[:, 1] * x1[:, 1], x2[:, 1],
                  x1[:, 0], x1[:, 1], np.ones(x1.shape[0])], axis=1)
    E0 = np.linalg.svd(Q, full_matrices=True)[2][8].reshape(3, 3)
    U, S, Vt = np.linalg.svd(E0)
    if not S[1] > 1e-12 * S[0]:
        return None
    return U @ np.diag([1.0, 1.0, 0.0]) @ Vt / np.sqrt(2.0)


def score_models(Es: np.ndarray, x1: np.ndarray, x2: np.ndarray, thresh: float | None):
    """K3 known-answer: per model the RANSAC inlier count (if thresh) and the LMedS median."""
    Es = np.asarray(Es, dtype=np.float64).reshape(-1, 3, 3)
    counts = np.zeros(len(Es), dtype=np.int32)
    medians = np.zeros(len(Es), dtype=np.float32)
    for i, E in enumerate(Es):
        err = sampson_err_f32(E, x1, x2)
        if thresh is not None:
            counts[i] = int(find_inliers(err, thresh).sum())
        medians[i] = np.float32(lmeds_median(err))
    return counts, medians


def find_essential_mat(p0, p1, K, method=RANSAC, prob=0.999, thr=1.0, max_iters=1000,
                       samples: np.ndarray | None = None, solver=five_point):
    """cv::findEssentialMat (RANSAC / LMEDS) restated: ptsetreg.cpp run() over the
    deterministic sample stream.  Returns (E 3x3 | None, mask uint8 {0,1}, info dict)."""
    x1 = normalize_points(p0, K)
    x2 = normalize_points(p1, K)
    n = x1.shape[0]
    info = {"iters": 0, "models": 0}
    if n < 5:
        return None, np.zeros(n, dtype=np.uint8), info
    if n == 5:
        Es = solver(x1, x2)
        if len(Es) == 0:
            return None, np.zeros(n, dtype=np.uint8), info
        return Es.reshape(-1, 3), np.ones(n, dtype=np.uint8), info
    t = ransac_threshold(thr, K)
    rng = CvRNG()
    best_E = None
    if method == RANSAC:
        niters = max(max_iters, 1)
        best_count = 0
        best_mask = np.zeros(n, dtype=np.uint8)
        it = 0
        while it < niters:
            idx = get_subset(rng, n) if samples is None else list(samples[it])
            for E in solver(x1[idx], x2[idx]):
                info["models"] += 1
                mask = find_inliers(sampson_err_f32(E, x1, x2), t)
                good = int(mask.sum())
                if good > max(best_count, 4):
                    best_count, best_mask, best_E = good, mask, E
                    niters = ransac_update_num_iters(prob, (n - good) / n, 5, niters)
            it += 1
            if samples is not None and it >= len(samples):
                break
        info["iters"] = it
        if best_count <= 0:
            return None, np.zeros(n, dtype=np.uint8), info
        return best_E, best_mask, info
    # LMEDS
    niters = max(ransac_update_num_iters(prob, 0.45, 5, max_iters), 3)
    if samples is not None:
        niters = min(niters, len(samples))
    min_median = np.inf
    for it in range(niters):
        idx = get_subset(rng, n) if samples is None else list(samples[it])
        for E in solver(x1[idx], x2[idx]):
            info["models"] += 1
            med = lmeds_median(sampson_err_f32(E, x1, x2))
            if med < min_median:
                min_median, best_E = med, E
    info["iters"] = niters
    if best_E is None:
        return None, np.zeros(n, dtype=np.uint8), info
    sigma = lmeds_sigma(min_median, n)
    info["sigma"] = sigma
    info["median"] = min_median
    return best_E, find_inliers(sampson_err_f32(best_E, x1, x2), sigma), info


# ======================================================================================
# P1: recoverPose                                   kitti_E.cpp:120, kitti_ba.cpp:715
# ======================================================================================

def decompose_essential(E: np.ndarray):
    """cv::decomposeEssentialMat: SVD, det sign fix, W, R1 = U W Vt, R2 = U W' Vt, t = U[:,2]."""
    U, _, Vt = np.linalg.svd(np.asarray(E, dtype=np.float64).reshape(3, 3))
    if np.linalg.det(U) < 0:
        U = -U
    if np.linalg.det(Vt) < 0:
        Vt = -Vt
    W = np.array([[0.0, 1.0, 0.0], [-1.0, 0.0, 0.0], [0.0, 0.0, 1.0]])
    return U @ W @ Vt, U @ W.T @ Vt, U[:, 2].copy()


def triangulate_dlt(P0: np.ndarray, P1: np.ndarray, x1: np.ndarray, x2: np.ndarray) -> np.ndarray:
    """cv::triangulatePoints (triangulate.cpp): per point the 4x4 DLT system
    rows x*P[2]-P[0], y*P[2]-P[1] per view; solution = right singular vector of the
    smallest singular value.  Returns (4, N) homogeneous points."""
    n = x1.shape[0]
    out = np.zeros((4, n))
    for i in range(n):
        A = np.stack([x1[i, 0] * P0[2] - P0[0], x1[i, 1] * P0[2] - P0[1],
                      x2[i, 0] * P1[2] - P1[0], x2[i, 1] * P1[2] - P1[1]])
        out[:, i] = np.linalg.svd(A)[2][3]
    return out


def recover_pose(E, p0, p1, K, dist_thresh: float = 50.0, in_mask=None):
    """cv::recoverPose(E, p0, p1, K, R, t, mask) -> (n_good, R, t, mask uint8 {0,255}).

    Candidates in OpenCV's order (R1,t) (R2,t) (R1,-t) (R2,-t); a point is good iff
    Qz*Qw > 0, Qz/Qw < dist, 0 < ([R|t] Q/Qw)_z < dist (and the input mask); the chosen
    candidate is the first whose count is >= all the others.
    """
    x1 = normalize_points(p0, K)
    x2 = normalize_points(p1, K)
    n = x1.shape[0]
    R1, R2, t = decompose_essential(E)
    if np.isnan(R1).any():
        return 0, R1, t, np.zeros(n, dtype=np.uint8)
    cands = [(R1, t), (R2, t), (R1, -t), (R2, -t)]
    P0 = np.hstack([np.eye(3), np.zeros((3, 1))])
    masks = []
    for R, tt in cands:
        P1 = np.hstack([R, tt.reshape(3, 1)])
        Q = triangulate_dlt(P0, P1, x1, x2)
        with np.errstate(divide="ignore", invalid="ignore"):
            m = (Q[2] * Q[3]) > 0
            Qn = Q / Q[3]
            m &= Qn[2] < dist_thresh
            z2 = (P1 @ Qn)[2]
            m &= (z2 > 0) & (z2 < dist_thresh)
        if in_mask is not None:
            m &= np.asarray(in_mask).reshape(-1) != 0
        masks.append(m)
    goods = [int(m.sum()) for m in masks]
    g1, g2, g3, g4 = goods
    if g1 >= g2 and g1 >= g3 and g1 >= g4:
        k = 0
    elif g2 >= g1 and g2 >= g3 and g2 >= g4:
        k = 1
    elif g3 >= g1 and g3 >= g2 and g3 >= g4:
        k = 2
    else:
        k = 3
    R, tt = cands[k]
    return goods[k], R.copy(), tt.copy(), (masks[k].astype(np.uint8) * 255)


# ======================================================================================
# L1-L5: residual, Jacobian, Levenberg-Marquardt                       jac_Rt_gen_.cpp
# ======================================================================================

HUBER_DELTA_SHIPPED = 1e-5      # jac_Rt_gen_.cpp:17
HUBER_DELTA_TESTED = 1.0        # test_jac_Rt_gen.cpp:16

_GEN = np.zeros((6, 4, 4))       # se(3) generators, translation first (jac_Rt_gen_.cpp:46-89)
_GEN[0, 0, 3] = _GEN[1, 1, 3] = _GEN[2, 2, 3] = 1.0
_GEN[3, 1, 2], _GEN[3, 2, 1] = -1.0, 1.0
_GEN[4, 0, 2], _GEN[4, 2, 0] = 1.0, -1.0
_GEN[5, 0, 1], _GEN[5, 1, 0] = -1.0, 1.0


def res(R0, t0, p, p_, huber_delta=HUBER_DELTA_SHIPPED) -> np.ndarray:
    """jac_Rt_gen_.cpp:212-259 -- scalar (already squared, Huberised) cost per correspondence."""
    n = p.shape[0]
    r = np.zeros(n)
    for i in range(n):
        P = np.array([[1.0, 0.0, -p_[i, 0]], [0.0, 1.0, -p_[i, 1]]])
        A = P @ t0                                                    # :238
        B = P @ R0 @ p[i]                                             # :239
        d = 0.0
        nb = np.linalg.norm(B)
        if nb > 0:
            d = np.linalg.norm(A) / nb                                # :242-244
        X_ = R0 @ (p[i] * d) + t0                                     # :248-249
        diff = p_[i] - X_ / X_[2]                                     # :250-252
        ri = float(diff @ diff) / 2.0                                 # :254
        if ri > huber_delta:
            ri = huber_delta * (math.sqrt(ri) - huber_delta / 2.0)    # :255-257
        r[i] = ri
    return r


def dr_deps(Tl0, Tr0, p, p_, reverse: bool, huber_delta=HUBER_DELTA_SHIPPED) -> np.ndarray:
    """jac_Rt_gen_.cpp:23-209 -- N x 6 Jacobian wrt eps of T = Tl0 exp(eps) Tr0 at eps = 0."""
    n = p.shape[0]
    J = np.zeros((n, 6))
    T0 = Tl0 @ Tr0                                                    # :96
    t0, R0 = T0[:3, 3], T0[:3, :3]
    s = -1.0 if reverse else 1.0                                      # :107
    M = np.stack([s * (Tl0 @ _GEN[j] @ Tr0) for j in range(6)])       # :127,142,171
    for i in range(n):
        P = np.array([[1.0, 0.0, -p_[i, 0]], [0.0, 1.0, -p_[i, 1]]])
        A = P @ t0                                                    # :116
        B = P @ R0 @ p[i]                                             # :117
        J_B = np.zeros((2, 6))
        for j in range(3, 6):
            J_B[:, j] = P @ M[j][:3, :3] @ p[i]                       # :125-135
        J_A = P @ np.stack([M[j][:3, 3] for j in range(6)], axis=1)   # :140-145
        ATA, BTB = float(A @ A), float(B @ B)
        if ATA == 0 or BTB == 0:                                      # :152-154
            continue
        sa, sb = math.sqrt(ATA), math.sqrt(BTB)
        J_d = ((1.0 / sa) * sb * (A @ J_A) - (1.0 / sb) * sa * (B @ J_B)) / BTB   # :162
        d0 = np.linalg.norm(A) / np.linalg.norm(B)                    # :164
        Hpd0 = np.append(p[i] * d0, 1.0)                              # :165-166
        J_X = np.stack([(M[j] @ Hpd0)[:3] for j in range(6)], axis=1)  # :169-172
        J_X = J_X + np.outer(R0 @ p[i], J_d)                          # :175-176
        X0 = R0 @ (p[i] * d0) + t0                                    # :178
        z = X0[2]
        J_pi = np.zeros((3, 3))
        if z != 0:                                                    # :182-189
            J_pi = np.array([[1.0 / z, 0.0, -X0[0] / (z * z)],
                             [0.0, 1.0 / z, -X0[1] / (z * z)],
                             [0.0, 0.0, 0.0]])
        e = np.array([X0[0] / z, X0[1] / z, 1.0]) - p_[i]             # :192-196
        JJ = J_pi @ J_X                                               # :191
        if float(e @ e) <= huber_delta:                               # :203-204
            J[i] = (2.0 * e) @ JJ / 2.0
        else:                                                         # :205-207 (reference quirk:
            J[i] = huber_delta * (e / np.linalg.norm(e)) @ JJ         #  sqrt(2) x grad of res)
    return J


def chain_memo(T0s):
    """jac_Rt_gen_.cpp:328-335 -- T0_mem[a][b] = T0s[b] ... T0s[a]  (a <= b)."""
    n = len(T0s)
    mem = {}
    for j in range(n):
        sT = T0s[j]
        mem[(j, j)] = T0s[j]
        for k in range(j + 1, n):
            sT = T0s[k] @ sT
            mem[(j, k)] = sT
    return mem


def rep_jacobian(mem, zeta: int, src: int, tgt: int, p, p_, huber_delta) -> np.ndarray:
    """RepJacobian::compute, jac_Rt_gen_.cpp:262-284."""
    assert (src <= zeta <= tgt) or (tgt <= zeta <= src)               # test_jac_Rt_gen.hpp:28
    Tl0, Tr0 = np.eye(4), np.eye(4)
    reverse = src > tgt
    if src <= tgt:
        if src < zeta:
            Tr0 = mem[(src, zeta - 1)]
        Tl0 = mem[(zeta, tgt)]
    else:
        if src > zeta:
            Tr0 = np.linalg.inv(mem[(zeta + 1, src)])
        Tl0 = np.linalg.inv(mem[(tgt, zeta)])
    return dr_deps(Tl0, Tr0, p, p_, reverse, huber_delta)


def se3_exp(delta) -> np.ndarray:
    """Sophus::SE3<double>::exp(delta).matrix(), delta = (upsilon, omega)  (jac_Rt_gen_.cpp:419)."""
    ups, om = np.asarray(delta[:3], dtype=np.float64), np.asarray(delta[3:], dtype=np.float64)
    th2 = float(om @ om)
    th = math.sqrt(th2)
    Om = np.array([[0, -om[2], om[1]], [om[2], 0, -om[0]], [-om[1], om[0], 0]])
    Om2 = Om @ Om
    if th < 1e-10:
        Rm = np.eye(3) + Om + 0.5 * Om2
        V = Rm                       # Sophus: `V = so3.matrix()` below epsilon = 1e-10 (pinned by oracle/_ref's stand-in)
    else:
        Rm = np.eye(3) + (math.sin(th) / th) * Om + ((1 - math.cos(th)) / th2) * Om2
        V = np.eye(3) + ((1 - math.cos(th)) / th2) * Om + ((th - math.sin(th)) / (th2 * th)) * Om2
    T = np.eye(4)
    T[:3, :3] = Rm
    T[:3, 3] = V @ ups
    return T


def levenberg_marquardt(n_zeta, epsilon, reps, wreps, lambda0, T0s, pr, p_r,
                        huber_delta=HUBER_DELTA_SHIPPED, max_iters=30):
    """jac_Rt_gen_.cpp:287-478.  T0s (n_zeta,4,4) is NOT modified; returns
    (T0s_out, dict(H_norm, r_norm, lambda, iters))."""
    T0s = [np.array(T, dtype=np.float64) for T in T0s]
    n_rep = len(reps)
    N = pr[0].shape[0]
    D = 6 * n_zeta
    lam = lambda0
    prev_E = 1e10
    H = np.zeros((D, D))
    r0 = np.zeros(n_rep * N)
    it_done = 0
    trace = []                                                        # (|delta|, candidate |r0| or None) per iteration
    for _ in range(max_iters):                                        # :323
        it_done += 1
        r0 = np.zeros(n_rep * N)
        J = np.zeros((n_rep * N, D))
        mem = chain_memo(T0s)                                         # :328-335
        for j, (z0, z1) in enumerate(reps):                           # :338-360
            T = mem[(z0, z1)] if z0 <= z1 else np.linalg.inv(mem[(z1, z0)])
            r0[j * N:(j + 1) * N] = wreps[j] * res(T[:3, :3], T[:3, 3], pr[j], p_r[j], huber_delta)
        for j, (z0, z1) in enumerate(reps):                           # :363-399
            lo, hi = (z0, z1) if z0 <= z1 else (z1, z0)
            for k in range(lo, hi + 1):
                Jz = rep_jacobian(mem, k, z0, z1, pr[j], p_r[j], huber_delta)
                J[j * N:(j + 1) * N, 6 * k:6 * k + 6] = wreps[j] * Jz
        b = J.T @ r0                                                  # :401
        H = J.T @ J                                                   # :402
        H = H + lam * np.diag(np.diag(H))                             # :403
        try:
            with np.errstate(all="ignore"):
                delta = -np.linalg.inv(H) @ b                         # :405
        except np.linalg.LinAlgError:
            delta = np.full(D, np.nan)
        trace.append((float(np.linalg.norm(delta)), None))
        if np.isnan(delta).any():                                     # :407-410
            break
        if np.linalg.norm(delta) < epsilon:                           # :412-414
            break
        T0s_ = [T0s[j] @ se3_exp(delta[6 * j:6 * j + 6]) for j in range(len(T0s))]   # :416-422
        for j, (z0, z1) in enumerate(reps):                           # :425-454
            T = np.eye(4)
            if z0 <= z1:
                for k in range(z0, z1 + 1):
                    T = T0s_[k] @ T
            else:
                for k in range(z0, z1 - 1, -1):
                    T = np.linalg.inv(T0s_[k]) @ T
            r0[j * N:(j + 1) * N] = res(T[:3, :3], T[:3, 3], pr[j], p_r[j], huber_delta)
        curr_E = float(np.linalg.norm(r0))                            # :456
        trace[-1] = (trace[-1][0], curr_E)
        if curr_E < prev_E:                                           # :457-467
            prev_E = curr_E
            T0s = T0s_
            lam /= 2.0
        else:
            lam *= 5.0
    out = {"H_norm": float(np.linalg.norm(H)), "r_norm": float(np.linalg.norm(r0)),
           "lambda": float(lam), "iters": it_done, "trace": trace}    # :473-475
    return np.stack(T0s), out


def single_pair_jacobian_closed_form(R0, t0, p, p_):
    """Independent statement of the same Jacobian for one pair (Tl0 = T0, Tr0 = I, no Huber),
    after deprecated/test_jac_Rt.cpp:12-222 (update T0 <- T0 exp(eps)): used only as a
    differential check of `dr_deps` in the tests."""
    n = p.shape[0]
    J = np.zeros((n, 6))
    for i in range(n):
        P = np.array([[1.0, 0.0, -p_[i, 0]], [0.0, 1.0, -p_[i, 1]]])
        A, B = P @ t0, P @ R0 @ p[i]
        na, nb = np.linalg.norm(A), np.linalg.norm(B)
        d = na / nb
        dt = R0                                          # d t / d upsilon
        dRp = -R0 @ _hat(p[i])                           # d (R p) / d omega
        dA = np.hstack([P @ dt, np.zeros((2, 3))])
        dB = np.hstack([np.zeros((2, 3)), P @ dRp])
        dd = (A @ dA) / (na * nb) - na * (B @ dB) / nb ** 3
        X = R0 @ (p[i] * d) + t0
        dX = np.hstack([dt, d * dRp]) + np.outer(R0 @ p[i], dd)
        z = X[2]
        Jpi = np.array([[1 / z, 0, -X[0] / z ** 2], [0, 1 / z, -X[1] / z ** 2]])
        e = X[:2] / z - p_[i, :2]
        J[i] = e @ Jpi @ dX
    return J


def _hat(v):
    return np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])
