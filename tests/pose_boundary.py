"""recoverPose's per-point decisions at their boundaries, with an exact reference (host only).

pose_kernel (epivo_b200/csrc/pose.cu) calls a correspondence "good" under a candidate (R, t) when the triangulated
point Q = (X, Y, Z, W) passes four tests:

    Qz Qw > 0,   Z = Qz / Qw < dist,   z2 = ([R | t] Q / Qw)_z > 0,   z2 < dist.

It does not compute Q as OpenCV does (an SVD of each point's 4 x 4 DLT matrix): it runs at most 12 steps of shifted
inverse iteration on the normal matrix M = A'A in double, serves (R, t) and (R, -t) from one solve, and falls back to
a cyclic Jacobi on M when the iteration does not converge.  This module gives those decisions an exact reference and
builds inputs that sit on them:

* `decide`: every point's decision per candidate from the DLT matrix of the doubles the kernel receives, solved at
  60 digits, candidates from an exact (60-digit) cv::decomposeEssentialMat.  The (R, -t) candidates get their own DLT
  matrices, so the kernel's sign-symmetry shortcut is checked, not assumed.  A vectorised double pre-pass decides every
  point whose margin is far outside what rounding could move; only the rest go to 60 digits.
* the "decided" rule (applied to every comparison): a decision counts only if it is unchanged under TRIALS random
  perturbations of ULPS double ulps on each normalised coordinate and a relative RHO on every entry of R and t, where
  RHO = max(1e-13, 16 eps s1 / (s3 + s4)) (s = singular values of A).  1e-13 covers the kernel's decomposition of E;
  the second term is the perturbation of A that is worth the kernel's squaring into M = A'A.  Undecided points are
  counted and reported, never compared.
* straddles: for one candidate, two correspondences one float32 pixel ulp apart that the exact reference decides
  differently, found by bisecting on float32 positions:
    - "Z<d":  x1 generic, the point at depth ~ dist; the candidate's t_z < 0 (the second camera is in front, so Z
              reaches dist before z2 does);
    - "z2<d": the same with t_z > 0;
    - "zw":   x2 next to the second image's epipole, x1 generic: the point sits next to the first camera's centre,
              where Z changes sign (t_z > 0 keeps z2 ~ t_z inside (0, dist));
    - "z2>0": x1 next to the first image's epipole: the point sits next to the second camera's centre (t_z < 0).
  The sign of Qw itself (a point crossing infinity) never decides a straddle with finite pixels: next to Qw = 0 the
  depth is ~1e7 or more on both sides, so "Z < dist" is already false on the side where Qz Qw > 0, for every dist
  used here.  The "zw" straddles flip Qz Qw through Qz instead.
* special inputs: noisy correspondences at the epipoles, where the inverse iteration cannot converge in 12 steps
  (`fallback_margin` restates the loop at 60 digits and measures how far it is from converging); an integer-exact E with
  dyadic correspondences, whose M is exactly singular in double; x1 == x2 (and x1 == -x2) under that E, where the
  kernel's start vector is exactly zero; points at infinity; NaN and +-inf pixels.
  The `d3 == 0` guard of the LDL' factorisation is not reached: the shift mu = 1e-15 trace(M) keeps d3 near mu even
  for an exactly singular M, so d3 is zero only if the factorisation's rounding cancels the shift exactly.
* ties: scenes whose points are good under two candidates in equal numbers.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import mpmath
import numpy as np

import sampson_boundary as SB
from oracle import oracle as O

POW2_K = SB.POW2_K
PSIZE = SB.IMAGE["pow2"]
KITTI_K = SB.KITTI_K
DISTS = (50.0, 3.0, 1e4)
DPS = 60
EPS = 2.0 ** -52
ULPS = 4
REL_RT = 1e-13
TRIALS = 4
SAFETY = 1e3
INEQ = ("zw", "Z<d", "z2>0", "z2<d")
TIGHT = 2.0 ** -25
W_CV = [[0, 1, 0], [-1, 0, 0], [0, 0, 1]]


# ---- exact decomposition and candidates -------------------------------------------------------------------

@dataclass
class Cands:
    mp: list              # 4 x (R 3x3, t 3x1) mpmath matrices, OpenCV's order (R1,t) (R2,t) (R1,-t) (R2,-t)
    f64: list             # the same rounded to double


def candidates(E) -> Cands:
    """cv::decomposeEssentialMat at DPS digits: U, Vt with det +1 (sign flips as OpenCV), R1 = U W Vt, R2 = U W' Vt,
    t = U[:, 2]."""
    with mpmath.workdps(DPS):
        Em = mpmath.matrix([[mpmath.mpf(float(v)) for v in row] for row in np.asarray(E, np.float64).reshape(3, 3)])
        U, _, Vt = mpmath.svd_r(Em)                  # singular values in descending order
        if mpmath.det(U) < 0:
            U = -U
        if mpmath.det(Vt) < 0:
            Vt = -Vt
        W = mpmath.matrix(W_CV)
        R1, R2, t = U * W * Vt, U * W.T * Vt, U[:, 2]
        mp = [(R1, t), (R2, t), (R1, -t), (R2, -t)]
        f64 = [(np.array(R.tolist(), dtype=np.float64), np.array(tt.tolist(), dtype=np.float64).reshape(3))
               for R, tt in mp]
    return Cands(mp, f64)


def match_candidate(C: Cands, R, t) -> int:
    """the index of the exact candidate a kernel's (R, t) stands for (both to 1e-6)"""
    R = np.asarray(R, np.float64).reshape(3, 3)
    t = np.asarray(t, np.float64).reshape(3)
    hits = [c for c, (Rc, tc) in enumerate(C.f64) if np.abs(Rc - R).max() < 1e-6 and np.abs(tc - t).max() < 1e-6]
    assert len(hits) == 1, (R, t)
    return hits[0]


# ---- the DLT matrix, the four tests as linear forms ---------------------------------------------------------

def _dlt(x, R, t):
    """(n, 4, 4) DLT matrices of triangulate.cpp for P0 = [I | 0], P1 = [R | t] (rows x P[2] - P[0], y P[2] - P[1])"""
    n = len(x)
    A = np.zeros((n, 4, 4))
    A[:, 0, 0] = A[:, 1, 1] = -1.0
    A[:, 0, 2], A[:, 1, 2] = x[:, 0], x[:, 1]
    for r, (c, i) in enumerate(((x[:, 2], 0), (x[:, 3], 1))):
        A[:, 2 + r, :3] = c[:, None] * R[2][None] - R[i][None]
        A[:, 2 + r, 3] = c * t[2] - t[i]
    return A


def _forms(R, t, dist):
    """(4, 4) rows L with: test j passes  <=>  (L_j . Q) Qw > 0  (Qw != 0)"""
    r = np.asarray(R)[2]
    return np.array([[0.0, 0.0, 1.0, 0.0],
                     [0.0, 0.0, -1.0, dist],
                     [r[0], r[1], r[2], t[2]],
                     [-r[0], -r[1], -r[2], dist - t[2]]])


def _tests_mp(x, R, t, dist):
    """the four tests, exactly: Q = eigenvector of A'A for its smallest eigenvalue at DPS digits"""
    with mpmath.workdps(DPS):
        a1, b1, a2, b2 = (mpmath.mpf(float(v)) for v in x)
        A = mpmath.matrix([[-1, 0, a1, 0], [0, -1, b1, 0],
                           [a2 * R[2, 0] - R[0, 0], a2 * R[2, 1] - R[0, 1], a2 * R[2, 2] - R[0, 2], a2 * t[2] - t[0]],
                           [b2 * R[2, 0] - R[1, 0], b2 * R[2, 1] - R[1, 1], b2 * R[2, 2] - R[1, 2], b2 * t[2] - t[1]]])
        ev, V = mpmath.eigsy(A.T * A)
        k = min(range(4), key=lambda i: ev[i])
        Q = [V[i, k] for i in range(4)]
        w = Q[3]
        if w == 0:
            return (False,) * 4
        z2 = R[2, 0] * Q[0] + R[2, 1] * Q[1] + R[2, 2] * Q[2] + t[2] * w
        L = (Q[2], dist * w - Q[2], z2, (dist - t[2]) * w - (z2 - t[2] * w))
        return tuple(bool(l * w > 0) for l in L)


def _mp_rt(R, t):
    with mpmath.workdps(DPS):
        return (mpmath.matrix([[mpmath.mpf(float(v)) for v in row] for row in R]),
                mpmath.matrix([mpmath.mpf(float(v)) for v in t]))


def _ulps(v: float, k: int) -> float:
    for _ in range(abs(k)):
        v = float(np.nextafter(v, math.copysign(math.inf, k)))
    return v


# ---- the exact reference with the decided rule ----------------------------------------------------------------

@dataclass
class Decision:
    good: np.ndarray                  # (n, 4) bool: exact decision per candidate (Cands order)
    decided: np.ndarray               # (n, 4) bool
    C: Cands
    n_exact: int = 0                  # (point, candidate) decisions that went to 60 digits

    def count_bounds(self, c: int):
        """(lowest, highest) possible count of candidate c: decided goods, plus every undecided point"""
        lo = int((self.good[:, c] & self.decided[:, c]).sum())
        return lo, lo + int((~self.decided[:, c]).sum())

    def summary(self, c: int) -> str:
        d = self.decided[:, c]
        return f"{int(d.sum())} decided, {int((~d).sum())} undecided, {self.n_exact} at 60 digits"


def decide(E, x, dist: float, in_mask=None, seed: int = 0, C: Cands | None = None) -> Decision:
    """The exact decision of every correspondence x (n, 4) = (a1, b1, a2, b2), K-normalised doubles, under the four
    candidates of E, with the decided rule.  A non-finite coordinate is no point: never good, always decided.  An input
    mask of 0 makes a point not good, decided."""
    C = C or candidates(E)
    x = np.asarray(x, np.float64).reshape(-1, 4)
    n = len(x)
    rng = np.random.default_rng(seed)
    good = np.zeros((n, 4), bool)
    decided = np.ones((n, 4), bool)
    live = np.isfinite(x).all(1)
    if in_mask is not None:
        live &= np.asarray(in_mask).reshape(-1) != 0
    idx = np.nonzero(live)[0]
    n_exact = 0
    for c, (R, t) in enumerate(C.f64):
        if not len(idx):
            break
        xs = x[idx]
        _, s, Vt = np.linalg.svd(_dlt(xs, R, t))
        Q = Vt[:, 3, :]
        with np.errstate(divide="ignore", invalid="ignore"):
            rho = np.maximum(REL_RT, 16 * EPS * s[:, 0] / (s[:, 2] + s[:, 3]))
            theta = SAFETY * rho * s[:, 0] / (s[:, 2] - s[:, 3])
        theta = np.where(np.isfinite(theta), theta, np.inf)
        L = _forms(R, t, dist)
        v = Q @ L.T
        w = Q[:, 3]
        band = 2 * theta[:, None] * np.linalg.norm(L, axis=1)[None]
        sure = (np.abs(v) > band) & (np.abs(w) > 2 * theta)[:, None]
        passes = v * w[:, None] > 0
        fast_good = (sure & passes).all(1)
        fast_bad = (sure & ~passes).any(1)
        # |Z| > dist for sure: Qz Qw > 0 and Z < dist cannot both hold
        fast_bad |= np.abs(Q[:, 2]) - dist * np.abs(w) > 2 * theta * (1 + dist)
        good[idx, c] = fast_good
        rest = idx[~(fast_good | fast_bad)]
        n_exact += len(rest)
        Rm, tm = C.mp[c]
        for i in rest:
            g0 = all(_tests_mp(x[i], Rm, tm, dist))
            good[i, c] = g0
            r = float(rho[np.searchsorted(idx, i)])
            r = r if np.isfinite(r) else 1e-6
            for _ in range(TRIALS):
                xp = [_ulps(float(v), int(k)) for v, k in zip(x[i], rng.integers(-ULPS, ULPS + 1, 4))]
                Rp = R * (1 + r * rng.uniform(-1, 1, (3, 3)))
                tp = t * (1 + r * rng.uniform(-1, 1, 3))
                if all(_tests_mp(xp, *_mp_rt(Rp, tp), dist)) != g0:
                    decided[i, c] = False
                    break
    return Decision(good, decided, C, n_exact)


def good_f64(x, R, t, dist) -> np.ndarray:
    """the four tests on a double SVD (for searching; every result that matters is re-decided by `decide`)"""
    x = np.asarray(x, np.float64).reshape(-1, 4)
    Q = np.linalg.svd(_dlt(x, R, t))[2][:, 3, :]
    v = Q @ _forms(R, t, dist).T
    return (v * Q[:, 3:4] > 0).all(1)


def tests_exact(x, R, t, dist) -> tuple:
    """the four tests (INEQ order) of one correspondence at DPS digits, for a double candidate"""
    return _tests_mp(x, *_mp_rt(R, t), dist)


# ---- geometry -------------------------------------------------------------------------------------------------

def rotation(w) -> np.ndarray:
    w = np.asarray(w, np.float64)
    th = np.linalg.norm(w)
    if th == 0:
        return np.eye(3)
    k = w / th
    Kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.eye(3) + math.sin(th) * Kx + (1 - math.cos(th)) * Kx @ Kx


def essential(R, t) -> np.ndarray:
    t = np.asarray(t, np.float64)
    E = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]]) @ R
    return E / np.linalg.norm(E)


def motion(seed: int):
    """a small rotation and a unit, mostly forward translation (t_z > 0: the second camera [R | t] is behind the
    first); its mirror (R, -t) has the second camera in front."""
    rng = np.random.default_rng(seed)
    R = rotation(rng.normal(0, 0.04, 3))
    t = np.array([rng.normal(0, 0.15), rng.normal(0, 0.08), 1.0])
    return R, t / np.linalg.norm(t)


def pixels(x2d, K) -> np.ndarray:
    K = np.asarray(K, np.float64)
    return np.stack([x2d[..., 0] * K[0, 0] + K[0, 2], x2d[..., 1] * K[1, 1] + K[1, 2]], -1)


def norm4(p0, p1, K) -> np.ndarray:
    """(n, 4) K-normalised doubles of float32 pixel pairs, as the kernels get them"""
    return np.concatenate([O.normalize_points(p0, K), O.normalize_points(p1, K)], axis=1)


def project(X, R, t):
    Y = X @ R.T + t
    return X[:, :2] / X[:, 2:3], Y[:, :2] / Y[:, 2:3], Y[:, 2]


def clear_points(R, t, dist, n, seed, K=POW2_K, size=PSIZE):
    """n noise-free correspondences (float32 pixels) well inside every test of the candidate (R, t): both depths in
    (0.15, 0.85) dist, both pixels in the image"""
    rng = np.random.default_rng(seed)
    W, H = size
    out0, out1 = [], []
    Kinv = np.linalg.inv(np.asarray(K, np.float64))
    while len(out0) < n:
        p = rng.uniform((20, 20), (W - 20, H - 20), (4 * n, 2))
        Z = rng.uniform(0.15 * dist, 0.85 * dist, 4 * n)
        X = (np.concatenate([p, np.ones((4 * n, 1))], 1) @ Kinv.T) * Z[:, None]
        _, x2, z2 = project(X, R, t)
        q = pixels(x2, K)
        ok = (z2 > 0.15 * dist) & (z2 < 0.85 * dist) & (q >= 0).all(1) & (q < (W, H)).all(1)
        out0 += list(p[ok])
        out1 += list(q[ok])
    return np.array(out0[:n], np.float32), np.array(out1[:n], np.float32)


# ---- straddles ------------------------------------------------------------------------------------------------

@dataclass
class Straddle:
    kind: str                 # the test that flips (INEQ)
    p0: np.ndarray            # (2, 2) float32: first-image pixel of the good, the bad member
    p1: np.ndarray            # (2, 2) float32: second-image pixel of the good, the bad member
    near_epipole: bool


def _f32_step(v: np.float32, k: int) -> np.float32:
    b = int(np.float32(v).view(np.int32)) + k
    return np.array([b], np.int32).view(np.float32)[0]


def _straddle_along(R, t, dist, K, p_fixed, p_var, var_img: int, dirn, near: bool, tight=None):
    """bisect the float32 coordinate of p_var (an image-`var_img` pixel) that moves most along dirn for a flip of
    good_f64; returns the Straddle (exactly re-checked) or None.  tight: keep only a flip whose good member lies
    within a relative `tight` of dist in the depth that flips"""
    j = int(np.argmax(np.abs(dirn)))
    base = np.asarray(p_var, np.float32).copy()

    def at(k):
        q = base.copy()
        q[j] = _f32_step(base[j], k)
        return q

    def pair(k):
        q = at(k)
        return (p_fixed, q) if var_img == 1 else (q, p_fixed)

    def dec(k):
        a, b = pair(k)
        return bool(good_f64(norm4(a[None], b[None], K), R, t, dist)[0])

    k = SB._bracket(dec, 1 << 22)
    if k is None:
        return None
    (a0, b0), (a1, b1) = pair(k), pair(k + 1)
    x0, x1 = norm4(a0[None], b0[None], K)[0], norm4(a1[None], b1[None], K)[0]
    if tight is not None:
        xg = x0 if dec(k) else x1
        Q = np.linalg.svd(_dlt(xg[None], R, t))[2][0, 3]
        depths = (Q[2] / Q[3], (R[2] @ Q[:3]) / Q[3] + t[2])
        if not any(0 < dist - d < tight * dist for d in depths):
            return None
    t0, t1 = tests_exact(x0, R, t, dist), tests_exact(x1, R, t, dist)
    if all(t0) == all(t1):
        return None
    if all(t1):
        (a0, b0), (a1, b1), t0, t1 = (a1, b1), (a0, b0), t1, t0
    flipped = [INEQ[i] for i in range(4) if t0[i] != t1[i]]
    if len(flipped) != 1:
        return None
    return Straddle(flipped[0], np.stack([a0, a1]).astype(np.float32), np.stack([b0, b1]).astype(np.float32), near)


def straddles(R, t, dist, count: int, seed: int, K=POW2_K, size=PSIZE, epipole: int = 0, tight=None) -> list[Straddle]:
    """straddles of the candidate (R, t): `count` of the depth kind ("z2<d" if t_z > 0, else "Z<d") and `epipole` of
    the epipole kind ("zw" next to the second image's epipole if t_z > 0, else "z2>0" next to the first image's).
    tight: depth straddles whose good member is within a relative `tight` below dist (TIGHT: dist - depth is below
    half a float32 ulp of dist, so the depth rounded to float would compare equal to dist)"""
    rng = np.random.default_rng(seed)
    W, H = size
    K = np.asarray(K, np.float64)
    Kinv = np.linalg.inv(K)
    out: list[Straddle] = []
    tries = 0
    while sum(not s.near_epipole for s in out) < count:
        tries += 1
        assert tries < (50 if tight is None else 20000) * count + 50
        p0 = rng.uniform((20, 20), (W - 20, H - 20)).astype(np.float32)
        x1h = Kinv @ np.array([p0[0], p0[1], 1.0])
        rz = (R @ x1h)[2]
        lam = dist if t[2] < 0 else (dist - t[2]) / rz          # Z = dist, or z2 = dist
        if not lam > 0:
            continue
        X = np.array([lam * x1h, lam * 1.001 * x1h])
        _, x2, z2 = project(X, R, t)
        q = pixels(x2, K)
        if not ((z2 > 0).all() and (q[0] >= 0).all() and (q[0] < (W, H)).all()):
            continue
        s = _straddle_along(R, t, dist, K, p0, q[0], 1, q[1] - q[0], False, tight)
        if s is not None:
            out.append(s)
    made = 0
    while made < epipole:
        tries += 1
        assert tries < 50 * (count + epipole) + 50
        if t[2] > 0:                                             # x2 at the image of the first camera's centre
            p0 = rng.uniform((20, 20), (W - 20, H - 20)).astype(np.float32)
            x1h = Kinv @ np.array([p0[0], p0[1], 1.0])
            e = t / t[2]
            d = (R @ x1h) * t[2] - t * (R @ x1h)[2]              # d/dlam of the projection of lam R x1h + t at 0
            q = pixels(e[None, :2], K)[0]
            s = _straddle_along(R, t, dist, K, p0, q, 1, d[:2], True)
        else:                                                    # x1 at the image of the second camera's centre
            p1 = rng.uniform((20, 20), (W - 20, H - 20)).astype(np.float32)
            x2h = Kinv @ np.array([p1[0], p1[1], 1.0])
            C2 = -R.T @ t
            r = R.T @ x2h
            d = r * C2[2] - C2 * r[2]
            q = pixels((C2 / C2[2])[None, :2], K)[0]
            s = _straddle_along(R, t, dist, K, p1, q, 0, d[:2], True)
        if s is not None:
            out.append(s)
            made += 1
    return out


def place(p0, p1, st: list[Straddle]):
    """append both members of every straddle; returns the pixel arrays and the index of each good / bad member"""
    a = [p0] + [s.p0 for s in st]
    b = [p1] + [s.p1 for s in st]
    n0 = len(p0)
    gi = n0 + 2 * np.arange(len(st))
    return np.concatenate(a).astype(np.float32), np.concatenate(b).astype(np.float32), gi, gi + 1


# ---- special inputs --------------------------------------------------------------------------------------------

E_EXACT = np.array([[0.0, -1.0, 0.0], [1.0, 0.0, 0.0], [0.0, 0.0, 0.0]])     # [z]x I: R = I, t = z exactly


def dyadic_points(n: int, seed: int, K=POW2_K):
    """noise-free correspondences of R = I, t = z (E_EXACT) whose normalised coordinates are dyadic with few bits,
    so M = A'A is exactly singular in double: x2 = x1 Z / (Z + 1) with Z / (Z + 1) in {1/2, 3/4, 7/8} (Z = 1, 3, 7),
    and a few with Z / (Z + 1) in {5/4, 2} (Z = -5, -2: behind the first camera).  Pixels are exact float32."""
    rng = np.random.default_rng(seed)
    f = np.asarray(K, np.float64)[0, 0]
    x1 = rng.integers(-96, 97, (n, 2)) / 256.0
    s = rng.choice([0.5, 0.75, 0.875, 1.25, 2.0], n, p=[0.3, 0.3, 0.3, 0.05, 0.05])
    x2 = x1 * s[:, None]
    p0 = pixels(x1, K).astype(np.float32)
    p1 = pixels(x2, K).astype(np.float32)
    assert np.array_equal(p0.astype(np.float64), pixels(x1, K)) and np.array_equal(p1.astype(np.float64), pixels(x2, K))
    assert f == 512.0
    return p0, p1


def zero_start_points(n: int, seed: int, K=POW2_K):
    """x1 == x2 and x1 == -x2 under E_EXACT: the kernel's start vector is exactly zero for R = I (resp. R = diag(-1,
    -1, 1)); the exact point is at infinity"""
    rng = np.random.default_rng(seed)
    x1 = rng.integers(-96, 97, (n, 2)) / 256.0
    x1[np.all(x1 == 0, 1)] = 0.25
    x2 = np.where((np.arange(n) % 2 == 0)[:, None], x1, -x1)
    return pixels(x1, K).astype(np.float32), pixels(x2, K).astype(np.float32)


def start_vector(x, R, t):
    """the kernel's start vector (a1 z, b1 z, z, w) in double, each rounding as written (no contraction can change a
    result that is exact, which is all this is used for)"""
    a1, b1, a2, b2 = (float(v) for v in x)
    r2 = [a2 * R[2, k] - R[0, k] for k in range(3)] + [a2 * t[2] - t[0]]
    r3 = [b2 * R[2, k] - R[1, k] for k in range(3)] + [b2 * t[2] - t[1]]
    c2 = (r2[0] * a1 + r2[1] * b1) + r2[2]
    c3 = (r3[0] * a1 + r3[1] * b1) + r3[2]
    z, w = -(c2 * r2[3] + c3 * r3[3]), c2 * c2 + c3 * c3
    return np.array([a1 * z, b1 * z, z, w])


def normal_matrix_exact(x, R, t):
    """M = A'A of the doubles, exactly (Fractions)"""
    from fractions import Fraction as F
    a1, b1, a2, b2 = (F(float(v)) for v in x)
    Rf = [[F(float(v)) for v in row] for row in R]
    tf = [F(float(v)) for v in t]
    A = [[-1, 0, a1, 0], [0, -1, b1, 0],
         [a2 * Rf[2][k] - Rf[0][k] for k in range(3)] + [a2 * tf[2] - tf[0]],
         [b2 * Rf[2][k] - Rf[1][k] for k in range(3)] + [b2 * tf[2] - tf[1]]]
    return [[sum(F(A[r][i]) * A[r][j] for r in range(4)) for j in range(4)] for i in range(4)]


def fallback_margin(x, R, t, steps: int = 12):
    """The kernel's inverse-iteration loop restated at DPS digits, on the exact normal matrix with the kernel's shift
    mu = 1e-15 trace(M) and its start vector.  Returns (margin, ratio, Q): the smallest sin(angle(y, Q)) over the first
    `steps` steps divided by the kernel's convergence bound 2e-15, the eigenvalue ratio (l4 + mu) / (l3 + mu), and the
    last iterate.  A margin far above 1 (the tests ask for 100) means the kernel cannot meet its test within its 12
    steps -- rounding moves the iterates by far less than that -- so the loop hands the point to the Jacobi fallback;
    Q is what the kernel would use without that fallback."""
    with mpmath.workdps(DPS):
        Mf = normal_matrix_exact(x, R, t)
        M = mpmath.matrix([[mpmath.mpf(v.numerator) / v.denominator for v in row] for row in Mf])
        mu = mpmath.mpf(1e-15) * ((M[0, 0] + M[1, 1]) + (M[2, 2] + M[3, 3]))
        Ms = M + mu * mpmath.eye(4)
        ev = sorted(mpmath.eigsy(M)[0])
        ratio = (ev[0] + mu) / (ev[1] + mu)
        q = mpmath.matrix(start_vector(x, R, t).tolist())
        worst = mpmath.inf
        for _ in range(steps):
            y = mpmath.lu_solve(Ms, q)
            qq, qy, yy = (q.T * q)[0], (q.T * y)[0], (y.T * y)[0]
            s2 = 1 - qy * qy / (qq * yy)
            worst = min(worst, mpmath.sqrt(max(s2, 0)))
            q = y / mpmath.norm(y)
        return float(worst / mpmath.mpf(2e-15)), float(ratio), np.array([float(v) for v in q])


def tests_of_q(Q, R, t, dist) -> tuple:
    """the four tests (INEQ order) of a given homogeneous point"""
    v = _forms(R, t, dist) @ np.asarray(Q, np.float64)
    return tuple(bool(vj * Q[3] > 0) for vj in v)


def epipole_points(n: int, seed: int, R, t, K=KITTI_K, sigma=1.0, spread=4.0):
    """noisy correspondences at and around both epipoles: x1 within `spread` pixels of the first image's epipole,
    x2 = the second view of a point on that ray near the baseline, plus `sigma` pixels of noise on both"""
    rng = np.random.default_rng(seed)
    K = np.asarray(K, np.float64)
    C2 = -R.T @ t
    e1 = pixels((C2 / C2[2])[None, :2], K)[0]
    e2 = pixels((t / t[2])[None, :2], K)[0]
    p0 = e1 + rng.normal(0, spread, (n, 2))
    p1 = e2 + rng.normal(0, spread, (n, 2))
    p0 += rng.normal(0, sigma, (n, 2))
    p1 += rng.normal(0, sigma, (n, 2))
    return p0.astype(np.float32), p1.astype(np.float32)


# ---- the comparison rule -----------------------------------------------------------------------------------------

def check_call(D: Decision, n_good: int, R, t, mask, what="") -> int:
    """A recoverPose result (count, R, t, {0,255} mask) against the exact reference: (R, t) must be one of the four
    candidates; the mask must be that candidate's exact decision on every decided point; the count must be the mask's,
    within the candidate's possible exact counts, and not below any other candidate's sure count (so it is a maximum;
    with every point decided, exactly the largest exact count).  Returns the candidate's index."""
    c = match_candidate(D.C, R, t)
    m = np.asarray(mask).reshape(-1)
    assert len(m) == len(D.good) and set(np.unique(m).tolist()) <= {0, 255}, what
    d = D.decided[:, c]
    wrong = np.nonzero(d & ((m == 255) != D.good[:, c]))[0]
    assert not len(wrong), (what, c, wrong[:10].tolist())
    assert n_good == int((m == 255).sum()), what
    b = [D.count_bounds(k) for k in range(4)]
    assert b[c][0] <= n_good <= b[c][1], (what, b, c, n_good)
    assert all(n_good >= lo for lo, _ in b), (what, b, n_good)
    if all(lo == hi for lo, hi in b):
        assert n_good == max(lo for lo, _ in b), (what, b, n_good)
    return c


# ---- scenes ------------------------------------------------------------------------------------------------------

@dataclass
class Scene:
    name: str
    E: np.ndarray
    K: np.ndarray
    dist: float
    p0: np.ndarray                    # (n, 2) float32
    p1: np.ndarray
    target: tuple | None = None       # (R, t) the scene is built to make the winner
    st: list | None = None            # straddles, members at gi (good) / bi (bad)
    gi: np.ndarray | None = None
    bi: np.ndarray | None = None

    def x(self):
        return norm4(self.p0, self.p1, self.K)


MOTIONS = (1, 2, 3, 4)
FWD = motion(11)                      # forward motion for the epipole and fallback scenes (KITTI camera)


def straddle_scene(mseed: int, sign: int, dist: float, n_clear: int = 160) -> Scene:
    """clear points of the candidate (R, sign t) plus its straddles: 8 depth straddles, 4 epipole straddles and
    (dist 50 and 3) 3 depth straddles within TIGHT of dist"""
    R, t = motion(mseed)
    t = sign * t
    seed = 1000 * mseed + (sign > 0) * 100 + int(math.log10(dist) * 10)
    st = straddles(R, t, dist, 8, seed, epipole=4)
    if dist < 1e3:
        st += straddles(R, t, dist, 3, seed + 1, tight=TIGHT)
    p0, p1 = clear_points(R, t, dist, n_clear, seed + 2)
    q0, q1, gi, bi = place(p0, p1, st)
    return Scene(f"straddle m{mseed} {'+' if sign > 0 else '-'}t d{dist:g}", essential(R, t), POW2_K, dist, q0, q1,
                 (R, t), st, gi, bi)


def straddle_scenes(dist: float) -> list[Scene]:
    return [straddle_scene(m, s, dist) for m in MOTIONS for s in (1, -1)]


def fallback_scene(dist: float, c: int) -> Scene:
    """KITTI camera, forward motion: 2800 noisy correspondences at and around both epipoles, and 400 clear points
    of candidate c (so that candidate wins and its mask is the one compared)"""
    R, t = FWD
    E = essential(R, t)
    Rc, tc = candidates(E).f64[c]
    ps = [epipole_points(400, 100 + s, R, t, sigma=0.5, spread=1.5) for s in range(6)]
    ps.append(epipole_points(400, 7, R, t, sigma=1.0, spread=4.0))
    ps.append(clear_points(Rc, tc, dist, 400, 50 + c, KITTI_K, synth_size()))
    return Scene(f"fallback d{dist:g} c{c}", E, KITTI_K, dist, np.concatenate([p[0] for p in ps]),
                 np.concatenate([p[1] for p in ps]), (Rc, tc))


def synth_size():
    from epivo_b200 import synth
    return synth.KITTI_SIZE


def special_scene(dist: float) -> Scene:
    """E_EXACT (R = I, t = z exactly): dyadic noise-free points (M exactly singular), x1 == +-x2 (zero start vector),
    NaN / +-inf pixels"""
    d0, d1 = dyadic_points(96, 3)
    z0, z1 = zero_start_points(32, 4)
    bad0 = np.array([[np.nan, 100], [300, 200], [np.inf, 10], [20, -np.inf], [np.nan, np.nan], [5, 5]], np.float32)
    bad1 = np.array([[200, 100], [np.nan, 200], [310, 20], [np.inf, 10], [1, 2], [-np.inf, np.nan]], np.float32)
    return Scene(f"special d{dist:g}", E_EXACT.copy(), POW2_K, dist, np.concatenate([d0, z0, bad0]),
                 np.concatenate([d1, z1, bad1]))


def infinity_scene(dist: float) -> Scene:
    """a generic motion: clear points, and points at infinity (x2 = the rounded image of the direction R x1)"""
    R, t = motion(5)
    p0, p1 = clear_points(R, t, dist, 120, 9)
    rng = np.random.default_rng(10)
    q0 = rng.uniform((20, 20), (PSIZE[0] - 20, PSIZE[1] - 20), (64, 2))
    Kinv = np.linalg.inv(POW2_K)
    d = np.concatenate([q0, np.ones((64, 1))], 1) @ Kinv.T @ R.T
    q1 = pixels(d[:, :2] / d[:, 2:3], POW2_K)
    return Scene(f"infinity d{dist:g}", essential(R, t), POW2_K, dist, np.concatenate([p0, q0]).astype(np.float32),
                 np.concatenate([p1, q1]).astype(np.float32), (R, t))


def tie_scenes() -> list[Scene]:
    """equal numbers of clear points of two candidates: (R, t) and (R, -t); (R1, t) and (R2, t); and a scene of
    points at infinity only, where every count is 0"""
    R, t = motion(6)
    E = essential(R, t)
    C = candidates(E)
    ca = match_candidate(C, R, t)
    out = []
    for other in (ca ^ 2, ca ^ 1):
        Ro, to = C.f64[other]
        a0, a1 = clear_points(R, t, 50.0, 60, 21)
        b0, b1 = clear_points(Ro, to, 50.0, 60, 22)
        out.append(Scene(f"tie c{ca}/c{other}", E, POW2_K, 50.0, np.concatenate([a0, b0]), np.concatenate([a1, b1])))
    inf = infinity_scene(50.0)
    out.append(Scene("all zero", inf.E, POW2_K, 50.0, inf.p0[120:], inf.p1[120:]))
    return out
