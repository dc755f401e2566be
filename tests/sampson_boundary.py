"""Correspondences and models on the Sampson inlier boundary, with an exact reference (host only).

The inlier test of the essential-matrix kernels (epivo_b200/csrc/essential.cu) has three tiers:
    1. a fused pre-filter (sampson_fast + prefilter_decide) that decides every point whose error is more
       than a relative ~2e-6 away from B, the largest double whose float rounding is <= thr32;
    2. the exact sign of B den - num (num, den in OpenCV's un-fused order), one FMA;
    3. the division (float)(num / den) <= thr32, for quotients within 2^-50 of B.
Real data lands in the 2e-6 band about once per million points, so this module builds points that land
there on purpose:
    * model-tuned straddles: for one correspondence, two models one double ulp of E[8] apart that the
      oracle decides differently ("last in", "first out"); both quotients lie within 2^-50 of B (tier 3);
    * point-tuned straddles: for one model, two correspondences one float32 pixel ulp apart that the oracle
      decides differently; both quotients lie within 2e-6 of B (tier 2, sometimes 3).
It also restates the kernel's tiers exactly (every rounded operation as the correctly rounded rational), so
a host test can show that these points get past the pre-filter without a GPU.
"""
from __future__ import annotations

import math
import struct
from dataclasses import dataclass
from fractions import Fraction

import numpy as np

from epivo_b200 import synth
from oracle import oracle as O

F = Fraction
KITTI_K = synth.KITTI_K
EUROC_K = synth.EUROC_K
POW2_K = np.array([[512.0, 0.0, 300.5], [0.0, 512.0, 180.25], [0.0, 0.0, 1.0]])   # p * (1/512) is exact
IMAGE = {"kitti": synth.KITTI_SIZE, "euroc": synth.EUROC_SIZE, "pow2": (640, 400)}
REL_TIER2 = 2e-6
REL_TIER3 = 2.0 ** -50


# ---- threshold: what make_samp_thr computes -------------------------------------------------------------

def thr32_of(thr_px: float, K) -> np.float32:
    """(float)(t * t) with t = thr / ((fx + fy) / 2): the float32 threshold the kernels compare against."""
    return np.float32(O.ransac_threshold(thr_px, K) ** 2)


def f32_bits(x) -> int:
    return struct.unpack("<I", struct.pack("<f", float(x)))[0]


def f64_bits(x: float) -> int:
    return struct.unpack("<q", struct.pack("<d", x))[0]


def f64_of_bits(b: int) -> float:
    return struct.unpack("<d", struct.pack("<q", b))[0]


def hi(x: float) -> int:
    """high 32 bits of a double as a signed int (__double2hiint)"""
    return f64_bits(x) >> 32


@dataclass
class SampThr:
    thr32: np.float32
    B: float
    C: float
    dmin: float
    eoff: int
    hdmin: int


def samp_thr(thr32) -> SampThr:
    """make_samp_thr restated: B = the midpoint between thr32 and the next float, one double ulp lower when the
    mantissa of thr32 is odd (the tie then rounds away from thr32)."""
    thr32 = np.float32(thr32)
    bits = f32_bits(thr32)
    up = struct.unpack("<f", struct.pack("<I", bits + 1))[0]
    mid = 0.5 * (float(thr32) + up)
    if (bits & 1) and 0.0 < mid < 1e300:
        mid = f64_of_bits(f64_bits(mid) - 1)
    assert thr32 >= 0 and thr32 < 3e38
    dmin = max(1e-8, 1e-13 / mid)
    e = math.frexp(mid * 2.1e-6)[1] if mid > 1e-200 else 0
    return SampThr(thr32, mid, mid * 8.881784197001252e-16, dmin, e * (1 << 20), hi(dmin))


def thresholds(K, base=(1.0, 0.3, 0.05)) -> list[float]:
    """The reference's RANSAC thresholds plus, for a thr32 mantissa parity none of them has, one more threshold
    near 0.5 px that has it: both branches of the odd-mantissa nudge get exercised."""
    out = list(base)
    have = {f32_bits(thr32_of(t, K)) & 1 for t in out}
    t = 0.5
    while len(have) < 2:
        if f32_bits(thr32_of(t, K)) & 1 not in have:
            out.append(t)
            have.add(f32_bits(thr32_of(t, K)) & 1)
        t = float(np.nextafter(t, 1.0) + 1e-9)
    return out


# ---- OpenCV's un-fused evaluation and the exact decision --------------------------------------------------

def num_den(E, a1, b1, a2, b2):
    """num, den of EMEstimatorCallback::computeError as doubles (Python floats: round to nearest, never fused)."""
    E = [float(e) for e in np.asarray(E, dtype=np.float64).reshape(9)]
    ex0 = (E[0] * a1 + E[1] * b1) + E[2]
    ex1 = (E[3] * a1 + E[4] * b1) + E[5]
    ex2 = (E[6] * a1 + E[7] * b1) + E[8]
    et0 = (E[0] * a2 + E[3] * b2) + E[6]
    et1 = (E[1] * a2 + E[4] * b2) + E[7]
    s = (a2 * ex0 + b2 * ex1) + ex2
    return s * s, ((ex0 * ex0 + ex1 * ex1) + et0 * et0) + et1 * et1


def inlier(E, x, thr32) -> bool:
    """OpenCV's decision: (float)(num / den) <= thr32."""
    num, den = num_den(E, *x)
    return bool(np.float32(num / den) <= np.float32(thr32))


def rel_to_B(E, x, T: SampThr) -> float:
    """|num / den - B| / B, exactly."""
    num, den = num_den(E, *x)
    return float(abs(F(num) / F(den) - F(T.B)) / F(T.B))


def rn(q: Fraction) -> float:
    """the double nearest to q (ties to even): CPython's int / int true division is correctly rounded"""
    return q.numerator / q.denominator


def fma(a: float, b: float, c: float) -> float:
    return rn(F(a) * F(b) + F(c))


def exact_tier(E, x, T: SampThr) -> int:
    """Which tier of sampson_inlier() decides: 2 (the sign of the FMA B den - num, or the 2^-50 early-out) or
    3 (the division)."""
    num, den = num_den(E, *x)
    r = fma(T.B, den, -num)
    if r >= 0.0 and den > 0.0:
        return 2
    if -r > T.C * den:          # C = B 2^-50: the product is exact
        return 2
    return 3


def prefilter(E, x, T: SampThr, hdmin: int):
    """sampson_fast + prefilter_decide restated, every fma and product correctly rounded, the high-word tests as
    integers.  Returns (decided, inlier)."""
    E = [float(e) for e in np.asarray(E, dtype=np.float64).reshape(9)]
    a1, b1, a2, b2 = (float(v) for v in x)
    ex0 = fma(E[0], a1, fma(E[1], b1, E[2]))
    ex1 = fma(E[3], a1, fma(E[4], b1, E[5]))
    ex2 = fma(E[6], a1, fma(E[7], b1, E[8]))
    et0 = fma(E[0], a2, fma(E[3], b2, E[6]))
    et1 = fma(E[1], a2, fma(E[4], b2, E[7]))
    sx = fma(a2, ex0, fma(b2, ex1, ex2))
    den = fma(ex0, ex0, fma(ex1, ex1, fma(et0, et0, et1 * et1)))
    num = sx * sx
    t = fma(-den, T.B, num)
    ht, hd = hi(t), hi(den)
    at = ht & 0x7FFFFFFF
    return (at > hd + T.eoff and at < 0x7FF00000 and hd > hdmin), ht < 0


def model_hdmin(E, T: SampThr) -> int:
    """score_count_kernel's per-model smallest trusted denominator: hi(dmin |E|_F^2)"""
    f2 = float(np.sum(np.asarray(E, dtype=np.float64) ** 2))
    return hi(abs(T.dmin * f2)) | (0 if f2 > 0 else 0x7FF00000)


# ---- straddle generators -------------------------------------------------------------------------------

def _flip(decide, lo: int, hi_: int) -> int:
    """k in [lo, hi) with decide(k) != decide(k + 1), given decide(lo) != decide(hi)"""
    dlo = decide(lo)
    assert dlo != decide(hi_)
    while hi_ - lo > 1:
        mid = (lo + hi_) // 2
        if decide(mid) == dlo:
            lo = mid
        else:
            hi_ = mid
    return lo


def _bracket(decide, reach=(1 << 24)):
    """a flip of decide within +-reach of 0, or None"""
    d0 = decide(0)
    k = 4
    while k <= reach:
        if decide(k) != d0:
            return _flip(decide, 0, k)
        if decide(-k) != d0:
            return _flip(decide, -k, 0)
        k *= 4
    return None


@dataclass
class ModelStraddle:
    p1: np.ndarray        # (2,) float32 pixels in the first image
    p2: np.ndarray        # (2,) float32 pixels in the second image
    E_in: np.ndarray      # (9,) the model that counts the correspondence as an inlier
    E_out: np.ndarray     # (9,) E_in with E[8] one double ulp further: an outlier


def model_straddles(K, thr_px: float, count: int, seed: int, image=(1241, 376)) -> list[ModelStraddle]:
    """Model-tuned straddles for the camera K.  The models are built so that no sum in x2' E x1 cancels (all
    terms of s = (a2 ex0 + b2 ex1) + ex2 and of ex2 = (E6 a1 + E7 b1) + E8 are positive and below |s|): one
    ulp of E[8] then moves s by at most one ulp, and the two models' quotients are adjacent, on both sides of
    B.  ex0 and ex1 themselves are small differences of O(1) terms, so a one-ulp change of a normalised
    coordinate of x1 moves the quotient by far more than one step: the pairs pin the K-normalisation."""
    T = samp_thr(thr32_of(thr_px, K))
    rng = np.random.default_rng(seed)
    W, H = image
    out: list[ModelStraddle] = []
    while len(out) < count:
        p1 = np.array([rng.uniform(0, W), rng.uniform(0, H)], dtype=np.float32)
        p2 = np.array([rng.uniform(0, W), rng.uniform(0, H)], dtype=np.float32)
        (a1, b1), (a2, b2) = O.normalize_points(p1[None], K)[0], O.normalize_points(p2[None], K)[0]
        if min(abs(a1), abs(b1), abs(a2), abs(b2)) < 0.05:
            continue
        E = np.zeros(9)
        E[[0, 1, 3, 4]] = rng.normal(0.0, 0.5, 4)
        den0 = (E[0] * a2 + E[3] * b2) ** 2 + (E[1] * a2 + E[4] * b2) ** 2
        s = math.sqrt(T.B * den0)
        E[2] = math.copysign(0.15 * s / abs(a2), a2) - (E[0] * a1 + E[1] * b1)
        E[5] = math.copysign(0.15 * s / abs(b2), b2) - (E[3] * a1 + E[4] * b1)
        E[6] = math.copysign(0.15 * s / abs(a1), a1)
        E[7] = math.copysign(0.15 * s / abs(b1), b1)
        x = (a1, b1, a2, b2)
        for _ in range(3):                                   # E[8] for s = sqrt(B den)
            num, den = num_den(E, *x)
            E[8] += math.sqrt(T.B * den) - math.sqrt(num)
        base = f64_bits(E[8])

        def decide(k, E=E, base=base, x=x):
            Ek = E.copy()
            Ek[8] = f64_of_bits(base + k)
            return inlier(Ek, x, T.thr32)

        k = _bracket(decide, 1 << 12)
        if k is None:
            continue
        Ein, Eout = E.copy(), E.copy()
        Ein[8], Eout[8] = f64_of_bits(base + k), f64_of_bits(base + k + 1)
        if not decide(k):                                    # s > 0 and increasing in E[8]: in below, out above
            continue
        out.append(ModelStraddle(p1, p2, Ein, Eout))
    return out


@dataclass
class PointStraddle:
    p1: np.ndarray        # (2,) float32
    p2_in: np.ndarray     # (2,) float32: an inlier of the model
    p2_out: np.ndarray    # (2,) float32: p2_in with one coordinate one float32 ulp further: an outlier


def point_straddles(E, K, thr32, count: int, seed: int, image=(640, 400), band=REL_TIER2 / 4) -> list[PointStraddle]:
    """Point-tuned straddles of the model E for a camera K whose focal lengths are powers of two (the
    K-normalisation is then exact, whichever way it is rounded).  x1 is put on the line ex_j = 0 (j = 0 or 1,
    whichever crosses the image), so stepping the j-th coordinate of x2 by one float32 ulp moves the error only
    through den: the two neighbours land within a relative `band` of B.  Pairs outside the band are skipped."""
    K = np.asarray(K, dtype=np.float64)
    f = (K[0, 0], K[1, 1])
    c = (K[0, 2], K[1, 2])
    assert all(math.frexp(v)[0] == 0.5 for v in f), "focal lengths must be powers of two"
    T = samp_thr(thr32)
    E = np.asarray(E, dtype=np.float64).reshape(9)
    rng = np.random.default_rng(seed)
    W, H = image
    size = (W, H)
    out: list[PointStraddle] = []
    tries = 0
    while len(out) < count:
        tries += 1
        assert tries < 200 * count, "no line of E crosses the image"
        j = int(rng.integers(2))                               # ex_j ~ 0; x2[j] is the stepped coordinate
        r = E[3 * j:3 * j + 3]
        # pixel of x1 on r . (a1, b1, 1) = 0: draw the coordinate with the smaller coefficient, solve the other
        g = 0 if abs(r[0]) < abs(r[1]) else 1
        q1 = np.zeros(2)
        q1[g] = rng.uniform(0, size[g])
        ng = (q1[g] - c[g]) / f[g]
        o = 1 - g
        no = -(r[g] * ng + r[2]) / r[o]
        q1[o] = no * f[o] + c[o]
        if not 0 <= q1[o] < size[o]:
            continue
        p1 = q1.astype(np.float32)
        a1, b1 = O.normalize_points(p1[None], K)[0]
        # x2: coordinate j drawn, coordinate 1 - j solved for s^2 = B den
        q2 = np.zeros(2)
        q2[j] = rng.uniform(0, size[j])
        m = 1 - j
        sign = 1.0 if rng.integers(2) else -1.0
        x2 = [(q2[0] - c[0]) / f[0], (q2[1] - c[1]) / f[1]]
        Em = E.reshape(3, 3)
        ex = Em @ np.array([a1, b1, 1.0])
        if abs(ex[m]) < 1e-3:
            continue
        for _ in range(4):
            et = Em.T @ np.array([x2[0], x2[1], 1.0])
            den = ex[0] ** 2 + ex[1] ** 2 + et[0] ** 2 + et[1] ** 2
            x2[m] = (sign * math.sqrt(T.B * den) - ex[2] - x2[j] * ex[j]) / ex[m]
        q2[m] = x2[m] * f[m] + c[m]
        if not 0 <= q2[m] < size[m]:
            continue
        p2 = q2.astype(np.float32)
        base = f32_bits(p2[j])

        def at(k, p2=p2, base=base, j=j):
            q = p2.copy()
            q[j] = struct.unpack("<f", struct.pack("<I", base + k))[0]
            return q

        def decide(k, p1=p1):
            x = np.concatenate([O.normalize_points(p1[None], K)[0], O.normalize_points(at(k)[None], K)[0]])
            return inlier(E, x, T.thr32)

        k = _bracket(decide, 1 << 20)
        if k is None:
            continue
        pin, pout = (at(k), at(k + 1)) if decide(k) else (at(k + 1), at(k))
        xs = [np.concatenate([O.normalize_points(p1[None], K)[0], O.normalize_points(p[None], K)[0]]) for p in (pin, pout)]
        if max(rel_to_B(E, xx, T) for xx in xs) > band:
            continue
        out.append(PointStraddle(p1, pin, pout))
    return out


def unit_essential(seed: int) -> np.ndarray:
    """[t]x R for a random small rotation and a mostly forward translation, unit Frobenius norm (a model of the
    kind the five-point solver emits)."""
    rng = np.random.default_rng(seed)
    w = rng.normal(0, 0.05, 3)
    th = np.linalg.norm(w)
    k = w / th
    Kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    R = np.eye(3) + math.sin(th) * Kx + (1 - math.cos(th)) * Kx @ Kx
    t = np.array([rng.normal(0, 0.3), rng.normal(0, 0.1), 1.0])
    E = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]]) @ R
    return (E / np.linalg.norm(E)).reshape(9)
