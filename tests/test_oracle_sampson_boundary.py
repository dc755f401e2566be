"""Host checks of the boundary-point generator (tests/sampson_boundary.py) and of the oracle's K-normalisation.

The straddles must be decided differently by the oracle, must lie as close to B as claimed (exact rationals),
and must get past the kernels' fused pre-filter, restated here with every operation correctly rounded: the
GPU tests in test_gpu_sampson_boundary.py then reach the exact tiers of the inlier test."""
from fractions import Fraction

import numpy as np
import pytest

import sampson_boundary as SB
from oracle import oracle as O

CAMERAS = [("kitti", SB.KITTI_K), ("euroc", SB.EUROC_K)]


def _x(p1, p2, K):
    return np.concatenate([O.normalize_points(p1[None], K)[0], O.normalize_points(p2[None], K)[0]])


def _oracle_in(E, x, thr32):
    err = O.sampson_err_f32(E, x[None, :2], x[None, 2:])[0]
    return bool(err <= thr32)


@pytest.mark.parametrize("name,K", CAMERAS)
def test_model_straddles_reach_the_division(name, K):
    ths = SB.thresholds(K)
    assert {1.0, 0.3, 0.05} <= set(ths)
    assert {SB.f32_bits(SB.thr32_of(t, K)) & 1 for t in ths} == {0, 1}       # both branches of the nudge
    for i, thr in enumerate(ths):
        T = SB.samp_thr(SB.thr32_of(thr, K))
        ties = 0
        for s in SB.model_straddles(K, thr, 24, 100 + i, SB.IMAGE[name]):
            x = _x(s.p1, s.p2, K)
            assert _oracle_in(s.E_in, x, T.thr32) and not _oracle_in(s.E_out, x, T.thr32)
            for E in (s.E_in, s.E_out):
                assert SB.rel_to_B(E, x, T) < SB.REL_TIER3
                assert not SB.prefilter(E, x, T, SB.model_hdmin(E, T))[0]
                assert not SB.prefilter(E, x, T, T.hdmin)[0]
            assert SB.exact_tier(s.E_out, x, T) == 3                          # "first out" takes the division
            num, den = SB.num_den(s.E_out, *x)
            ties += SB.f64_bits(num / den) == SB.f64_bits(T.B) + 1             # RN(q) is the midpoint itself
        if SB.f32_bits(T.thr32) & 1:
            assert ties > 0, "no quotient rounds to the tie the odd-mantissa nudge exists for"


def test_point_straddles_reach_the_exact_test():
    K = SB.POW2_K
    for seed in range(3):
        E = SB.unit_essential(seed)
        for thr in SB.thresholds(K):
            T = SB.samp_thr(SB.thr32_of(thr, K))
            for s in SB.point_straddles(E, K, T.thr32, 8, seed, SB.IMAGE["pow2"]):
                xin, xout = _x(s.p1, s.p2_in, K), _x(s.p1, s.p2_out, K)
                assert _oracle_in(E, xin, T.thr32) and not _oracle_in(E, xout, T.thr32)
                d = np.abs(s.p2_in.view(np.int32).astype(np.int64) - s.p2_out.view(np.int32))
                assert sorted(d.tolist()) == [0, 1]                            # one float32 ulp in one coordinate
                for x in (xin, xout):
                    assert SB.rel_to_B(E, x, T) < SB.REL_TIER2
                    assert not SB.prefilter(E, x, T, T.hdmin)[0]


def test_prefilter_restatement_decides_clear_points():
    """The restated pre-filter is not vacuous: points well away from the boundary are decided, and rightly."""
    K = SB.KITTI_K
    rng = np.random.default_rng(5)
    E = SB.unit_essential(7)
    T = SB.samp_thr(SB.thr32_of(1.0, K))
    p = rng.uniform(0, 376, (200, 4)).astype(np.float32)
    decided = 0
    for r in p:
        x = _x(r[:2], r[2:], K)
        d, inl = SB.prefilter(E, x, T, T.hdmin)
        if d:
            decided += 1
            assert inl == _oracle_in(E, x, T.thr32)
    assert decided == len(p)


def test_samp_thr_is_the_largest_double_that_rounds_to_thr32():
    for t32 in (np.float32(1.0), np.float32(0.09), np.float32(3.3e-6), np.nextafter(np.float32(2e-7), np.float32(1))):
        T = SB.samp_thr(t32)
        assert np.float32(T.B) <= t32
        assert np.float32(np.nextafter(T.B, np.inf)) > t32


def test_normalize_points_is_the_correctly_rounded_fma():
    """The oracle's vectorised fused scale-and-shift against exact rationals."""
    rng = np.random.default_rng(11)
    for _, K in CAMERAS:
        p = rng.uniform(-100, 1400, (4000, 2)).astype(np.float32)
        got = O.normalize_points(p, K)
        for c in range(2):
            a = 1.0 / K[c, c]
            b = -K[c, 2] * a
            ref = [SB.rn(Fraction(float(v)) * Fraction(a) + Fraction(b)) for v in p[:, c]]
            assert np.array_equal(got[:, c], ref)


def test_cv2_normalisation_is_fused():
    """OpenCV evaluates `(col - cx) / fx` as convertTo(col, CV_64F, 1/fx, -cx/fx).  cv2 exposes that conversion
    through normalize(NORM_MINMAX): with the column [cx, u, cx + fx] it computes scale = 1/fx and shift =
    -cx * (1/fx) (when cx + fx - cx is exactly fx), OpenCV's alpha and beta.  The source is a strided CV_64F
    column, as in five-point.cpp.  Where the fused and the un-fused results differ, cv2 must give the fused one."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(3)
    differ = 0
    for _, K in CAMERAS:
        for c in range(2):
            f, cc = K[c, c], K[c, 2]
            smax = cc + f
            scale = 1.0 * (1.0 / (smax - cc))          # normalize(): (dmax - dmin) / (smax - smin), shift = dmin - smin scale
            shift = 0.0 - cc * scale
            if smax - cc == f:
                assert (scale, shift) == (1.0 / f, -cc * (1.0 / f))
            u = rng.uniform(cc, smax, 1500).astype(np.float32).astype(np.float64)
            buf = np.zeros((3, 2))
            for v in u:
                buf[:, 0] = (cc, v, smax)
                got = cv2.normalize(buf[:, :1], None, 0.0, 1.0, cv2.NORM_MINMAX, cv2.CV_64F)[1, 0]
                fused = O.fma_f32_scalar(np.array([v]), scale, shift)[0]
                assert got == fused
                differ += fused != v * scale + shift
    assert differ > 1000
