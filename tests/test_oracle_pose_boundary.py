"""Host checks of the recoverPose boundary cases (tests/pose_boundary.py) and of their exact reference.

The straddles must really flip in the exact reference, the special inputs must reach what they are built for, and on
every decided point the exact reference must agree with live cv2.recoverPose and with the oracle: that agreement is
what makes the decided rule a fair basis for the GPU comparison in test_gpu_pose_boundary.py."""
from fractions import Fraction

import numpy as np
import pytest

import pose_boundary as PB
from oracle import oracle as O


@pytest.fixture(scope="module")
def scenes():
    out = [s for d in PB.DISTS for s in PB.straddle_scenes(d)]
    out += [PB.fallback_scene(d, c) for d in PB.DISTS for c in range(4)]
    out += [PB.special_scene(d) for d in PB.DISTS] + [PB.infinity_scene(d) for d in PB.DISTS] + PB.tie_scenes()
    return out


def test_straddles_flip():
    kinds = {}
    for d in PB.DISTS:
        for s in PB.straddle_scenes(d):
            R, t = s.target
            D = PB.decide(s.E, s.x(), d)
            c = PB.match_candidate(D.C, R, t)
            x = s.x()
            for k, st in enumerate(s.st):
                g, b = s.gi[k], s.bi[k]
                # one float32 ulp in one coordinate of one pixel
                diff = np.abs(np.concatenate([st.p0[0], st.p1[0]]).view(np.int32).astype(np.int64)
                              - np.concatenate([st.p0[1], st.p1[1]]).view(np.int32))
                assert sorted(diff.tolist()) == [0, 0, 0, 1]
                tg, tb = PB.tests_exact(x[g], R, t, d), PB.tests_exact(x[b], R, t, d)
                assert all(tg) and not all(tb)
                assert [PB.INEQ[i] for i in range(4) if tg[i] != tb[i]] == [st.kind]
                assert D.good[g, c] and not D.good[b, c]
                key = (st.kind, d, st.near_epipole)
                n_dec, n = kinds.get(key, (0, 0))
                kinds[key] = (n_dec + int(D.decided[g, c] and D.decided[b, c]), n + 1)
    print({k: v for k, v in sorted(kinds.items())})
    for d in PB.DISTS:
        for kind in ("Z<d", "z2<d"):
            n_dec, n = kinds[(kind, d, False)]
            assert n >= 8 and n_dec >= 0.9 * n, (kind, d, n_dec, n)
        for kind in ("zw", "z2>0"):
            n_dec, n = kinds[(kind, d, True)]
            assert n >= 8 and n_dec >= 0.5 * n, (kind, d, n_dec, n)


def test_tight_straddles_are_within_half_a_float_ulp():
    """the TIGHT depth straddles: the good member's depth rounds to dist in float32, the bad one does not fall below"""
    tight = 0
    for d in (50.0, 3.0):
        for s in PB.straddle_scenes(d):
            R, t = s.target
            for k, st in enumerate(s.st[-3:]):
                xg = s.x()[s.gi[len(s.st) - 3 + k]]
                Q = np.linalg.svd(PB._dlt(xg[None], R, t))[2][0, 3]
                dep = Q[2] / Q[3] if st.kind == "Z<d" else (R[2] @ Q[:3]) / Q[3] + t[2]
                assert dep < d and np.float32(dep) == np.float32(d)
                tight += 1
    assert tight == 2 * 2 * len(PB.MOTIONS) * 3


def _finite(s):
    return np.isfinite(s.p0).all(1) & np.isfinite(s.p1).all(1)


def test_exact_reference_agrees_with_cv2_and_oracle(scenes):
    cv2 = pytest.importorskip("cv2")
    total = [0, 0]
    for s in scenes:
        f = _finite(s)                       # cv2 is not asked about NaN / inf pixels
        p0, p1 = s.p0[f], s.p1[f]
        D = PB.decide(s.E, PB.norm4(p0, p1, s.K), s.dist)
        total[0] += int(D.decided.sum())
        total[1] += D.decided.size
        n, R, t, m = cv2.recoverPose(np.asarray(s.E, np.float64).reshape(3, 3), p0.astype(np.float64),
                                     p1.astype(np.float64), np.asarray(s.K, np.float64), distanceThresh=s.dist)[:4]
        PB.check_call(D, int(n), R, t.reshape(3), m.reshape(-1), "cv2 " + s.name)
        n, R, t, m = O.recover_pose(s.E, p0, p1, s.K, s.dist)
        PB.check_call(D, int(n), R, t, m, "oracle " + s.name)
    print(f"decided {total[0]} of {total[1]} (point, candidate) decisions")
    assert total[0] >= 0.99 * total[1]


def test_exact_reference_with_an_input_mask():
    cv2 = pytest.importorskip("cv2")
    s = PB.straddle_scene(2, -1, 50.0)
    im = (np.random.default_rng(4).random(len(s.p0)) < 0.8).astype(np.uint8)
    D = PB.decide(s.E, s.x(), s.dist, in_mask=im)
    n, R, t, m = cv2.recoverPose(s.E.reshape(3, 3), s.p0.astype(np.float64), s.p1.astype(np.float64), s.K,
                                 distanceThresh=s.dist, mask=255 * im.reshape(-1, 1))[:4]   # cv2 ANDs it in
    PB.check_call(D, int(n), R, t.reshape(3), m.reshape(-1), "cv2 masked")
    n, R, t, m = O.recover_pose(s.E, s.p0, s.p1, s.K, s.dist, in_mask=im)
    PB.check_call(D, int(n), R, t, m, "oracle masked")


def test_fallback_points_cannot_converge_in_twelve_steps():
    """Near the epipoles the inverse iteration contracts slowly: the exact restatement of the kernel's loop is more
    than 100x its convergence bound away after 12 steps for many points, and for some of them the 12th iterate --
    what the kernel would use without its Jacobi fallback -- decides differently from the exact reference on the
    candidate the fallback scenes make the winner."""
    R, t = PB.FWD
    C = PB.candidates(PB.essential(R, t))
    s = PB.fallback_scene(50.0, 0)
    x = s.x()
    n_fb = n_tried = 0
    for i in range(0, 400):                                  # the first noisy block, both rotations
        for c in (0, 1):
            n_tried += 1
            n_fb += PB.fallback_margin(x[i], *C.f64[c])[0] > 100
    print(f"{n_fb} of {n_tried} (point, rotation) solves of the first block take the fallback")
    assert n_fb >= 0.1 * n_tried
    # the slow ones of every block: points the no-fallback kernel would get wrong
    wrong = set()
    for c in (0, 1):
        Rc, tc = C.f64[c]
        _, sv, _ = np.linalg.svd(PB._dlt(x[:2800], Rc, tc))
        for i in np.nonzero((sv[:, 3] / sv[:, 2]) ** 2 > 0.6)[0]:
            m, _, Q = PB.fallback_margin(x[i], Rc, tc)
            if m <= 100:
                continue
            for cc, Qs in ((c, Q), (c + 2, Q * np.array([1, 1, 1, -1.0]))):
                for d in PB.DISTS:
                    if all(PB.tests_of_q(Qs, *C.f64[cc], d)) != all(PB.tests_exact(x[i], *C.f64[cc], d)):
                        wrong.add((int(i), cc, d))
    print(f"{len(wrong)} (point, candidate, dist) decisions the 12th iterate gets wrong")
    assert len(wrong) >= 3
    for i, cc, d in wrong:                                   # ... and they are decided points of the fallback scenes
        assert PB.decide(s.E, x[i:i + 1], d).decided[0, cc]


def test_singular_normal_matrix_and_zero_start_vector():
    C = PB.candidates(PB.E_EXACT)
    assert [c[0].tolist() for c in C.f64[:2]] == [np.eye(3).tolist(), np.diag([-1.0, -1.0, 1.0]).tolist()]
    assert [c[1].tolist() for c in C.f64[:3:2]] == [[0.0, 0.0, 1.0], [0.0, 0.0, -1.0]]
    R, t = C.f64[0]
    d0, d1 = PB.dyadic_points(96, 3)
    x = PB.norm4(d0, d1, PB.POW2_K)
    singular = 0
    for xi in x:
        M = PB.normal_matrix_exact(xi, R, t)
        j = 0 if xi[0] != 0 else 1
        if xi[j] == 0:
            continue
        # exactly singular: x2 = x1 Z / (Z + 1), so (a1 Z, b1 Z, Z, 1) is a null vector of M
        Z = 1 / (Fraction(float(xi[j])) / Fraction(float(xi[2 + j])) - 1)
        v = [Fraction(float(xi[0])) * Z, Fraction(float(xi[1])) * Z, Z, Fraction(1)]
        assert all(sum(M[i][k] * v[k] for k in range(4)) == 0 for i in range(4))
        singular += 1
        # and the kernel's double entries are those exact values (no rounding anywhere)
        a1, b1, a2, b2 = (float(v) for v in xi)
        r2 = [a2 * R[2, k] - R[0, k] for k in range(3)] + [a2 * t[2] - t[0]]
        r3 = [b2 * R[2, k] - R[1, k] for k in range(3)] + [b2 * t[2] - t[1]]
        assert 1.0 + (r2[0] * r2[0] + r3[0] * r3[0]) == M[0][0]
        assert (a1 * a1 + b1 * b1) + (r2[2] * r2[2] + r3[2] * r3[2]) == M[2][2]
        assert r2[2] * r2[3] + r3[2] * r3[3] == M[2][3] and r2[3] * r2[3] + r3[3] * r3[3] == M[3][3]
    assert singular >= 90
    D = PB.decide(PB.E_EXACT, x, 50.0)
    assert D.decided.all() and D.good[:, 0].sum() > 48
    z0, z1 = PB.zero_start_points(32, 4)
    xz = PB.norm4(z0, z1, PB.POW2_K)
    for k, xi in enumerate(xz):
        c = 0 if k % 2 == 0 else 1                           # x1 == x2 under R = I, x1 == -x2 under R = diag(-1, -1, 1)
        assert not PB.start_vector(xi, *C.f64[c]).any()
    for d in PB.DISTS:
        D = PB.decide(PB.E_EXACT, xz, d)
        assert D.decided.all() and not D.good.any()          # at infinity: never good, for every candidate


def test_ties():
    for s in PB.tie_scenes():
        D = PB.decide(s.E, s.x(), s.dist)
        assert D.decided.all()
        counts = D.good.sum(0)
        assert (counts == counts.max()).sum() >= 2, (s.name, counts)
