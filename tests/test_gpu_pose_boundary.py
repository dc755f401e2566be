"""recoverPose's per-point decisions at their boundaries, on every GPU path, against the exact reference.

Cases and the reference come from tests/pose_boundary.py (host checks in test_oracle_pose_boundary.py): straddles of
each of the four tests one float32 ulp apart, noisy points at the epipoles that take the Jacobi fallback, an exactly
singular normal matrix, zero start vectors, points at infinity, NaN / inf pixels and candidate ties.  Every result is
compared by pose_boundary.check_call: the mask bytes on the decided points, the count, and (R, t) as one of the
exact candidates.  Paths:
    api.recoverPose           epivo_recover_pose (with / without an input mask, several sizes)
    process_points            the sequence pipeline's pose stage (E from RANSAC, per-pair stride, skipped pairs)
"""
import numpy as np
import pytest

import pose_boundary as PB
from epivo_b200 import api, synth

pytestmark = pytest.mark.gpu


def _gpu(ctx, s, p0=None, p1=None, mask=None):
    p0 = s.p0 if p0 is None else p0
    p1 = s.p1 if p1 is None else p1
    return api.recoverPose(s.E, p0, p1, s.K, s.dist, mask=mask, ctx=ctx)


def _lane(ctx, s, c_target):
    """+1 if the kernel serves the scene's candidate from its own +t, -1 from -t: with no points the kernel returns
    its (R1, t)"""
    _, _, t0, _ = api.recoverPose(s.E, np.zeros((0, 2), np.float32), np.zeros((0, 2), np.float32), s.K, s.dist,
                                  ctx=ctx)
    C = PB.candidates(s.E)
    return 1 if np.abs(C.f64[c_target][1] - t0).max() < 1e-6 else -1


@pytest.mark.parametrize("dist", PB.DISTS)
def test_recover_pose_straddles(ctx, dist):
    lanes = set()
    rng = np.random.default_rng(int(dist))
    for s in PB.straddle_scenes(dist):
        D = PB.decide(s.E, s.x(), dist)
        n, R, t, m = _gpu(ctx, s)
        c = PB.check_call(D, n, R, t, m, s.name)
        assert c == PB.match_candidate(D.C, *s.target)
        assert (m[s.gi] == 255).all() and (m[s.bi] == 0).all()
        lane = _lane(ctx, s, c)
        lanes |= {(st.kind, lane) for st in s.st}
        im = (rng.random(len(s.p0)) < 0.8).astype(np.uint8)
        Dm = PB.decide(s.E, s.x(), dist, in_mask=im)
        n, R, t, m = _gpu(ctx, s, mask=im)
        PB.check_call(Dm, n, R, t, m, s.name + " masked")
    print(sorted(lanes))
    assert lanes == {(k, ln) for k in PB.INEQ for ln in (1, -1)}          # every test, in both lanes of the kernel


@pytest.mark.parametrize("n", [0, 1, 127, 128, 129, 3000])
def test_recover_pose_sizes(ctx, n):
    """per-thread loops (128 threads) and the warp-count reduction across their edges; straddles spread over the
    whole range"""
    R, t = PB.motion(7)
    st = PB.straddles(R, t, 50.0, 8, 70, epipole=4)
    p0, p1 = PB.clear_points(R, t, 50.0, max(n, 1), 71)
    q0, q1, _, _ = PB.place(p0, p1, st)
    order = np.random.default_rng(n).permutation(len(q0))[:n]
    s = PB.Scene(f"n{n}", PB.essential(R, t), PB.POW2_K, 50.0, q0[order], q1[order])
    D = PB.decide(s.E, s.x(), 50.0)
    ng, Rg, tg, m = _gpu(ctx, s)
    assert len(m) == n
    PB.check_call(D, ng, Rg, tg, m, s.name)
    if n == 0:
        assert ng == 0


@pytest.mark.parametrize("dist", PB.DISTS)
def test_recover_pose_special(ctx, dist):
    scenes = [PB.fallback_scene(dist, c) for c in range(4)] + [PB.special_scene(dist), PB.infinity_scene(dist)]
    for s in scenes:
        D = PB.decide(s.E, s.x(), dist)
        n, R, t, m = _gpu(ctx, s)
        c = PB.check_call(D, n, R, t, m, s.name)
        if s.target is not None:
            assert c == PB.match_candidate(D.C, *s.target), s.name
        bad = ~(np.isfinite(s.p0).all(1) & np.isfinite(s.p1).all(1))
        assert (m[bad] == 0).all()
        print(s.name, D.summary(c))


def test_recover_pose_ties(ctx):
    for s in PB.tie_scenes():
        D = PB.decide(s.E, s.x(), s.dist)
        n, R, t, m = _gpu(ctx, s)
        c = PB.check_call(D, n, R, t, m, s.name)
        counts = D.good.sum(0)
        assert n == counts.max() and counts[c] == n


# ---- the sequence pipeline -------------------------------------------------------------------------------------

K = synth.KITTI_K
SIZE = synth.KITTI_SIZE


def _pair(seed, depth, n, px=0.3, t=(0.02, -0.01, 1.0), near=0, extra=None):
    """n correspondences of a KITTI-camera pair (forward motion, depths uniform in `depth`), `near` noisy ones at
    both epipoles; extra = (k, depth) adds k points at other depths"""
    rng = np.random.default_rng(seed)
    R = PB.rotation(rng.normal(0, 0.01, 3))
    t = np.asarray(t, np.float64)
    Kinv = np.linalg.inv(K)
    out0, out1 = [], []
    for cnt, dep in [(n, depth)] + ([extra] if extra else []):
        got = 0
        while got < cnt:
            p = rng.uniform((0, 0), SIZE, (4 * cnt, 2))
            Z = rng.uniform(dep[0], dep[1], 4 * cnt)
            X = (np.concatenate([p, np.ones((4 * cnt, 1))], 1) @ Kinv.T) * Z[:, None]
            Y = X @ R.T + t
            q = PB.pixels(Y[:, :2] / Y[:, 2:3], K)
            ok = (Y[:, 2] > 0.1) & (q >= 0).all(1) & (q < SIZE).all(1)
            p, q = p[ok][:cnt - got], q[ok][:cnt - got]
            out0.append(p + rng.normal(0, px, p.shape))
            out1.append(q + rng.normal(0, px, q.shape))
            got += len(p)
    if near and np.linalg.norm(t) > 0:
        e0, e1 = PB.epipole_points(near, seed + 1, R, t / np.linalg.norm(t), K, sigma=0.5, spread=2.0)
        out0.append(e0)
        out1.append(e1)
    return np.concatenate(out0).astype(np.float32), np.concatenate(out1).astype(np.float32)


def _check_pipeline(ctx, pipe, prm, pairs, want_good=None):
    out = pipe.process_points(prm, [p[0] for p in pairs], [p[1] for p in pairs])
    stats = []
    for i, (p0, p1) in enumerate(pairs):
        r = out[i]
        em, pm = pipe.masks(i)
        if r["n_inliers"] == 0 or not np.abs(r["E"]).any():            # a failed pair: the pose stage skipped it
            assert r["n_good"] == 0 and r["lm_ran"] == 0 and not pm.any()
            stats.append("skipped")
            continue
        sel = em != 0
        c0, c1 = p0[sel], p1[sel]
        E = r["E"].reshape(3, 3)
        s = PB.Scene(f"pair {i}", E, K, prm.dist_thresh, c0, c1)
        D = PB.decide(E, s.x(), prm.dist_thresh)
        c = PB.check_call(D, int(r["n_good"]), r["R"], r["t"], pm, s.name)
        # the standalone call on the same E and inlier pixels: the same bytes
        n2, R2, t2, m2 = api.recoverPose(E, c0, c1, K, prm.dist_thresh, ctx=ctx)
        assert n2 == r["n_good"] and np.array_equal(m2, pm)
        assert np.array_equal(R2, r["R"]) and np.array_equal(t2, r["t"])
        lo, hi = D.count_bounds(c)
        if min(lo, len(c0)) >= prm.lm_points or hi < prm.lm_points or len(c0) < prm.lm_points:
            assert bool(r["lm_ran"]) == (len(c0) >= prm.lm_points and lo >= prm.lm_points), (i, lo, hi)
        if want_good is not None and want_good[i] is not None:
            assert lo == hi == want_good[i], (i, lo, hi)
        stats.append(f"{len(c0)} inliers: {D.summary(c)}")
    print(stats)
    return out


def test_pipeline_pose_boundary(ctx):
    pipe = api.SequencePipeline(8, 1500, ctx=ctx)
    # dist 50 (the reference's): depths across the cut, points at both epipoles, a rotation-only pair, pairs whose
    # good count is 47 / 48 / 49 (near points plus far ones no candidate calls good), a pair too small to estimate
    pairs = [_pair(1, (5.0, 60.0), 900, near=60),
             _pair(2, (5.0, 60.0), 600, px=1.0, near=120),
             _pair(3, (5.0, 60.0), 500, t=(0.0, 0.0, 0.0)),
             _pair(4, (8.0, 30.0), 47, px=0.0, extra=(300, (60.0, 200.0))),
             _pair(5, (8.0, 30.0), 48, px=0.0, extra=(300, (60.0, 200.0))),
             _pair(6, (8.0, 30.0), 49, px=0.0, extra=(300, (60.0, 200.0))),
             _pair(7, (5.0, 60.0), 3)]
    out = _check_pipeline(ctx, pipe, api.default_params(K), pairs, [None, None, None, 47, 48, 49, None])
    assert [bool(out[i]["lm_ran"]) for i in (3, 4, 5)] == [False, True, True]
    # distanceThresh through the pipeline parameters
    for dist, dep in ((3.0, (0.5, 4.0)), (1e4, (20.0, 2e4))):
        prm = api.default_params(K, dist_thresh=dist)
        pairs = [_pair(10 + k, dep, 700, px=0.3 if k else 0.1, near=60) for k in range(3)]
        _check_pipeline(ctx, pipe, prm, pairs)
    pipe.close()
