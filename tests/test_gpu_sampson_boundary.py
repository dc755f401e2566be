"""The Sampson inlier decision AT the threshold, on every GPU scoring path, against the oracle.

Points and models come from tests/sampson_boundary.py: pairs the oracle decides differently one ulp apart, whose
quotients lie within 2e-6 (point-tuned) or 2^-50 (model-tuned) of B -- past the fused pre-filter, into the exact
sign test and the division (test_oracle_sampson_boundary.py shows that on the host).  Paths:
    scoreSampson           score_count_kernel's warp-uniform fallback (per-model hdmin), mask_of_model_kernel
    findEssentialMat       ess_round_kernel: count_one / count_two recounts, the bounded pass, the final mask
    process_points         the same kernels through the sequence pipeline (per-pair stride)
"""
import numpy as np
import pytest

import sampson_boundary as SB
from epivo_b200 import api, synth
from oracle import oracle as O

pytestmark = pytest.mark.gpu
PK = SB.POW2_K
PSIZE = SB.IMAGE["pow2"]


def _ppt(n):
    """score_count_kernel's correspondences per thread for n points (epv_score_launch)"""
    ppt, best = 6, 0
    for c in (6, 5, 4):
        slots = -(-n // (256 * c)) * c
        if c == 6 or slots < best:
            ppt, best = c, slots
    return ppt


def _scene(n, seed, outliers=0):
    """n correspondences of a forward-moving camera (POW2_K), the last `outliers` of them random"""
    pr = synth.make_pair(seed=seed, n=3 * n, K=PK, size=PSIZE, outlier_frac=0.0, px_sigma=0.3)
    keep = np.nonzero(pr.gt_match >= 0)[0]
    ok = (pr.kp1[pr.gt_match[keep]] >= 0).all(1) & (pr.kp1[pr.gt_match[keep]] < PSIZE).all(1)
    keep = keep[ok][:n]
    assert len(keep) == n
    p0 = pr.kp0[keep].astype(np.float32).copy()
    p1 = pr.kp1[pr.gt_match[keep]].astype(np.float32).copy()
    rng = np.random.default_rng(seed)
    if outliers:
        p1[n - outliers:] = rng.uniform((0, 0), PSIZE, (outliers, 2)).astype(np.float32)
    return p0, p1


class _GpuSolver:
    """The oracle's RANSAC / LMedS loop run on the GPU solver's models (the models of a sample depend only on its
    five points, so they are the bits the round kernel scores)."""

    def __init__(self, ctx):
        self.ctx = ctx

    def __call__(self, x1, x2):
        return api.fivePoint(x1[None], x2[None], ctx=self.ctx)[0]


def _oracle(ctx, p0, p1, method, prob, thr, S, max_iters=1000):
    return O.find_essential_mat(p0, p1, PK, method, prob, thr, max_iters, samples=S, solver=_GpuSolver(ctx))


def _check_call(ctx, p0, p1, method, prob, thr, S, max_iters=1000):
    E, mask, info = api.findEssentialMat(p0, p1, PK, method, prob, thr, max_iters, samples=S, ctx=ctx,
                                         return_info=True)
    Eo, mo, io = _oracle(ctx, p0, p1, method, prob, thr, S, max_iters)
    assert E is not None and np.array_equal(E.reshape(9), np.asarray(Eo).reshape(9))      # the scored model, bit for bit
    assert np.array_equal(mask, mo)
    assert info["n_inliers"] == int(mo.sum())
    assert info["iters"] == io["iters"]
    return E.reshape(9), mask, info


def _place(p0, p1, idx, straddles, variants):
    """correspondence idx[i] := straddle i, as its inlier (True) or outlier (False) variant"""
    p0, p1 = p0.copy(), p1.copy()
    for i, s, v in zip(idx, straddles, variants):
        p0[i] = s.p1
        p1[i] = s.p2_in if v else s.p2_out
    return p0, p1


# ---- scoreSampson: model-tuned straddles, several model tiles, SC_PPT 4 / 5 / 6 with a ragged last tile ----------

@pytest.mark.parametrize("n,ppt", [(1998, 4), (2500, 5), (3000, 6)])
@pytest.mark.parametrize("cam", ["kitti", "euroc"])
def test_score_sampson_model_straddles(ctx, cam, n, ppt):
    K = {"kitti": SB.KITTI_K, "euroc": SB.EUROC_K}[cam]
    assert _ppt(n) == ppt and n % (256 * ppt)
    W, H = SB.IMAGE[cam]
    rng = np.random.default_rng(n)
    for i, thr in enumerate(SB.thresholds(K)):
        st = SB.model_straddles(K, thr, 24, 1000 * i + n, (W, H))
        base = np.concatenate([np.stack([s.E_in, s.E_out]) for s in st])
        Es = np.concatenate([base, -3.0 * base, 1e-3 * base, 1e3 * base])          # 192 models: two tiles at least
        p0 = rng.uniform((0, 0), (W, H), (n, 2)).astype(np.float32)
        p1 = rng.uniform((0, 0), (W, H), (n, 2)).astype(np.float32)
        at = rng.choice(n, len(st), replace=False)
        p0[at] = [s.p1 for s in st]
        p1[at] = [s.p2 for s in st]
        counts, med, best, mask = api.scoreSampson(Es, p0, p1, K, thr, ctx=ctx)
        x1, x2 = O.normalize_points(p0, K), O.normalize_points(p1, K)
        t = O.ransac_threshold(thr, K)
        oc, om = O.score_models(Es, x1, x2, t)
        assert np.array_equal(counts, oc), (thr, np.nonzero(counts != oc)[0][:8])
        assert np.array_equal(med, om)
        assert best == int(np.argmax(oc))                                          # first maximum
        assert np.array_equal(mask, O.find_inliers(O.sampson_err_f32(Es[best], x1, x2), t))


def test_score_sampson_point_straddles(ctx):
    """One unit model and its scaled copies against its point-tuned straddles: the counts and the exact-path
    mask of the first maximum."""
    rng = np.random.default_rng(17)
    E = SB.unit_essential(4)
    Es = np.stack([E, -3.0 * E, 1e-3 * E, 1e3 * E, 0.5 * E])
    for i, thr in enumerate(SB.thresholds(PK)):
        thr32 = SB.thr32_of(thr, PK)
        st = SB.point_straddles(E, PK, thr32, 48, 50 + i, PSIZE)
        variants = rng.integers(0, 2, len(st)).astype(bool)
        p0 = rng.uniform((0, 0), PSIZE, (700, 2)).astype(np.float32)
        p1 = rng.uniform((0, 0), PSIZE, (700, 2)).astype(np.float32)
        at = rng.choice(700, len(st), replace=False)
        p0, p1 = _place(p0, p1, at, st, variants)
        counts, _, best, mask = api.scoreSampson(Es, p0, p1, PK, thr, ctx=ctx, medians=False)
        x1, x2 = O.normalize_points(p0, PK), O.normalize_points(p1, PK)
        t = O.ransac_threshold(thr, PK)
        oc, _ = O.score_models(Es, x1, x2, t)
        assert np.array_equal(counts, oc)
        assert best == int(np.argmax(oc))
        om = O.find_inliers(O.sampson_err_f32(Es[best], x1, x2), t)
        assert np.array_equal(mask, om)
        if best == 0:
            assert np.array_equal(mask[at].astype(bool), variants)


# ---- findEssentialMat with injected samples: ess_round_kernel ------------------------------------------------

@pytest.mark.parametrize("n", [400, 20000])              # points staged in shared memory / read from global memory
def test_find_essential_point_straddles(ctx, n):
    p0, p1 = _scene(n, 300 + n)
    S = np.arange(15, dtype=np.int32).reshape(3, 5)
    rng = np.random.default_rng(n)
    for i, thr in enumerate(SB.thresholds(PK)):
        E, _, _ = _check_call(ctx, p0, p1, api.RANSAC, 0.99, thr, S)
        st = SB.point_straddles(E, PK, SB.thr32_of(thr, PK), 48, 7 + i, PSIZE)
        variants = rng.integers(0, 2, len(st)).astype(bool)
        at = 15 + rng.choice(n - 15, len(st), replace=False)            # never a sample point: same models
        q0, q1 = _place(p0, p1, at, st, variants)
        E2, mask, _ = _check_call(ctx, q0, q1, api.RANSAC, 0.99, thr, S)
        assert np.array_equal(E2, E)
        assert np.array_equal(mask[at].astype(bool), variants)


def _models(ctx, p0, p1, s):
    x1, x2 = O.normalize_points(p0[s], PK), O.normalize_points(p1[s], PK)
    return api.fivePoint(x1[None], x2[None], ctx=ctx)[0].reshape(-1, 9)


def test_find_essential_strictly_better(ctx):
    """Model B (sample 8, the second sub-chunk) ties model A (sample 0) and must not win; one more inlier of B --
    a straddle of B switched to its inlier variant -- and it must win.  The deciding points are straddles of B
    that A decides with a margin, so only B's count moves."""
    n_good, n_out = 300, 60
    p0, p1 = _scene(n_good + n_out, 77, outliers=n_out)          # the deciding points are appended to these
    thr, prob = 1.0, 0.99
    thr32 = SB.thr32_of(thr, PK)
    T = SB.samp_thr(thr32)
    good = np.arange(n_good)
    outl = np.arange(n_good, n_good + n_out)
    rng = np.random.default_rng(5)
    x1, x2 = O.normalize_points(p0, PK), O.normalize_points(p1, PK)

    def count(E):
        return int(O.find_inliers(O.sampson_err_f32(E, x1, x2), O.ransac_threshold(thr, PK)).sum())

    # A: the model with the most inliers among the best models of the first ten samples of good points
    cands = []
    for j in range(10):
        sA = good[5 * j:5 * j + 5]
        E1, _ = api.findEssentialMat(p0, p1, PK, api.RANSAC, prob, thr, samples=sA[None], ctx=ctx)
        cands.append((count(E1), j, E1.reshape(9)))
    cA0, j, EA = max(cands, key=lambda c: (c[0], -c[1]))
    sA = good[5 * j:5 * j + 5]
    # B: the best model of a later good sample with a few inliers fewer than A, at an even position among that
    # sample's models (the first model of a pair in count_two)
    for tries in range(10, 60):
        sB = good[5 * tries:5 * tries + 5]
        EB, _ = api.findEssentialMat(p0, p1, PK, api.RANSAC, prob, thr, samples=sB[None], ctx=ctx)
        pos = [k for k, M in enumerate(_models(ctx, p0, p1, sB)) if np.array_equal(M, EB.reshape(9))]
        assert len(pos) == 1                                        # the scored model is the solver's, bit for bit
        if pos[0] % 2 == 0 and 0 <= cA0 - count(EB) <= 25:
            break
    else:
        pytest.fail("no suitable second sample")
    EB = EB.reshape(9)
    cB0 = count(EB)
    fill = [rng.choice(outl, 5, replace=False) for _ in range(22)]
    S = np.stack([sA] + fill[:7] + [sB] + fill[7:]).astype(np.int32)         # A at 0, B at 8 (second sub-chunk)

    # deciding points: k + 1 straddles of B that A rejects, clear of A's boundary by 10x the pre-filter band.  The tie
    # takes k of them as B's inliers and one as an outlier; one more inlier switches the last one.  Every one of them
    # is left open by B's pre-filter, so at the end of B's bounded pass "decided inliers + undecided" is exactly
    # the bound + 1 in both calls: only the recount tells a tie from a win.
    k = cA0 - cB0
    chosen = []
    for s in SB.point_straddles(EB, PK, thr32, 4 * k + 16, 9, PSIZE):
        xs = [np.concatenate([O.normalize_points(s.p1[None], PK)[0], O.normalize_points(p[None], PK)[0]])
              for p in (s.p2_in, s.p2_out)]
        if min(SB.rel_to_B(EA, x, T) for x in xs) > 10 * SB.REL_TIER2 and not any(SB.inlier(EA, x, thr32) for x in xs):
            chosen.append(s)
    chosen = chosen[:k + 1]
    assert len(chosen) == k + 1
    n = len(p0) + len(chosen)
    dec = np.arange(len(p0), n)
    # a prob for which RANSACUpdateNumIters, after A, stops the loop past the second sub-chunk but before the end
    cA = cA0
    prob = next(p for p in (0.99, 0.995, 0.98, 0.999, 0.95, 0.9)
                if 17 <= O.ransac_update_num_iters(p, (n - cA) / n, 5, len(S)) < len(S))
    z = np.zeros((len(chosen), 2), np.float32)
    for extra, winner in ((0, EA), (1, EB)):
        variants = np.zeros(len(chosen), bool)
        variants[:k + extra] = True
        q0, q1 = _place(np.concatenate([p0, z]), np.concatenate([p1, z]), dec, chosen, variants)
        E, mask, info = _check_call(ctx, q0, q1, api.RANSAC, prob, thr, S)
        assert np.array_equal(E, winner), extra
        assert info["n_inliers"] == cA + extra                      # the winner's count
        assert info["iters"] < len(S)                               # RANSACUpdateNumIters ended the loop


def test_lmeds_final_mask_straddles(ctx):
    """LMedS: straddles at thr32 = float(sigma^2) of the best median.  Placeholders and replacements both lie
    above the median, so the median -- and the threshold -- is the same in both calls."""
    n, n_dec = 400, 40
    p0, p1 = _scene(n, 91, outliers=60)
    S = np.arange(5, dtype=np.int32)[None]
    dec = np.arange(n - n_dec, n)
    rng = np.random.default_rng(3)
    p1[dec] = np.clip(p0[dec] + rng.uniform(40, 80, (n_dec, 2)), 0, 399).astype(np.float32)      # far off any line
    E, _, _ = _check_call(ctx, p0, p1, api.LMEDS, 0.99, 0.0, S)
    x1, x2 = O.normalize_points(p0, PK), O.normalize_points(p1, PK)
    err = O.sampson_err_f32(E, x1, x2)
    med = O.lmeds_median(err)
    assert (err[dec] > med).all()
    sigma = O.lmeds_sigma(med, n)
    thr32 = np.float32(sigma * sigma)
    st = SB.point_straddles(E, PK, thr32, n_dec, 21, PSIZE)
    variants = rng.integers(0, 2, n_dec).astype(bool)
    q0, q1 = _place(p0, p1, dec, st, variants)
    E2, mask, _ = _check_call(ctx, q0, q1, api.LMEDS, 0.99, 0.0, S)
    err2 = O.sampson_err_f32(E, O.normalize_points(q0, PK), O.normalize_points(q1, PK))
    assert O.lmeds_median(err2) == med and (err2[dec] > med).all()
    assert np.array_equal(E2, E)
    assert np.array_equal(mask[dec].astype(bool), variants)


# ---- the sequence pipeline ---------------------------------------------------------------------------------

def test_pipeline_point_straddles(ctx):
    """process_points shares the essential kernels with a per-pair row stride: pair 1 is shorter than pair 0.  The
    outliers of each pair's model that no sample of the first 64 draws touches are replaced by straddles of that
    model, so the models are unchanged and the model gains inliers only: it stays the winner.  The whole call
    against the oracle's loop over OpenCV's sample stream, on the GPU solver's models."""
    thr = 0.3
    prm = api.default_params(PK, threshold=thr)
    sizes = (500, 360)
    pts = [_scene(m, 500 + m, outliers=80) for m in sizes]
    pipe = api.SequencePipeline(3, max(sizes), ctx=ctx)
    out1 = pipe.process_points(prm, [p[0] for p in pts], [p[1] for p in pts]).copy()
    rng = np.random.default_rng(8)
    placed = []
    for i, (m, (p0, p1)) in enumerate(zip(sizes, pts)):
        assert out1[i]["ransac_iters"] < 64
        E = out1[i]["E"].reshape(9)
        em, _ = pipe.masks(i)
        free = np.setdiff1d(np.nonzero(em == 0)[0], O.generate_samples(m, 64))
        st = SB.point_straddles(E, PK, SB.thr32_of(thr, PK), 24, 30 + i, PSIZE)
        at = rng.choice(free, len(st), replace=False)
        variants = np.arange(len(st)) >= 4                           # 20 inliers, 4 outliers of the model
        placed.append((at, variants, *_place(p0, p1, at, st, variants)))
    out2 = pipe.process_points(prm, [p[2] for p in placed], [p[3] for p in placed])
    for i, (at, variants, q0, q1) in enumerate(placed):
        Eo, mo, io = O.find_essential_mat(q0, q1, PK, api.RANSAC, prm.prob, thr, prm.max_iters, solver=_GpuSolver(ctx))
        em, _ = pipe.masks(i)
        assert np.array_equal(out2[i]["E"].reshape(9), np.asarray(Eo).reshape(9))
        assert np.array_equal(out2[i]["E"].reshape(9), out1[i]["E"].reshape(9))
        assert np.array_equal(em, mo)
        assert out2[i]["n_inliers"] == int(mo.sum()) and out2[i]["ransac_iters"] == io["iters"]
        assert np.array_equal(em[at].astype(bool), variants)
    pipe.close()
