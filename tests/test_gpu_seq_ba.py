"""epivo_seq_bundle_adjust: the mono windowed bundle adjustment of kitti_ba.cpp:757-905 over the pairs of the last run,
without the per-pair downloads of `ba.match_kp`.

The exact reference is built in numpy from what the pinned per-pair views return (`matches` / `points`, `masks`, the
results): the selection rule of `ba.match_kp`, the first 32 kept points K-normalised elementwise as cam_ * (u, v, 1)
without fusion, the initial chains from the (j, j+1) estimates, then `api.Levenberg_Marquardt_batch` and a numpy
restatement of `ba.finish` with the norm written out.  The device call must return the same bytes.  Against the existing
route (`ba.match_kp` -> `ba.bundle_adjustment`, whose `h @ Kinv.T` may round an ulp differently) the results agree within
test_gpu_ba's tolerances."""
import numpy as np
import pytest

from epivo_b200 import _lib, api, ba, synth
from test_gpu_frames import _parallax

pytestmark = pytest.mark.gpu

FALLBACK_T = np.array([0.1, 0.1, -0.9])


@pytest.fixture(autouse=True)
def _default_lm_shape(monkeypatch):
    monkeypatch.delenv("EPIVO_LM_SHAPE", raising=False)


def window_ws(ws):
    """main(): kitti_ba.cpp:1131-1144."""
    w = []
    for i in range(ws - 1):
        w.append((i, i + 1))
        if i < ws - 2:
            w.append((i, i + 2))
    return w


def _params(K):
    return api.default_params(np.asarray(K, dtype=np.float32), method=api.LMEDS, prob=0.99, threshold=0.1)


def _unfused(px, Kinv):
    u = px[:, 0].astype(np.float64)
    v = px[:, 1].astype(np.float64)
    return np.stack([(Kinv[r, 0] * u + Kinv[r, 1] * v) + Kinv[r, 2] for r in range(3)], axis=1)


def _kept(pipe, res, p, fq, ft, kps):
    """ba.match_kp's selection for pair p: pixels of the E-inliers with rec_mask == 255, and the pair's R, t."""
    if not (res[p]["n_matches"] >= 8 and res[p]["n_inliers"] > 0):
        return np.zeros((0, 2), np.float32), np.zeros((0, 2), np.float32), np.eye(3), FALLBACK_T
    em, pm = pipe.masks(p)
    keep = np.flatnonzero(em == 1)[pm == 255]
    if kps is None:
        a, b = pipe.points(p)
        p0, p1 = a[keep], b[keep]
    else:
        qi, ti, _ = pipe.matches(p)
        p0, p1 = kps[fq][qi[keep]], kps[ft][ti[keep]]
    return p0, p1, res[p]["R"].copy(), res[p]["t"].copy()


def _reference(ctx, pipe, res, pairs, window, stride, F, K, kps=None, huber_delta=1e-5):
    """The exact numpy / primitive-call restatement: (opt_T, lm, reverted, starts, chains, iters, kept counts)."""
    Kinv = np.linalg.inv(np.asarray(K, dtype=np.float64))
    index = {}
    for p, key in enumerate(pairs):
        index.setdefault(key, p)                 # a key listed twice: its first entry
    starts = ba.window_starts(window, stride, F)
    reps = ba.window_reps(window)
    lo = min(min(a, b) for a, b in window)
    hi = max(max(a, b) for a, b in window)
    nz, B, n_rep = hi - lo, len(starts), len(window)
    cache = {}

    def get(key):
        if key not in cache:
            cache[key] = _kept(pipe, res, index[key], key[0], key[1], kps)
        return cache[key]

    T0s = np.tile(np.eye(4), (B, nz, 1, 1))
    pr = np.ones((B, n_rep, 32, 3))
    p_r = np.ones((B, n_rep, 32, 3))
    w = np.zeros((B, n_rep))
    kept = np.zeros((B, n_rep), np.int64)
    for b, i in enumerate(starts):
        for j, (a, c) in enumerate(window):
            p0, p1, _, _ = get((i + a, i + c))
            kept[b, j] = len(p0)
            if len(p0) < 32:
                continue
            w[b, j] = 1.0
            pr[b, j] = _unfused(p0[:32], Kinv)
            p_r[b, j] = _unfused(p1[:32], Kinv)
        for k in range(nz):
            _, _, R, t = get((i + lo + k, i + lo + k + 1))
            T0s[b, k, :3, :3] = R
            T0s[b, k, :3, 3] = t
    opt = np.tile(np.eye(4), (F, 1, 1))
    if B == 0:
        return opt, np.zeros((0, 3)), np.zeros(0, bool), starts, np.zeros((0, nz, 4, 4)), np.zeros(0, np.int32), kept
    T_opt, lm, its = api.Levenberg_Marquardt_batch(nz, 1e-8, reps, w, 1e-2, T0s, pr, p_r, huber_delta=huber_delta,
                                                   ctx=ctx)
    optimized = np.zeros(F, bool)
    reverted = np.zeros(B, bool)
    for b, i in enumerate(starts):                # ba.finish with the norm spelt out: sqrt((x*x + y*y) + z*z)
        w0 = i + lo
        scale = 1.0
        if optimized[w0]:
            x, y, z = opt[w0][0, 3], opt[w0][1, 3], opt[w0][2, 3]
            scale = np.sqrt((x * x + y * y) + z * z)
        Ts = T_opt[b]
        if lm[b, 1] > 1e-2:
            Ts = T0s[b]
            reverted[b] = True
        for k in range(nz):
            opt[w0 + k] = Ts[k]
            opt[w0 + k][:3, 3] /= scale
            optimized[w0 + k] = True
    return opt, lm, reverted, starts, T_opt, its, kept


def _assert_exact(got, want):
    opt, lm, rev, starts, chains, its = got
    o_opt, o_lm, o_rev, o_starts, o_chains, o_its, _ = want
    assert starts == o_starts
    assert chains.tobytes() == o_chains.tobytes()
    assert lm.tobytes() == o_lm.tobytes()
    assert np.array_equal(its, o_its)
    assert np.array_equal(rev, o_rev)
    assert opt.tobytes() == o_opt.tobytes()


def _descriptor_run(ctx, seq, window, stride, counts=None, pairs=None):
    F, kp = seq.kps.shape[:2]
    pairs = ba.window_pairs(window, stride, F) if pairs is None else pairs
    pipe = api.SequencePipeline(F, kp, ctx=ctx, max_pairs=max(len(pairs), F - 1))
    if counts is not None:
        pipe.set_counts(counts)
    pipe.set_pairs([p[0] for p in pairs], [p[1] for p in pairs])
    res = pipe.process(_params(seq.K), seq.kps, seq.descs).copy()
    return pipe, res, pairs


@pytest.fixture(scope="module")
def seq21():
    return synth.make_sequence(21, 800)


@pytest.mark.parametrize("delta", [1e-5, 1.0])
def test_descriptor_route_exact(ctx, seq21, delta):
    """ws = 3, stride 2 (the mono driver's shape): byte-identical with the composed inputs fed to the batched LM."""
    window = window_ws(3)
    pipe, res, pairs = _descriptor_run(ctx, seq21, window, 2)
    got = pipe.bundle_adjust(window, 2, seq21.K, huber_delta=delta, chains=True)
    want = _reference(ctx, pipe, res, pairs, window, 2, 21, seq21.K, kps=seq21.kps, huber_delta=delta)
    _assert_exact(got, want)
    assert got[3] == list(range(0, 19, 2))
    assert (want[6] >= 32).mean() > 0.5          # most reps have their 32 points here
    pipe.close()


def test_equals_existing_route(ctx, seq21):
    """ba.match_kp -> ba.bundle_adjustment on the same data, within test_gpu_ba._compare's tolerances."""
    window = window_ws(3)
    pipe, res, pairs = _descriptor_run(ctx, seq21, window, 2)
    opt, lm, rev, starts = pipe.bundle_adjust(window, 2, seq21.K)
    pipe.close()
    reprojs = ba.match_kp(seq21.kps, seq21.descs, window, 2, seq21.K, ctx=ctx)
    o_opt, o_lm, o_rev, o_starts = ba.bundle_adjustment(reprojs, window, 2, 21, seq21.K, False, 1e-5, ctx=ctx)
    assert starts == o_starts and len(starts) == 10
    assert np.array_equal(rev, o_rev)
    assert opt.shape == o_opt.shape == (21, 4, 4)
    for k in range(len(opt)):
        Rg, Ro, tg, to = opt[k][:3, :3], o_opt[k][:3, :3], opt[k][:3, 3], o_opt[k][:3, 3]
        assert np.arccos(np.clip((np.trace(Rg.T @ Ro) - 1) / 2, -1, 1)) < 1e-4, k
        if np.linalg.norm(to) > 0:
            c = tg @ to / (np.linalg.norm(tg) * np.linalg.norm(to))
            assert np.arccos(np.clip(c, -1, 1)) < 1e-3, k
            assert abs(np.linalg.norm(tg) / np.linalg.norm(to) - 1) < 5e-3, k
        else:
            assert np.linalg.norm(tg) == 0
    ok = np.isfinite(o_lm[:, 1])
    assert np.allclose(lm[ok, 1], o_lm[ok, 1], rtol=1e-4, atol=1e-15)


def test_starved_and_short_pairs(ctx, seq21):
    """Frame 7 keeps 5 keypoints: its pairs have < 8 matches -> identity / (0.1, 0.1, -0.9) and weight-0 reps.  Frames 11
    and 15 keep 40 and 25: some of their pairs have 8..31 kept points -> recoverPose's R, t but weight 0, all-ones rows."""
    window = window_ws(3)
    counts = np.full(21, 800, np.int32)
    counts[7], counts[11], counts[15] = 5, 40, 25
    pipe, res, pairs = _descriptor_run(ctx, seq21, window, 2, counts=counts)
    got = pipe.bundle_adjust(window, 2, seq21.K, chains=True)
    want = _reference(ctx, pipe, res, pairs, window, 2, 21, seq21.K, kps=seq21.kps)
    _assert_exact(got, want)
    idx = {key: p for p, key in reversed(list(enumerate(pairs)))}
    starved = [idx[k] for k in [(6, 7), (7, 8), (5, 7), (7, 9)] if k in idx]
    assert starved and all(res[p]["n_matches"] < 8 for p in starved)
    kept = want[6]
    short = [(b, j) for b, i in enumerate(want[3]) for j, (a, c) in enumerate(window)
             if res[idx[(i + a, i + c)]]["n_matches"] >= 8 and res[idx[(i + a, i + c)]]["n_inliers"] > 0
             and 8 <= kept[b, j] < 32]
    assert short, kept
    pipe.close()


def test_overlapping_windows_scale_carry(ctx, seq21):
    """ws = 4 with stride 1: every window overlaps the previous one, so the scale is carried and the overlap overwritten."""
    window = window_ws(4)
    pipe, res, pairs = _descriptor_run(ctx, seq21, window, 1)
    got = pipe.bundle_adjust(window, 1, seq21.K, chains=True)
    want = _reference(ctx, pipe, res, pairs, window, 1, 21, seq21.K, kps=seq21.kps)
    _assert_exact(got, want)
    assert got[3] == list(range(0, 18))
    pipe.close()


def test_duplicate_key_takes_first_entry(ctx, seq21):
    """A pair list with extra duplicate keys (one in front, one at the end): the first entry of a key is used."""
    window = window_ws(3)
    pairs = ba.window_pairs(window, 2, 21)
    pairs = [(4, 6)] + pairs + [(8, 9)]
    pipe, res, pairs = _descriptor_run(ctx, seq21, window, 2, pairs=pairs)
    got = pipe.bundle_adjust(window, 2, seq21.K, chains=True)
    want = _reference(ctx, pipe, res, pairs, window, 2, 21, seq21.K, kps=seq21.kps)
    _assert_exact(got, want)
    pipe.close()


def test_lk_route_exact(ctx):
    """process_frames over the window pair list: pixels come from the kept tracks (pipe.points)."""
    frames = _parallax(11, 376, 1241, 12)
    window = window_ws(3)
    pairs = ba.window_pairs(window, 2, 11)
    pipe = api.SequencePipeline(11, 4096, ctx=ctx, max_pairs=max(len(pairs), 10))
    pipe.set_pairs([p[0] for p in pairs], [p[1] for p in pairs])
    res = pipe.process_frames(_params(synth.KITTI_K), frames, 40).copy()
    got = pipe.bundle_adjust(window, 2, synth.KITTI_K, chains=True)
    want = _reference(ctx, pipe, res, pairs, window, 2, 11, synth.KITTI_K)
    _assert_exact(got, want)
    assert got[3] == [0, 2, 4, 6, 8]
    assert (want[6] >= 32).any()
    pipe.close()


def _code(fn):
    with pytest.raises(api.EpivoError) as e:
        fn()
    return e.value.code


def test_bad_arguments_launch_nothing(ctx, seq21):
    window = window_ws(3)
    K = seq21.K
    F, kp = seq21.kps.shape[:2]
    pairs = ba.window_pairs(window, 2, F)
    # no run at all
    fresh = api.SequencePipeline(F, kp, ctx=ctx, max_pairs=len(pairs))
    fresh.set_pairs([p[0] for p in pairs], [p[1] for p in pairs])
    before = ctx.launch_count
    assert _code(lambda: fresh.bundle_adjust(window, 2, K, num_frames=F)) == _lib.ERR_INVALID
    assert ctx.launch_count == before
    # a missing pair: the message names it
    missing = [p for p in pairs if p != (4, 6)]
    pipe, res, _ = _descriptor_run(ctx, seq21, window, 2, pairs=missing)
    before = ctx.launch_count
    with pytest.raises(api.EpivoError) as e:
        pipe.bundle_adjust(window, 2, K)
    assert e.value.code == _lib.ERR_INVALID and "(4,6)" in str(e.value)
    assert ctx.launch_count == before
    pipe.close()
    # a pair outside the last run: run only the first half of the list
    pipe = api.SequencePipeline(F, kp, ctx=ctx, max_pairs=len(pairs))
    pipe.set_pairs([p[0] for p in pairs], [p[1] for p in pairs])
    pipe.upload(seq21.kps, seq21.descs)
    pipe.run(_params(K), 0, len(pairs) // 2)
    ctx.sync()
    before = ctx.launch_count
    assert _code(lambda: pipe.bundle_adjust(window, 2, K, num_frames=F)) == _lib.ERR_INVALID
    assert ctx.launch_count == before
    pipe.close()
    # the other refusals on a pipeline whose last run is valid
    pipe, res, _ = _descriptor_run(ctx, seq21, window, 2)
    before = ctx.launch_count
    codes = [
        _code(lambda: pipe.bundle_adjust([(0, 1), (1, 1)], 2, K)),           # first == second
        _code(lambda: pipe.bundle_adjust([(0, 1), (-1, 1)], 2, K)),          # negative offset
        _code(lambda: pipe.bundle_adjust(window, 0, K)),                     # stride < 1
        _code(lambda: pipe.bundle_adjust(window, 2, K, num_frames=1)),       # num_frames outside [2, max_frames]
        _code(lambda: pipe.bundle_adjust(window, 2, K, num_frames=F + 1)),
    ]
    assert codes == [_lib.ERR_INVALID] * 5
    assert _code(lambda: pipe.bundle_adjust([(0, 1), (0, 40)], 2, K)) == _lib.ERR_UNSUPPORTED     # n_zeta = 40
    assert ctx.launch_count == before
    # no window fits: identity, no window, nothing launched
    opt, lm, rev, starts = pipe.bundle_adjust(window, 2, K, num_frames=2)
    assert starts == [] and lm.shape == (0, 3) and rev.shape == (0,)
    assert np.array_equal(opt, np.tile(np.eye(4), (2, 1, 1)))
    assert ctx.launch_count == before
    # a new pair list invalidates the last run
    pipe.set_pairs([p[0] for p in pairs], [p[1] for p in pairs])
    assert _code(lambda: pipe.bundle_adjust(window, 2, K)) == _lib.ERR_INVALID
    # a last run of process_points keeps no pixels
    pts = [np.zeros((8, 2), np.float32)] * len(pairs)
    pipe.process_points(_params(K), pts, pts)
    before = ctx.launch_count
    assert _code(lambda: pipe.bundle_adjust(window, 2, K)) == _lib.ERR_INVALID
    assert ctx.launch_count == before
    pipe.close()
    fresh.close()
