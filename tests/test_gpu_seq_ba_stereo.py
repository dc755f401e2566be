"""epivo_seq_bundle_adjust_stereo: the stereo windowed bundle adjustment of kitti_ba.cpp:908-1068 over the pairs of the last
run.  Frame f of the rig is node 2f (left) and 2f + 1 (right); the frame slots of the sequence are the nodes.

The exact reference is a numpy restatement built from what the pinned per-pair views return, with test_gpu_seq_ba's
selection rule (`_kept`) and unfused K-normalisation (`_unfused`): the stereo window expansion, window starts in frames
with node step 2, a full rep weighted by its pair's weight (and its real rows even when that weight is 0), the initial
chains from the (j, j+1) node pairs, then `api.Levenberg_Marquardt_batch` and `ba.finish` without the scale carry.  The
device call must return the same bytes.  Against the composed route (`ba.match_kp` -> reproj.w -> `ba.bundle_adjustment(
stereo=True)`) the results agree within test_gpu_ba's tolerances."""
import numpy as np
import pytest

from epivo_b200 import _lib, api, ba, synth
from test_gpu_frames import _parallax
from test_gpu_seq_ba import _code, _kept, _params, _unfused, window_ws

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _default_lm_shape(monkeypatch):
    monkeypatch.delenv("EPIVO_LM_SHAPE", raising=False)


def _stereo_pairs(window, stride, F):
    """The node pair list of the stereo driver: every key its windows read, chain pairs (2f+1, 2f+2) included."""
    return ba.window_pairs(ba.expand_stereo_window(window), 2 * stride, 2 * F)


def _rig_weights(pairs):
    """The driver's reproj.w: 0 on the left -> right pairs (2f, 2f+1), which freezes the rig extrinsics."""
    return np.array([0.0 if a % 2 == 0 and b == a + 1 else 1.0 for a, b in pairs])


def _reference(ctx, pipe, res, pairs, window, stride, F, K, pw=None, kps=None, huber_delta=1e-5):
    """The exact restatement: (opt_T, lm, reverted, starts, chains, iters, kept counts, rep weights, T0s)."""
    Kinv = np.linalg.inv(np.asarray(K, dtype=np.float64))
    index = {}
    for p, key in enumerate(pairs):
        index.setdefault(key, p)                 # a key listed twice: its first entry, for the points and the weight
    win = ba.expand_stereo_window(window)
    starts = ba.window_starts(win, stride, 2 * F, 2)
    reps = ba.window_reps(win)
    lo = min(min(a, b) for a, b in win)
    hi = max(max(a, b) for a, b in win)
    nz, B, n_rep = hi - lo, len(starts), len(win)
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
        base = 2 * i
        for j, (a, c) in enumerate(win):
            key = (base + a, base + c)
            p0, p1, _, _ = get(key)
            kept[b, j] = len(p0)
            if len(p0) < 32:
                continue
            w[b, j] = 1.0 if pw is None else pw[index[key]]
            pr[b, j] = _unfused(p0[:32], Kinv)
            p_r[b, j] = _unfused(p1[:32], Kinv)
        for k in range(nz):
            _, _, R, t = get((base + lo + k, base + lo + k + 1))
            T0s[b, k, :3, :3] = R
            T0s[b, k, :3, 3] = t
    opt = np.tile(np.eye(4), (2 * F, 1, 1))
    if B == 0:
        return opt, np.zeros((0, 3)), np.zeros(0, bool), starts, np.zeros((0, nz, 4, 4)), np.zeros(0, np.int32), kept, w, T0s
    T_opt, lm, its = api.Levenberg_Marquardt_batch(nz, 1e-8, reps, w, 1e-2, T0s, pr, p_r, huber_delta=huber_delta,
                                                   ctx=ctx)
    reverted = np.zeros(B, bool)
    for b, i in enumerate(starts):                # ba.finish, stereo: no scale carry
        Ts = T_opt[b]
        if lm[b, 1] > 1e-2:
            Ts = T0s[b]
            reverted[b] = True
        for k in range(nz):
            opt[2 * i + lo + k] = Ts[k]
    return opt, lm, reverted, starts, T_opt, its, kept, w, T0s


def _assert_exact(got, want):
    opt, lm, rev, starts, chains, its = got
    o_opt, o_lm, o_rev, o_starts, o_chains, o_its = want[:6]
    assert starts == o_starts
    assert chains.tobytes() == o_chains.tobytes()
    assert lm.tobytes() == o_lm.tobytes()
    assert np.array_equal(its, o_its)
    assert np.array_equal(rev, o_rev)
    assert opt.tobytes() == o_opt.tobytes()


def _descriptor_run(ctx, seq, pairs, counts=None):
    F, kp = seq.kps.shape[:2]
    pipe = api.SequencePipeline(F, kp, ctx=ctx, max_pairs=max(len(pairs), F - 1))
    if counts is not None:
        pipe.set_counts(counts)
    pipe.set_pairs([p[0] for p in pairs], [p[1] for p in pairs])
    res = pipe.process(_params(seq.K), seq.kps, seq.descs).copy()
    return pipe, res


@pytest.fixture(scope="module")
def seq22():
    """11 stereo frames = 22 nodes."""
    return synth.make_sequence(22, 800)


@pytest.mark.parametrize("delta", [1e-5, 1.0])
def test_descriptor_route_exact(ctx, seq22, delta):
    """The shipped shape, ws = 3, stride 2, weight 0 on every (2f, 2f+1): 9 reps over n_zeta = 4, byte-identical with the
    composed inputs fed to the batched LM."""
    window = window_ws(3)
    pairs = _stereo_pairs(window, 2, 11)
    pw = _rig_weights(pairs)
    pipe, res = _descriptor_run(ctx, seq22, pairs)
    got = pipe.bundle_adjust_stereo(window, 2, seq22.K, pair_weights=pw, huber_delta=delta, chains=True)
    want = _reference(ctx, pipe, res, pairs, window, 2, 11, seq22.K, pw=pw, kps=seq22.kps, huber_delta=delta)
    _assert_exact(got, want)
    assert got[3] == [0, 2, 4, 6, 8] and got[0].shape == (22, 4, 4) and got[4].shape == (5, 4, 4, 4)
    kept, w = want[6], want[7]
    assert ((kept >= 32) & (w == 0)).any()       # full reps with weight 0: real rows, zero weight
    assert ((kept >= 32) & (w == 1)).any()
    pipe.close()


def test_weights_pass_through(ctx, seq22):
    """pair_weights None is 1.0 everywhere; a non-binary weight reaches the LM as its value.  Both differ from the
    rig-frozen run."""
    window = window_ws(3)
    pairs = _stereo_pairs(window, 2, 11)
    pipe, res = _descriptor_run(ctx, seq22, pairs)
    frozen = pipe.bundle_adjust_stereo(window, 2, seq22.K, pair_weights=_rig_weights(pairs), chains=True)
    ones = pipe.bundle_adjust_stereo(window, 2, seq22.K, chains=True)
    _assert_exact(ones, _reference(ctx, pipe, res, pairs, window, 2, 11, seq22.K, kps=seq22.kps))
    half = _rig_weights(pairs)
    half[1::3] = 0.5
    got = pipe.bundle_adjust_stereo(window, 2, seq22.K, pair_weights=half, chains=True)
    want = _reference(ctx, pipe, res, pairs, window, 2, 11, seq22.K, pw=half, kps=seq22.kps)
    _assert_exact(got, want)
    assert ((want[6] >= 32) & (want[7] == 0.5)).any()
    assert ones[4].tobytes() != frozen[4].tobytes()
    assert got[4].tobytes() != frozen[4].tobytes()
    pipe.close()


def test_starved_and_short_nodes(ctx, seq22):
    """Node 7 keeps 5 keypoints: its pairs have < 8 matches -> identity / (0.1, 0.1, -0.9).  Nodes 10 and 14 keep 40 and
    25: some of their pairs have 8..31 kept points -> recoverPose's R, t, all-ones rows.  Both weigh 0 with pair weight 1."""
    window = window_ws(3)
    pairs = _stereo_pairs(window, 2, 11)
    counts = np.full(22, 800, np.int32)
    counts[7], counts[10], counts[14] = 5, 40, 25
    pipe, res = _descriptor_run(ctx, seq22, pairs, counts=counts)
    got = pipe.bundle_adjust_stereo(window, 2, seq22.K, chains=True)
    want = _reference(ctx, pipe, res, pairs, window, 2, 11, seq22.K, kps=seq22.kps)
    _assert_exact(got, want)
    idx = {key: p for p, key in reversed(list(enumerate(pairs)))}
    starved = [idx[k] for k in [(6, 7), (7, 8), (5, 7), (7, 9), (7, 10)] if k in idx]
    assert starved and all(res[p]["n_matches"] < 8 for p in starved)
    kept, w = want[6], want[7]
    win = ba.expand_stereo_window(window)
    short = [(b, j) for b, i in enumerate(want[3]) for j, (a, c) in enumerate(win)
             if res[idx[(2 * i + a, 2 * i + c)]]["n_matches"] >= 8 and res[idx[(2 * i + a, 2 * i + c)]]["n_inliers"] > 0
             and 8 <= kept[b, j] < 32]
    assert short, kept
    assert all(w[b, j] == 0 for b, j in short)
    pipe.close()


def test_overlap_without_scale_carry(ctx, seq22):
    """ws = 3, stride 1: every window overlaps the previous one and overwrites it, with its translations unscaled."""
    window = window_ws(3)
    pairs = _stereo_pairs(window, 1, 11)
    pw = _rig_weights(pairs)
    pipe, res = _descriptor_run(ctx, seq22, pairs)
    got = pipe.bundle_adjust_stereo(window, 1, seq22.K, pair_weights=pw, chains=True)
    want = _reference(ctx, pipe, res, pairs, window, 1, 11, seq22.K, pw=pw, kps=seq22.kps)
    _assert_exact(got, want)
    opt, _, rev, starts, chains, _ = got
    assert starts == list(range(9))
    T0s = want[8]
    for node in range(2 * starts[-1] + 4):      # the last window reaching a node wrote it, as its chain says
        b = max(b for b, i in enumerate(starts) if 2 * i <= node < 2 * i + 4)
        src = T0s[b] if rev[b] else chains[b]
        assert opt[node].tobytes() == src[node - 2 * starts[b]].tobytes(), node
    # the mono tail would divide window b by the norm its start node has after window b - 1: that is not 1 here
    carried = [np.linalg.norm((T0s[b - 1] if rev[b - 1] else chains[b - 1])[2][:3, 3]) for b in range(1, len(starts))]
    assert any(s != 1.0 for s in carried)
    pipe.close()


def test_duplicate_key_takes_first_entry(ctx, seq22):
    """Extra duplicate keys, one in front with its own weight and one at the end: the first entry of a key gives both the
    points and the weight."""
    window = window_ws(3)
    pairs = [(4, 6)] + _stereo_pairs(window, 2, 11) + [(9, 10)]
    pw = _rig_weights(pairs)
    pw[0] = 0.25                                  # the later (4, 6) entry keeps weight 1
    pw[-1] = 0.75
    pipe, res = _descriptor_run(ctx, seq22, pairs)
    got = pipe.bundle_adjust_stereo(window, 2, seq22.K, pair_weights=pw, chains=True)
    want = _reference(ctx, pipe, res, pairs, window, 2, 11, seq22.K, pw=pw, kps=seq22.kps)
    _assert_exact(got, want)
    assert (want[7] == 0.25).any() and not (want[7] == 0.75).any()
    pipe.close()


def test_lk_route_exact(ctx):
    """process_frames over 12 node frames with the stereo pair list: pixels come from the kept tracks (pipe.points)."""
    frames = _parallax(12, 376, 1241, 12)
    window = window_ws(3)
    pairs = _stereo_pairs(window, 2, 6)
    pw = _rig_weights(pairs)
    pipe = api.SequencePipeline(12, 4096, ctx=ctx, max_pairs=max(len(pairs), 11))
    pipe.set_pairs([p[0] for p in pairs], [p[1] for p in pairs])
    res = pipe.process_frames(_params(synth.KITTI_K), frames, 40).copy()
    got = pipe.bundle_adjust_stereo(window, 2, synth.KITTI_K, pair_weights=pw, chains=True)
    want = _reference(ctx, pipe, res, pairs, window, 2, 6, synth.KITTI_K, pw=pw)
    _assert_exact(got, want)
    assert got[3] == [0, 2] and got[0].shape == (12, 4, 4)
    assert (want[6] >= 32).any()
    pipe.close()


def test_equals_composed_route(ctx, seq22):
    """ba.match_kp -> reproj.w -> ba.bundle_adjustment(stereo=True) on the same data, within test_gpu_ba's tolerances."""
    window = window_ws(3)
    pairs = _stereo_pairs(window, 2, 11)
    pipe, res = _descriptor_run(ctx, seq22, pairs)
    opt, lm, rev, starts = pipe.bundle_adjust_stereo(window, 2, seq22.K, pair_weights=_rig_weights(pairs))
    pipe.close()
    reprojs = ba.match_kp(seq22.kps, seq22.descs, ba.expand_stereo_window(window), 4, seq22.K, ctx=ctx)
    for (a, b), r in reprojs.items():
        r.w = 0.0 if a % 2 == 0 and b == a + 1 else 1.0
    o_opt, o_lm, o_rev, o_starts = ba.bundle_adjustment(reprojs, window, 2, 11, seq22.K, True, 1e-5, ctx=ctx)
    assert starts == o_starts and len(starts) == 5
    assert np.array_equal(rev, o_rev)
    assert opt.shape == o_opt.shape == (22, 4, 4)
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


def test_bad_arguments_launch_nothing(ctx):
    seq = synth.make_sequence(40, 300)           # 20 stereo frames: room for a window too large for the LM
    window = window_ws(3)
    K = seq.K
    nodes, kp = seq.kps.shape[:2]
    F = nodes // 2
    pairs = _stereo_pairs(window, 2, F)
    # no run at all
    fresh = api.SequencePipeline(nodes, kp, ctx=ctx, max_pairs=len(pairs))
    fresh.set_pairs([p[0] for p in pairs], [p[1] for p in pairs])
    before = ctx.launch_count
    assert _code(lambda: fresh.bundle_adjust_stereo(window, 2, K, num_frames=F)) == _lib.ERR_INVALID
    assert ctx.launch_count == before
    # missing pairs, named in the message: a rep pair and a chain pair (2f+1, 2f+2)
    for gone in [(4, 8), (5, 6)]:
        pipe, _ = _descriptor_run(ctx, seq, [p for p in pairs if p != gone])
        before = ctx.launch_count
        with pytest.raises(api.EpivoError) as e:
            pipe.bundle_adjust_stereo(window, 2, K)
        assert e.value.code == _lib.ERR_INVALID and "(%d,%d)" % gone in str(e.value)
        assert ctx.launch_count == before
        pipe.close()
    # a pair outside the last run: run only the first half of the list
    pipe = api.SequencePipeline(nodes, kp, ctx=ctx, max_pairs=len(pairs))
    pipe.set_pairs([p[0] for p in pairs], [p[1] for p in pairs])
    pipe.upload(seq.kps, seq.descs)
    pipe.run(_params(K), 0, len(pairs) // 2)
    ctx.sync()
    before = ctx.launch_count
    assert _code(lambda: pipe.bundle_adjust_stereo(window, 2, K, num_frames=F)) == _lib.ERR_INVALID
    assert ctx.launch_count == before
    pipe.close()
    # the other refusals on a pipeline whose last run is valid
    pipe, _ = _descriptor_run(ctx, seq, pairs)
    before = ctx.launch_count
    nan_w, inf_w = np.ones(len(pairs)), np.ones(len(pairs))
    nan_w[3], inf_w[-1] = np.nan, np.inf
    codes = [
        _code(lambda: pipe.bundle_adjust_stereo([(0, 1), (1, 1)], 2, K)),           # first == second
        _code(lambda: pipe.bundle_adjust_stereo([(0, 1), (-1, 1)], 2, K)),          # negative offset
        _code(lambda: pipe.bundle_adjust_stereo([(0, 1), (0, F)], 2, K)),           # offset past the frames
        _code(lambda: pipe.bundle_adjust_stereo(window, 0, K)),                     # stride < 1
        _code(lambda: pipe.bundle_adjust_stereo(window, 2, K, num_frames=1)),       # num_frames outside [2, max_frames / 2]
        _code(lambda: pipe.bundle_adjust_stereo(window, 2, K, num_frames=F + 1)),
        _code(lambda: pipe.bundle_adjust_stereo(window, 2, K, pair_weights=nan_w)),  # non-finite weights
        _code(lambda: pipe.bundle_adjust_stereo(window, 2, K, pair_weights=inf_w)),
    ]
    assert codes == [_lib.ERR_INVALID] * 8
    # (0, 19) expands to n_zeta = 38 nodes
    assert _code(lambda: pipe.bundle_adjust_stereo([(0, 1), (0, 19)], 2, K)) == _lib.ERR_UNSUPPORTED
    with pytest.raises(ValueError):
        pipe.bundle_adjust_stereo(window, 2, K, pair_weights=np.ones(len(pairs) - 1))
    assert ctx.launch_count == before
    # no window fits: identity for the 2 * num_frames nodes, no window, nothing launched
    opt, lm, rev, starts = pipe.bundle_adjust_stereo(window, 2, K, num_frames=2)
    assert starts == [] and lm.shape == (0, 3) and rev.shape == (0,)
    assert np.array_equal(opt, np.tile(np.eye(4), (4, 1, 1)))
    assert ctx.launch_count == before
    # a new pair list invalidates the last run
    pipe.set_pairs([p[0] for p in pairs], [p[1] for p in pairs])
    assert _code(lambda: pipe.bundle_adjust_stereo(window, 2, K)) == _lib.ERR_INVALID
    # a last run of process_points keeps no pixels
    pts = [np.zeros((8, 2), np.float32)] * len(pairs)
    pipe.process_points(_params(K), pts, pts)
    before = ctx.launch_count
    assert _code(lambda: pipe.bundle_adjust_stereo(window, 2, K)) == _lib.ERR_INVALID
    assert ctx.launch_count == before
    pipe.close()
    fresh.close()
