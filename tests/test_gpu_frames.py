"""epivo_seq_process_frames: the optical-flow loop body of kitti_E.cpp:54-201 / euroc_E.cpp:169-208 from frames on the
device.  The reference for every comparison is the composed route through the calls that are pinned to OpenCV one by
one: fastDetect (capped at kp_per_frame) -> trackSequenceLK / calcOpticalFlowPyrLK on each listed pair -> the status
filter of kitti_E.cpp:86-95 on the host -> process_points.  The fused call must return the same bytes."""
import ctypes as C

import numpy as np
import pytest

from epivo_b200 import api, synth
from epivo_b200 import datasets as D
from lk_util import check_lk

pytestmark = pytest.mark.gpu


def _texture(rows, cols, seed, passes=4):
    """Smoothed noise (the texture of bench.py's front-end measurement): about 3000 FAST-40 corners per KITTI frame."""
    rng = np.random.default_rng(seed)
    tex = rng.integers(0, 256, (rows, cols)).astype(np.float32)
    for _ in range(passes):
        tex = sum(np.roll(np.roll(tex, dy, 0), dx, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1)) / 9.0
    return ((tex - tex.min()) / (tex.max() - tex.min()) * 255).astype(np.uint8)


def _drive(n, rows, cols, seed, dx=1):
    """n frames of rows x cols cut from one texture along a forward drift with a little vertical wobble."""
    tex = _texture(rows + 16, cols + dx * n + 8, seed)
    return np.stack([tex[4 + (k % 5):4 + (k % 5) + rows, dx * k:dx * k + cols] for k in range(n)])


def _parallax(n, rows, cols, seed, far=12, near=20):
    """n frames of a sideways camera translation over two fronto-parallel planes: the upper half of the image (the far
    plane) moves `far` px per frame, the lower half (the near plane) `near` px.  The near plane lies within recoverPose's
    distance threshold, so the pose has cheirality-good points and LM runs (a single shifted texture has no parallax)."""
    tex = _texture(rows + 16, cols + near * n + 8, seed)
    h = rows // 2
    out = np.empty((n, rows, cols), np.uint8)
    for k in range(n):
        out[k, :h] = tex[4:4 + h, far * k:far * k + cols]
        out[k, h:] = tex[4 + h:4 + rows, near * k:near * k + cols]
    return out


@pytest.fixture(scope="module")
def kitti_frames():
    return _parallax(40, 376, 1241, 12)


def _track_pairs(ctx, frames, fq, ft, corners):
    """calcOpticalFlowPyrLK(frames[fq[i]], frames[ft[i]], corners[fq[i]]) for every listed pair, in one trackSequenceLK
    call over the frames (fq0, ft0, fq1, ft1, ...): the pairs (ft_i, fq_i+1) in between track nothing."""
    seq = np.stack([frames[f] for pr in zip(fq, ft) for f in pr])
    pts = []
    for i in range(len(fq)):
        pts.append(corners[fq[i]])
        if i + 1 < len(fq):
            pts.append(np.zeros((0, 2), np.float32))
    nxt, st = api.trackSequenceLK(seq, pts, ctx=ctx)
    return nxt[0::2], st[0::2]


def _composed(ctx, prm, frames, kp, thr, pairs=None):
    """The route through the pinned calls: kept tracks (p0, p1), their corner indices and the process_points results."""
    n = len(frames)
    det = api.fastDetect(frames, thr, True, max_keypoints=kp, ctx=ctx)
    corners = [d[0] for d in det]
    if pairs is None:
        fq, ft = np.arange(n - 1), np.arange(1, n)
        nxt, st = api.trackSequenceLK(frames, corners[:-1], ctx=ctx)
    else:
        fq, ft = pairs
        nxt, st = _track_pairs(ctx, frames, fq, ft, corners)
    idx = [np.nonzero(s == 1)[0] for s in st]
    p0 = [corners[fq[i]][idx[i]] for i in range(len(fq))]
    p1 = [nxt[i][idx[i]] for i in range(len(fq))]
    pipe = api.SequencePipeline(n, kp, ctx=ctx, max_pairs=max(n - 1, len(fq)))
    if pairs is not None:
        pipe.set_pairs(fq, ft)
    res = pipe.process_points(prm, p0, p1).copy()
    masks = [pipe.masks(i) for i in range(len(fq))]
    pipe.close()
    return dict(p0=p0, p1=p1, idx=idx, res=res, masks=masks)


def _fused(ctx, prm, frames, kp, thr, pairs=None, maps=None):
    n = len(frames)
    npairs = n - 1 if pairs is None else len(pairs[0])
    pipe = api.SequencePipeline(n, kp, ctx=ctx, max_pairs=max(n - 1, npairs))
    if pairs is not None:
        pipe.set_pairs(*pairs)
    res, corners = pipe.process_frames(prm, frames, thr, maps=maps, corners=True)
    out = dict(res=res.copy(), corners=corners, masks=[pipe.masks(i) for i in range(npairs)],
               points=[pipe.points(i) for i in range(npairs)], matches=[pipe.matches(i) for i in range(npairs)])
    pipe.close()
    return out


def _assert_same(f, r, what=""):
    assert f["res"].tobytes() == r["res"].tobytes(), what
    for i in range(len(r["p0"])):
        assert np.array_equal(f["masks"][i][0], r["masks"][i][0]) and np.array_equal(f["masks"][i][1], r["masks"][i][1]), (what, i)
        p0, p1 = f["points"][i]
        assert np.array_equal(p0, r["p0"][i]) and np.array_equal(p1, r["p1"][i]), (what, i)
        qi, ti, d = f["matches"][i]
        assert np.array_equal(qi, r["idx"][i]) and np.array_equal(ti, r["idx"][i]) and not d.any(), (what, i)


def _found(ctx, frames, thr):
    return np.array([len(d[0]) for d in api.fastDetect(frames, thr, True, ctx=ctx)], np.int32)


@pytest.mark.parametrize("method,threshold", [(api.LMEDS, 0.01), (api.RANSAC, 1.0)])   # kitti_E.cpp:101, kitti.cpp:101
def test_kitti_consecutive_equals_composed_route(ctx, kitti_frames, method, threshold):
    prm = api.default_params(synth.KITTI_K.astype(np.float32), method=method, prob=0.99, threshold=threshold)
    kp = 6144
    r = _composed(ctx, prm, kitti_frames, kp, 40)
    f = _fused(ctx, prm, kitti_frames, kp, 40)
    _assert_same(f, r)
    assert np.array_equal(f["corners"], _found(ctx, kitti_frames, 40))
    assert f["corners"].max() < kp and f["corners"].min() > 1500
    assert (f["res"]["n_matches"] > 0.9 * f["corners"][:-1]).all()
    assert (f["res"]["n_good"] >= 48).all() and f["res"]["lm_ran"].all()


def test_euroc_remap_equals_composed_route(ctx):
    raw = _drive(12, 480, 752, 5, dx=2)
    xy, fr = D.undistort_rectify_maps(D.EUROC_CAM0_K, D.EUROC_CAM0_DIST, D.EUROC_CAM0_RECT, D.EUROC_CAM0_PROJ, (752, 480))
    prm = api.default_params(synth.EUROC_K.astype(np.float32), method=api.RANSAC, prob=0.99, threshold=0.3)   # euroc_E.cpp:202-208
    kp = 12288                                                              # FAST(10) finds ~10 k corners here
    und = api.remap(raw, xy, fr, ctx=ctx)
    r = _composed(ctx, prm, und, kp, 10)                                   # FAST(10): euroc_E.cpp:177
    f = _fused(ctx, prm, raw, kp, 10, maps=(xy, fr))
    _assert_same(f, r)
    assert np.array_equal(f["corners"], _found(ctx, und, 10))
    assert (f["res"]["n_matches"] > 100).all()


def test_pair_lists_equal_composed_route(ctx):
    # kitti_ba's window walk: (0,1), (0,2), (1,2) at stride 2, listed out of order
    frames = _drive(21, 240, 400, 3, dx=2)
    walk = [(i + a, i + b) for i in range(0, 19, 2) for a, b in ((0, 1), (0, 2), (1, 2))]
    order = np.random.default_rng(1).permutation(len(walk))
    fq = np.array([walk[o][0] for o in order], np.int32)
    ft = np.array([walk[o][1] for o in order], np.int32)
    prm = api.default_params(np.array([[400.0, 0, 200.0], [0, 400.0, 120.0], [0, 0, 1]], np.float32), method=api.LMEDS,
                             threshold=0.01)
    r = _composed(ctx, prm, frames, 2048, 40, pairs=(fq, ft))
    f = _fused(ctx, prm, frames, 2048, 40, pairs=(fq, ft))
    _assert_same(f, r, "window walk")
    assert (f["res"]["n_matches"] > 100).all()
    # a stereo-like layout: node 2f is the left and 2f + 1 the right image of time f; pairs left-right and left-left
    tex = _texture(260, 520, 9)
    stereo = np.stack([tex[8:248, x:x + 400] for f in range(8) for x in (3 * f, 3 * f + 6)])
    fq = np.array([2 * f for f in range(8)] + [2 * f for f in range(7)], np.int32)
    ft = np.array([2 * f + 1 for f in range(8)] + [2 * f + 2 for f in range(7)], np.int32)
    r = _composed(ctx, prm, stereo, 2048, 40, pairs=(fq, ft))
    f = _fused(ctx, prm, stereo, 2048, 40, pairs=(fq, ft))
    _assert_same(f, r, "stereo")


def _long(n):
    tex = _texture(120 + 40, 160 + 60, 21, passes=3)
    return np.stack([tex[(k // 7) % 30:(k // 7) % 30 + 120, k % 50:k % 50 + 160] for k in range(n)])


def test_windows_equal_composed_route(ctx):
    """330 frames: more than one 256-frame window, so tracks cross window boundaries (consecutive pairs, and a list of
    span 2); a list whose span does not fit a window is refused before anything is launched."""
    frames = _long(330)
    prm = api.default_params(np.array([[200.0, 0, 80.0], [0, 200.0, 60.0], [0, 0, 1]], np.float32), method=api.LMEDS,
                             threshold=0.01)
    kp = 1024
    r = _composed(ctx, prm, frames, kp, 40)
    f = _fused(ctx, prm, frames, kp, 40)
    _assert_same(f, r, "consecutive")
    assert np.array_equal(f["corners"], _found(ctx, frames, 40))
    n = len(frames)
    fq = np.array([i for i in range(n - 1)] + [i for i in range(n - 2)], np.int32)
    ft = np.array([i + 1 for i in range(n - 1)] + [i + 2 for i in range(n - 2)], np.int32)
    r = _composed(ctx, prm, frames, kp, 40, pairs=(fq, ft))
    f = _fused(ctx, prm, frames, kp, 40, pairs=(fq, ft))
    _assert_same(f, r, "span 2")
    pipe = api.SequencePipeline(n, kp, ctx=ctx, max_pairs=n)
    pipe.set_pairs(np.append(fq[:5], 0), np.append(ft[:5], n - 1))
    before = ctx.launch_count
    with pytest.raises(api.EpivoError) as e:
        pipe.process_frames(prm, frames, 40)
    assert e.value.code == -3 and ctx.launch_count == before
    pipe.close()


def test_more_corners_than_capacity(ctx, kitti_frames):
    frames = kitti_frames[:6]
    prm = api.default_params(synth.KITTI_K.astype(np.float32), method=api.RANSAC, prob=0.99, threshold=1.0)
    kp = 700
    r = _composed(ctx, prm, frames, kp, 40)                 # fastDetect(max_keypoints = kp): the first kp corners
    f = _fused(ctx, prm, frames, kp, 40)
    _assert_same(f, r)
    found = _found(ctx, frames, 40)
    assert np.array_equal(f["corners"], found) and (found > kp).all()
    assert (f["res"]["n_matches"] <= kp).all() and (f["res"]["n_matches"] > 0.9 * kp).all()


def test_degenerate_frames(ctx):
    """A flat frame (no corners) and a frame with three corners (fewer than the five points findEssentialMat needs)."""
    tex = _texture(140, 200, 4)
    flat = np.full((120, 160), 128, np.uint8)
    few = flat.copy()
    few[30, 40] = few[60, 100] = few[90, 70] = 250
    few2 = np.roll(few, 1, axis=1)
    frames = np.stack([flat, tex[:120, :160], tex[2:122, 3:163], few, few2, flat])
    prm = api.default_params(np.array([[200.0, 0, 80.0], [0, 200.0, 60.0], [0, 0, 1]], np.float32))
    r = _composed(ctx, prm, frames, 1024, 40)
    f = _fused(ctx, prm, frames, 1024, 40)
    _assert_same(f, r)
    assert f["corners"][0] == 0 and f["corners"][3] == 3
    assert f["res"]["n_matches"][0] == 0 and f["res"]["n_matches"][3] < 5 and f["res"]["n_matches"][1] > 50
    assert not f["res"]["lm_ran"][0] and not f["res"]["lm_ran"][3]


def _raw(ctx, pipe, prm, n, im, rows, cols, m1=None, m2=None, drows=0, dcols=0, thr=40):
    out = np.zeros(max(pipe.max_pairs, 1), dtype=api.RESULT_DTYPE)
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    return ctx.lib.epivo_seq_process_frames(pipe.h, C.byref(prm), n, p(im), rows, cols, p(m1), p(m2), drows, dcols, thr,
                                            None, p(out))


def test_bad_arguments_launch_nothing(ctx):
    frames = _long(6)
    n, rows, cols = frames.shape
    prm = api.default_params(np.array([[200.0, 0, 80.0], [0, 200.0, 60.0], [0, 0, 1]], np.float32))
    pipe = api.SequencePipeline(n, 512, ctx=ctx, max_pairs=8)
    m1 = np.zeros((rows, cols, 2), np.int16)
    m2 = np.zeros((rows, cols), np.uint16)
    n0 = np.zeros(1, np.uint8)
    before = ctx.launch_count
    bad = [
        _raw(ctx, pipe, prm, 1, frames, rows, cols),                         # fewer than two frames
        _raw(ctx, pipe, prm, n + 1, np.concatenate([frames, frames[:1]]), rows, cols),   # more than max_frames
        _raw(ctx, pipe, prm, n, frames, 21, cols),                           # not larger than the 21 x 21 window
        _raw(ctx, pipe, prm, n, frames, rows, cols, thr=-1),
        _raw(ctx, pipe, prm, n, frames, rows, cols, thr=256),
        _raw(ctx, pipe, prm, n, frames, rows, cols, m1=m1, drows=rows, dcols=cols),   # one map only
        _raw(ctx, pipe, prm, n, frames, rows, cols, m2=m2, drows=rows, dcols=cols),
        _raw(ctx, pipe, prm, n, frames, rows, cols, m1=m1, m2=m2, drows=0, dcols=cols),
        _raw(ctx, pipe, prm, n, frames, rows, cols, m1=m1[:21, :21].copy(), m2=m2[:21, :21].copy(), drows=21, dcols=21),
        _raw(ctx, pipe, prm, n, n0, 0, 0),
    ]
    for kw in (dict(method=5), dict(lm_points=0), dict(lm_points=65)):
        bad.append(_raw(ctx, pipe, api.default_params(np.eye(3), **kw), n, frames, rows, cols))
    pipe2 = api.SequencePipeline(n + 2, 512, ctx=ctx, max_pairs=8)
    pipe2.set_pairs([0, 1], [1, n + 1])
    bad.append(_raw(ctx, pipe2, prm, n, frames, rows, cols))               # the list references frame n + 1 of n frames
    assert all(rc in (-1, -3) for rc in bad), bad
    assert ctx.launch_count == before
    pp = C.c_int(0)
    assert ctx.lib.epivo_seq_get_points(pipe.h, 0, None, None, C.byref(pp)) == -1      # no process_frames run yet
    pipe.process_points(prm, [np.zeros((8, 2), np.float32)], [np.zeros((8, 2), np.float32)])
    assert ctx.lib.epivo_seq_get_points(pipe.h, 0, None, None, C.byref(pp)) == -1      # the last run was process_points
    pipe.close()
    pipe2.close()


def test_live_cv2_corners_and_tracks(ctx, kitti_frames):
    cv2 = pytest.importorskip("cv2")
    frames = kitti_frames[:3]
    prm = api.default_params(synth.KITTI_K.astype(np.float32), method=api.LMEDS, prob=0.99, threshold=0.01)
    f = _fused(ctx, prm, frames, 6144, 40)
    det = cv2.FastFeatureDetector_create(40)
    for i in range(2):
        kps = det.detect(frames[i], None)
        c = np.array([k.pt for k in kps], np.float32).reshape(-1, 2)
        assert f["corners"][i] == len(c)
        qi = f["matches"][i][0]
        p0, p1 = f["points"][i]
        assert np.array_equal(p0, c[qi])                                   # the tracked points are cv2's corners
        ref_nxt, ref_st, _ = cv2.calcOpticalFlowPyrLK(frames[i], frames[i + 1], c, None)
        st = np.zeros(len(c), np.uint8)
        st[qi] = 1
        nxt = np.zeros_like(c)
        nxt[qi] = p1
        check_lk(nxt, st, ref_nxt, ref_st.ravel(), "pair %d" % i)
    assert f["corners"][2] == len(det.detect(frames[2], None))
