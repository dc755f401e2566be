"""Host-side mirror of the reference's call shapes over the C ABI (ctypes, numpy buffers).

The reference drivers call, per frame pair (SURVEY.md section 8b):
    cv::BFMatcher(NORM_HAMMING2, true).match(desc0, desc1, matches)      kitti_ba.cpp:602,641
    cv::findEssentialMat(p0, p1, cam, method, prob, thr, mask)           kitti_E.cpp:98-104
    cv::recoverPose(E, p0, p1, cam, R, t, mask)                          kitti_E.cpp:120
    Levenberg_Marquardt(n_zeta, eps, reps, wreps, lambda0, T0s, pr, p_r, lm_res)
                                                                         jac_Rt_gen_.cpp:287
The functions here keep those names, argument meanings and error behaviour (empty result /
None where OpenCV returns an empty Mat) and run on the GPU through libepivo_b200.so.  The
C++ equivalents (what an unmodified driver links against) are in include/epivo_shims.hpp.
"""
from __future__ import annotations

import ctypes as C
import weakref

import numpy as np

from . import _lib
from ._lib import (EpivoError, LmRes, PairResult, PipelineParams, LMEDS, RANSAC, NORM_HAMMING,  # noqa: F401
                   NORM_HAMMING2, MATCH_NN, MATCH_CROSSCHECK, MATCH_RATIO)


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Context:
    """One CUDA stream + workspace on one device (`epivo_ctx`).  Not shared between threads."""

    def __init__(self, device: int = 0):
        self.lib = _lib.load()
        h = C.c_void_p()
        rc = self.lib.epivo_create(C.byref(h), int(device))
        if rc != 0 or not h.value:
            raise EpivoError(rc, f"epivo_create(device={device}) failed: no usable CUDA device "
                                 "(there is no CPU fallback)")
        self.h = h
        self.device = device
        self._children = weakref.WeakSet()       # SequencePipelines: destroyed before the context

    def close(self):
        if getattr(self, "h", None) is not None and self.h.value:
            for child in list(self._children):
                child.close()
            self.lib.epivo_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc: int, allow=()):
        if rc != 0 and rc not in allow:
            raise EpivoError(rc, self.lib.epivo_last_error(self.h).decode())
        return rc

    @property
    def stream(self) -> int:
        return int(self.lib.epivo_stream(self.h) or 0)

    @property
    def launch_count(self) -> int:
        return int(self.lib.epivo_launch_count(self.h))

    def sync(self):
        self.check(self.lib.epivo_sync(self.h))

    def last_kernel_ms(self) -> float:
        """Device time of the kernels of the last Levenberg_Marquardt[_batch] call (no copies)."""
        ms = C.c_float(0.0)
        self.check(self.lib.epivo_last_kernel_ms(self.h, C.byref(ms)))
        return float(ms.value)

    def microbench(self, which: int) -> float:
        v = C.c_double()
        self.check(self.lib.epivo_microbench(self.h, which, C.byref(v)))
        return v.value


_default_ctx = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


class BFMatcher:
    """cv::BFMatcher(normType, crossCheck) for binary descriptors (kitti_ba.cpp:602)."""

    def __init__(self, normType: int = NORM_HAMMING2, crossCheck: bool = False, ctx: Context | None = None):
        self.normType = normType
        self.crossCheck = bool(crossCheck)
        self.ctx = ctx or default_context()

    def _descs(self, q, t):
        q = np.ascontiguousarray(q, dtype=np.uint8)
        t = np.ascontiguousarray(t, dtype=np.uint8)
        if q.ndim != 2 or t.ndim != 2:
            raise ValueError("descriptors must be 2-D uint8 arrays")
        if q.shape[0] and t.shape[0] and q.shape[1] != t.shape[1]:
            raise ValueError("descriptor sizes differ")
        return q, t

    def match(self, queryDescriptors, trainDescriptors):
        """-> (queryIdx, trainIdx, distance) int32 arrays, sorted by queryIdx (DMatch fields)."""
        mode = MATCH_CROSSCHECK if self.crossCheck else MATCH_NN
        return self._run(queryDescriptors, trainDescriptors, mode, 0.0)[:3]

    def ratioMatch(self, queryDescriptors, trainDescriptors, ratio: float = 0.8):
        """knnMatch(k=2) + Lowe ratio test -> (queryIdx, trainIdx, distance, distance2)."""
        return self._run(queryDescriptors, trainDescriptors, MATCH_RATIO, ratio)

    def knnMatch2(self, queryDescriptors, trainDescriptors):
        """knnMatch(k=2) -> (trainIdx (nq,2), distance (nq,2))."""
        q, t = self._descs(queryDescriptors, trainDescriptors)
        nq, nt = q.shape[0], t.shape[0]
        idx = np.full((nq, 2), -1, dtype=np.int32)
        dist = np.full((nq, 2), -1, dtype=np.int32)
        db = q.shape[1] if nq else (t.shape[1] if nt else 32)
        self.ctx.check(self.ctx.lib.epivo_knn2_hamming(self.ctx.h, _p(q), nq, _p(t), nt, db, self.normType,
                                                       _p(idx), _p(dist)))
        return idx, dist

    def _run(self, q, t, mode, ratio):
        q, t = self._descs(q, t)
        nq, nt = q.shape[0], t.shape[0]
        qi = np.empty(max(nq, 1), dtype=np.int32)
        ti = np.empty(max(nq, 1), dtype=np.int32)
        d = np.empty(max(nq, 1), dtype=np.int32)
        d2 = np.empty(max(nq, 1), dtype=np.int32)
        n = C.c_int(0)
        db = q.shape[1] if nq else (t.shape[1] if nt else 32)
        self.ctx.check(self.ctx.lib.epivo_match_hamming(self.ctx.h, _p(q), nq, _p(t), nt, db, self.normType,
                                                        mode, float(ratio), _p(qi), _p(ti), _p(d), _p(d2),
                                                        C.byref(n)))
        k = n.value
        return qi[:k].copy(), ti[:k].copy(), d[:k].copy(), d2[:k].copy()


def _pts(p):
    p = np.ascontiguousarray(p, dtype=np.float32).reshape(-1, 2)
    return p


def _K(K):
    return np.ascontiguousarray(np.asarray(K, dtype=np.float64).reshape(3, 3))


def findEssentialMat(points1, points2, cameraMatrix, method: int = RANSAC, prob: float = 0.999,
                     threshold: float = 1.0, maxIters: int = 1000, samples=None, ctx: Context | None = None,
                     return_info: bool = False):
    """cv::findEssentialMat -> (E 3x3 float64 | None, mask (n,) uint8 in {0,1}).

    `samples` (m x 5 int32) injects a fixed hypothesis set; None replays OpenCV's own
    deterministic sample stream so the whole call reproduces cv2."""
    ctx = ctx or default_context()
    p0, p1 = _pts(points1), _pts(points2)
    if p0.shape != p1.shape:
        raise ValueError("point sets differ in size")
    n = p0.shape[0]
    K = _K(cameraMatrix)
    E = np.zeros(9, dtype=np.float64)
    mask = np.zeros(max(n, 1), dtype=np.uint8)
    ninl, iters = C.c_int(0), C.c_int(0)
    s = None
    m = 0
    if samples is not None:
        s = np.ascontiguousarray(samples, dtype=np.int32).reshape(-1, 5)
        m = s.shape[0]
    rc = ctx.check(ctx.lib.epivo_find_essential(ctx.h, _p(p0), _p(p1), n, _p(K), int(method), float(prob),
                                                float(threshold), int(maxIters), _p(s), m, _p(E), _p(mask),
                                                C.byref(ninl), C.byref(iters)), allow=(_lib.ERR_NOMODEL,))
    Eo = None if rc == _lib.ERR_NOMODEL else E.reshape(3, 3)
    if return_info:
        return Eo, mask[:n], {"n_inliers": ninl.value, "iters": iters.value}
    return Eo, mask[:n]


def fivePoint(x1, x2, ctx: Context | None = None):
    """The minimal solver alone on m samples (m,5,2) of K-normalised points -> list of (k,3,3)."""
    E, nm = fivePointRaw(x1, x2, ctx)
    return [E[i, :nm[i]] for i in range(E.shape[0])]


def fivePointRaw(x1, x2, ctx: Context | None = None):
    """As fivePoint, without the per-sample Python list: (E (m,10,3,3) with the first n_models[i] valid, n_models (m,))."""
    ctx = ctx or default_context()
    x1 = np.ascontiguousarray(x1, dtype=np.float64).reshape(-1, 5, 2)
    x2 = np.ascontiguousarray(x2, dtype=np.float64).reshape(-1, 5, 2)
    m = x1.shape[0]
    E = np.zeros((m, 10, 9), dtype=np.float64)
    nm = np.zeros(m, dtype=np.int32)
    ctx.check(ctx.lib.epivo_five_point(ctx.h, _p(x1), _p(x2), m, _p(E), _p(nm)))
    return E.reshape(m, 10, 3, 3), nm


def eightPoint(x1, x2, ctx: Context | None = None):
    """8-point hypotheses: m samples (m, 8, 2) of K-normalised points -> (E (m, 3, 3) unit Frobenius norm, ok (m,))."""
    ctx = ctx or default_context()
    x1 = np.ascontiguousarray(x1, dtype=np.float64).reshape(-1, 8, 2)
    x2 = np.ascontiguousarray(x2, dtype=np.float64).reshape(-1, 8, 2)
    m = x1.shape[0]
    E = np.zeros((m, 9), dtype=np.float64)
    ok = np.zeros(m, dtype=np.int32)
    ctx.check(ctx.lib.epivo_eight_point(ctx.h, _p(x1), _p(x2), m, _p(E), _p(ok)))
    return E.reshape(m, 3, 3), ok


def fastDetect(images, threshold: int = 10, nonmaxSuppression: bool = True, max_keypoints: int | None = None,
               ctx: Context | None = None):
    """cv2.FastFeatureDetector_create(threshold, nonmaxSuppression).detect for a batch of equally sized 8-bit
    images (kitti_E.cpp:71-74: threshold 40; kitti_ba.cpp:98: the default 10).  images: (rows, cols) or
    (n, rows, cols) uint8.  Returns a list of (pts (k, 2) float32 [x, y], response (k,) float32) per image, in
    OpenCV's keypoint order; bit-exact with OpenCV.  max_keypoints bounds the per-image output buffer (default: a
    quarter of the pixels, which no 8-bit image exceeds after suppression); a frame that exceeds it is re-run."""
    ctx = ctx or default_context()
    im = np.ascontiguousarray(images, dtype=np.uint8)
    single = im.ndim == 2
    if single:
        im = im[None]
    if im.ndim != 3:
        raise ValueError("images must be (rows, cols) or (n, rows, cols) uint8")
    n, rows, cols = im.shape
    cap = int(max_keypoints) if max_keypoints is not None else max(1024, rows * cols // (4 if nonmaxSuppression else 1))
    while True:
        kps = np.zeros((n, cap, 2), dtype=np.float32)
        resp = np.zeros((n, cap), dtype=np.float32)
        counts = np.zeros(n, dtype=np.int32)
        ctx.check(ctx.lib.epivo_fast_detect(ctx.h, _p(im), n, rows, cols, int(threshold), 1 if nonmaxSuppression else 0,
                                            cap, _p(kps), _p(resp), _p(counts)))
        if max_keypoints is not None or n == 0 or counts.max() <= cap:
            break
        cap = int(counts.max())
    out = [(kps[i, :min(counts[i], cap)].copy(), resp[i, :min(counts[i], cap)].copy()) for i in range(n)]
    return out[0] if single else out


KEYPOINT_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"),
                           ("octave", "<i4"), ("class_id", "<i4")])          # = cv::KeyPoint = epivo_keypoint


def orbDetectAndCompute(images, nfeatures: int = 10000, scaleFactor: float = 1.2, nlevels: int = 8, edgeThreshold: int = 15,
                        fastThreshold: int = 20, max_keypoints: int | None = None, ctx: Context | None = None):
    """cv2.ORB_create(nfeatures, scaleFactor, nlevels, edgeThreshold, 0, 2, cv2.ORB_FAST_SCORE, 31, fastThreshold)
    .detectAndCompute(img, None) for a batch of equally sized 8-bit images (kitti_ba.cpp:128-152 runs it with
    10000, 1.2f, 8, 15).  images: (rows, cols) or (n, rows, cols) uint8.  Returns per image (keypoints: structured
    array of KEYPOINT_DTYPE in OpenCV's order, descriptors (k, 32) uint8); identical to OpenCV's.  max_keypoints bounds
    the per-image output buffer (default: nfeatures plus room for ties; a frame that exceeds it is re-run)."""
    ctx = ctx or default_context()
    im = np.ascontiguousarray(images, dtype=np.uint8)
    single = im.ndim == 2
    if single:
        im = im[None]
    if im.ndim != 3:
        raise ValueError("images must be (rows, cols) or (n, rows, cols) uint8")
    n, rows, cols = im.shape
    cap = int(max_keypoints) if max_keypoints is not None else int(nfeatures) + int(nfeatures) // 8 + 256
    while True:
        kps = np.empty((n, cap), dtype=KEYPOINT_DTYPE)            # only the first counts[i] entries of a frame are written and read
        desc = np.empty((n, cap, 32), dtype=np.uint8)
        counts = np.zeros(n, dtype=np.int32)
        ctx.check(ctx.lib.epivo_orb_detect_and_compute(ctx.h, _p(im), n, rows, cols, int(nfeatures), float(scaleFactor),
                                                       int(nlevels), int(edgeThreshold), int(fastThreshold), cap, _p(kps),
                                                       _p(desc), _p(counts)))
        if max_keypoints is not None or n == 0 or counts.max() <= cap:
            break
        cap = int(counts.max())
    out = [(kps[i, :min(counts[i], cap)].copy(), desc[i, :min(counts[i], cap)].copy()) for i in range(n)]
    return out[0] if single else out


def orbLevelGeometry(rows: int, cols: int, nfeatures: int = 10000, scaleFactor: float = 1.2, nlevels: int = 8):
    """The pyramid orbDetectAndCompute builds: (level rows, level cols, retainBest budget per level) as int32 arrays.
    Host arithmetic only -- needs the library but no GPU and no context."""
    from . import _lib
    lib = _lib.load()
    r = np.zeros(max(int(nlevels), 1), dtype=np.int32)
    c = np.zeros_like(r)
    f = np.zeros_like(r)
    rc = lib.epivo_orb_level_geometry(int(rows), int(cols), int(nfeatures), float(scaleFactor), int(nlevels), _p(r), _p(c), _p(f))
    if rc:
        raise EpivoError(rc, "epivo_orb_level_geometry(%d x %d, scale %g, %d levels) refused" % (rows, cols, scaleFactor, nlevels))
    return r, c, f


def calcOpticalFlowPyrLK(prevImg, nextImg, prevPts, maxLevel: int = 3, maxCount: int = 30, epsilon: float = 0.01,
                         minEigThreshold: float = 1e-4, ctx: Context | None = None, returnErr: bool = False):
    """cv2.calcOpticalFlowPyrLK(prevImg, nextImg, prevPts, None) with the 21 x 21 window (kitti_E.cpp:79-84):
    (nextPts (n, 2) float32, status (n,) uint8 [, err (n,) float32 with returnErr])."""
    seq = np.stack([np.ascontiguousarray(prevImg, dtype=np.uint8), np.ascontiguousarray(nextImg, dtype=np.uint8)])
    out = trackSequenceLK(seq, [prevPts], maxLevel, maxCount, epsilon, minEigThreshold, ctx=ctx, returnErr=returnErr)
    return tuple(o[0] for o in out)


def trackSequenceLK(images, points, maxLevel: int = 3, maxCount: int = 30, epsilon: float = 0.01,
                    minEigThreshold: float = 1e-4, ctx: Context | None = None, returnErr: bool = False):
    """The LK step of the kitti_E loop for a whole sequence in one call: images (n, rows, cols) uint8, points = one
    (k_i, 2) float32 array per pair i (the detector's output on frame i); returns (list of nextPts, list of status),
    pair i tracked from frame i into frame i + 1.  The pyramid of every frame is built once."""
    ctx = ctx or default_context()
    im = np.ascontiguousarray(images, dtype=np.uint8)
    if im.ndim != 3 or im.shape[0] < 2:
        raise ValueError("images must be (n >= 2, rows, cols) uint8")
    n, rows, cols = im.shape
    if len(points) != n - 1:
        raise ValueError("one point set per consecutive pair")
    pl = [np.ascontiguousarray(p, dtype=np.float32).reshape(-1, 2) for p in points]
    cap = max(1, max(len(p) for p in pl))
    pts = np.zeros((n - 1, cap, 2), dtype=np.float32)
    counts = np.zeros(n - 1, dtype=np.int32)
    for i, p in enumerate(pl):
        pts[i, :len(p)] = p
        counts[i] = len(p)
    nxt = np.zeros_like(pts)
    st = np.zeros((n - 1, cap), dtype=np.uint8)
    err = np.zeros((n - 1, cap), dtype=np.float32)          # always passed, as cv2 and the reference do (see the header)
    ctx.check(ctx.lib.epivo_lk_track(ctx.h, _p(im), n, rows, cols, _p(pts), _p(counts), cap, int(maxLevel), int(maxCount),
                                     float(epsilon), float(minEigThreshold), _p(nxt), _p(st), _p(err)))
    out = ([nxt[i, :counts[i]].copy() for i in range(n - 1)], [st[i, :counts[i]].copy() for i in range(n - 1)])
    if returnErr:
        out += ([err[i, :counts[i]].copy() for i in range(n - 1)],)
    return out


def remap(images, map1, map2, borderValue: int = 0, ctx: Context | None = None):
    """cv2.remap(src, map1, map2, cv2.INTER_LINEAR) (BORDER_CONSTANT) with fixed-point maps -- map1 (h, w, 2) int16,
    map2 (h, w) uint16, as cv2.initUndistortRectifyMap(..., m1type=cv2.CV_16SC2) / convertMaps make them
    (euroc_E.cpp:105-113, 169-174) -- for one (rows, cols) image or a batch (n, rows, cols).  Bit-exact with OpenCV."""
    ctx = ctx or default_context()
    im = np.ascontiguousarray(images, dtype=np.uint8)
    single = im.ndim == 2
    if single:
        im = im[None]
    m1 = np.ascontiguousarray(map1, dtype=np.int16)
    m2 = np.ascontiguousarray(map2, dtype=np.uint16)
    if im.ndim != 3 or m1.ndim != 3 or m1.shape[2] != 2 or m2.shape != m1.shape[:2]:
        raise ValueError("images (n, rows, cols) uint8, map1 (h, w, 2) int16, map2 (h, w) uint16")
    n, rows, cols = im.shape
    out = np.zeros((n,) + m2.shape, dtype=np.uint8)
    ctx.check(ctx.lib.epivo_remap(ctx.h, _p(im), n, rows, cols, _p(m1), _p(m2), m2.shape[0], m2.shape[1], int(borderValue), _p(out)))
    return out[0] if single else out


def scoreSampson(Es, points1, points2, cameraMatrix, threshold: float, ctx: Context | None = None,
                 medians: bool = True):
    """K3 alone: (counts (m,), medians (m,) f32, best index, mask of best (n,) {0,1}).
    medians=False skips the LMedS medians (they cost a select over all points per model)."""
    ctx = ctx or default_context()
    Es = np.ascontiguousarray(Es, dtype=np.float64).reshape(-1, 9)
    p0, p1 = _pts(points1), _pts(points2)
    n, m = p0.shape[0], Es.shape[0]
    K = _K(cameraMatrix)
    counts = np.zeros(max(m, 1), dtype=np.int32)
    med = np.zeros(max(m, 1), dtype=np.float32)
    mask = np.zeros(max(n, 1), dtype=np.uint8)
    best = C.c_int(-1)
    ctx.check(ctx.lib.epivo_score_sampson(ctx.h, _p(Es), m, _p(p0), _p(p1), n, _p(K), float(threshold),
                                          _p(counts), _p(med) if medians else None, C.byref(best), _p(mask)))
    return counts[:m], med[:m], best.value, mask[:n]


def recoverPose(E, points1, points2, cameraMatrix, distanceThresh: float = 50.0, mask=None,
                ctx: Context | None = None):
    """cv::recoverPose -> (n_good, R 3x3, t (3,), mask (n,) uint8 in {0,255})."""
    ctx = ctx or default_context()
    p0, p1 = _pts(points1), _pts(points2)
    n = p0.shape[0]
    K = _K(cameraMatrix)
    Ein = np.ascontiguousarray(np.asarray(E, dtype=np.float64).reshape(9))
    R = np.zeros(9)
    t = np.zeros(3)
    out = np.zeros(max(n, 1), dtype=np.uint8)
    im = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8).reshape(-1)
    ng = C.c_int(0)
    ctx.check(ctx.lib.epivo_recover_pose(ctx.h, _p(Ein), _p(p0), _p(p1), n, _p(K), float(distanceThresh), _p(im),
                                         _p(R), _p(t), _p(out), C.byref(ng)))
    return ng.value, R.reshape(3, 3), t, out[:n]


def Levenberg_Marquardt(n_zeta: int, epsilon: float, reps, wreps, lambda0: float, T0s, pr, p_r,
                        huber_delta: float = 1e-5, max_iters: int = 30, ctx: Context | None = None):
    """jac_Rt_gen_.cpp:287 -- returns (T0s_out (n_zeta,4,4), LM_res dict); T0s is not modified.

    `wreps=None` is the 7-argument form called at kitti_E.cpp:196 (unit weights)."""
    ctx = ctx or default_context()
    reps = np.ascontiguousarray(reps, dtype=np.int32).reshape(-1, 2)
    n_rep = reps.shape[0]
    w = np.ones(n_rep) if wreps is None else np.ascontiguousarray(wreps, dtype=np.float64).reshape(-1)
    if w.shape[0] != n_rep:
        raise ValueError("reps.size() != wreps.size()")            # jac_Rt_gen_.cpp:297
    T = np.array(T0s, dtype=np.float64).reshape(n_zeta, 16).copy()
    pr = np.ascontiguousarray(pr, dtype=np.float64)
    p_r = np.ascontiguousarray(p_r, dtype=np.float64)
    N = pr.shape[1]
    res = LmRes()
    it = C.c_int(0)
    ctx.check(ctx.lib.epivo_lm_rt(ctx.h, int(n_zeta), float(epsilon), _p(reps), _p(w), n_rep, float(lambda0),
                                  int(max_iters), float(huber_delta), _p(T), _p(pr), _p(p_r), int(N),
                                  C.byref(res), C.byref(it)))
    return T.reshape(n_zeta, 4, 4), {"H_norm": res.H_norm, "r_norm": res.r_norm, "lambda": res.lambda_,
                                     "iters": it.value}


def Levenberg_Marquardt_batch(n_zeta, epsilon, reps, wreps, lambda0, T0s, pr, p_r, huber_delta=1e-5,
                              max_iters=30, ctx: Context | None = None):
    """B independent windows of identical shape in one launch (kitti_ba windows per GPU)."""
    ctx = ctx or default_context()
    reps = np.ascontiguousarray(reps, dtype=np.int32).reshape(-1, 2)
    n_rep = reps.shape[0]
    T = np.array(T0s, dtype=np.float64).copy()
    B = T.shape[0]
    T = T.reshape(B, n_zeta, 16)
    w = np.ascontiguousarray(np.broadcast_to(np.asarray(wreps, dtype=np.float64), (B, n_rep)))
    pr = np.ascontiguousarray(pr, dtype=np.float64)
    p_r = np.ascontiguousarray(p_r, dtype=np.float64)
    N = pr.shape[2]
    res = np.zeros((B, 3), dtype=np.float64)
    its = np.zeros(B, dtype=np.int32)
    ctx.check(ctx.lib.epivo_lm_rt_batch(ctx.h, B, int(n_zeta), float(epsilon), _p(reps), _p(w), n_rep,
                                        float(lambda0), int(max_iters), float(huber_delta), _p(T), _p(pr),
                                        _p(p_r), int(N), _p(res), _p(its)))
    return T.reshape(B, n_zeta, 4, 4), res, its


def chain_poses(T_pairs, scales=None, ctx: Context | None = None) -> np.ndarray:
    """kitti_E.cpp:218-228 on the device for poses that are already on the host (the all-gathered poses of a sharded
    sequence): (n, 4, 4) refined pair transforms -> (n + 1, 4, 4) chained camera poses."""
    ctx = ctx or default_context()
    T = np.ascontiguousarray(T_pairs, dtype=np.float64).reshape(-1, 16)
    n = T.shape[0]
    sc = None if scales is None else np.ascontiguousarray(scales, dtype=np.float64)
    assert sc is None or sc.shape == (n,)
    poses = np.zeros((n + 1, 16), dtype=np.float64)
    ctx.check(ctx.lib.epivo_chain_poses(ctx.h, _p(T), _p(sc) if sc is not None else None, n, _p(poses)))
    return poses.reshape(n + 1, 4, 4)


def default_params(K=None, **kw) -> PipelineParams:
    p = PipelineParams()
    _lib.load().epivo_pipeline_params_default(C.byref(p))
    if K is not None:
        Kf = np.asarray(K, dtype=np.float64).reshape(9)
        for i in range(9):
            p.K[i] = float(Kf[i])
    for k, v in kw.items():
        if k == "fallback_t":
            for i in range(3):
                p.fallback_t[i] = float(v[i])
        else:
            setattr(p, k, v)
    return p


class SequencePipeline:
    """Device-resident frame sequence + the fused per-pair pipeline (`epivo_seq`)."""

    def __init__(self, max_frames: int, kp_per_frame: int, ctx: Context | None = None, max_pairs: int | None = None):
        self.ctx = ctx or default_context()
        self.max_frames, self.kp = int(max_frames), int(kp_per_frame)
        self.max_pairs = self.max_frames - 1 if max_pairs is None else int(max_pairs)
        self.n_pairs = self.max_frames - 1
        self._pair_list = False
        self._frames = self.max_frames          # frames given to the last process / process_frames call
        h = C.c_void_p()
        self.ctx.check(self.ctx.lib.epivo_seq_create_pairs(self.ctx.h, C.byref(h), self.max_frames, self.kp,
                                                           self.max_pairs))
        self.h = h
        self.ctx._children.add(self)

    def close(self):
        if getattr(self, "h", None) is not None and self.h.value:
            if self.ctx.h.value:                 # a closed context has already destroyed us
                self.ctx.lib.epivo_seq_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def upload(self, kps: np.ndarray, descs: np.ndarray, first_frame: int = 0):
        """kps (F, kp, 2) f32 and descs (F, kp, 32) u8 host arrays (ideally pinned) -> device (async)."""
        assert kps.dtype == np.float32 and descs.dtype == np.uint8
        assert kps.flags.c_contiguous and descs.flags.c_contiguous
        F = kps.shape[0]
        assert kps.shape == (F, self.kp, 2) and descs.shape == (F, self.kp, 32)
        self.ctx.check(self.ctx.lib.epivo_seq_upload(self.h, int(first_frame), F, _p(kps), _p(descs)))

    def set_counts(self, counts, first_frame: int = 0):
        """Keypoints actually present per frame slot (<= kp_per_frame); the remainder of a slot is ignored."""
        c = np.ascontiguousarray(counts, dtype=np.int32)
        self.ctx.check(self.ctx.lib.epivo_seq_set_counts(self.h, int(first_frame), int(c.shape[0]), _p(c)))

    def extract_orb(self, images, first_frame: int = 0, nfeatures: int = 10000, scaleFactor: float = 1.2, nlevels: int = 8,
                    edgeThreshold: int = 15, fastThreshold: int = 20):
        """kitti_ba.cpp:114-156 into the sequence: ORB on images (n, rows, cols) uint8; positions, descriptors and counts of
        frame slots first_frame.. are filled on the device (no download / re-upload).  Returns the keypoints found per frame
        (a frame with more than kp_per_frame keeps the first kp_per_frame)."""
        im = np.ascontiguousarray(images, dtype=np.uint8)
        if im.ndim == 2:
            im = im[None]
        n, rows, cols = im.shape
        counts = np.zeros(n, dtype=np.int32)
        self.ctx.check(self.ctx.lib.epivo_seq_extract_orb(self.h, int(first_frame), n, _p(im), rows, cols, int(nfeatures),
                                                          float(scaleFactor), int(nlevels), int(edgeThreshold),
                                                          int(fastThreshold), _p(counts)))
        return counts

    def set_pairs(self, fq=None, ft=None):
        """Explicit pair list: pair p matches frame fq[p] (query) against ft[p] (train), as the window walk of
        kitti_ba.cpp:603-607 does; None restores the consecutive pairs (p, p + 1)."""
        if fq is None or ft is None or len(fq) == 0:
            self.ctx.check(self.ctx.lib.epivo_seq_set_pairs(self.h, 0, None, None))
            self.n_pairs = self.max_frames - 1
            self._pair_list = False
            return
        a = np.ascontiguousarray(fq, dtype=np.int32)
        b = np.ascontiguousarray(ft, dtype=np.int32)
        assert a.shape == b.shape and a.ndim == 1
        self.ctx.check(self.ctx.lib.epivo_seq_set_pairs(self.h, int(a.shape[0]), _p(a), _p(b)))
        self.n_pairs = int(a.shape[0])
        self._pair_list = True

    def run(self, params: PipelineParams, first_pair: int, n_pairs: int):
        self.ctx.check(self.ctx.lib.epivo_seq_run(self.h, C.byref(params), int(first_pair), int(n_pairs)))

    def process(self, params: PipelineParams, kps: np.ndarray, descs: np.ndarray, out=None):
        """Host buffers in, per-pair results out (the reference-facing call): the upload is pipelined
        under the matcher; returns after the results are on the host."""
        assert kps.dtype == np.float32 and descs.dtype == np.uint8
        assert kps.flags.c_contiguous and descs.flags.c_contiguous
        F = kps.shape[0]
        assert kps.shape == (F, self.kp, 2) and descs.shape == (F, self.kp, 32)
        n_out = self.n_pairs if self._pair_list else F - 1
        if out is None:
            out = np.zeros(n_out, dtype=RESULT_DTYPE)
        assert out.dtype == RESULT_DTYPE and out.shape[0] >= n_out
        self.ctx.check(self.ctx.lib.epivo_seq_process(self.h, C.byref(params), F, _p(kps), _p(descs), _p(out)))
        self._frames = F
        return out

    def process_points(self, params: PipelineParams, points0, points1, out=None):
        """The geometry for correspondences the caller already has (the LK tracks of kitti_E.cpp:86-95) instead of
        descriptor matches: points0[i], points1[i] are the (k_i, 2) float32 pixel positions of pair i in its two frames.
        findEssentialMat -> recoverPose -> fallbacks -> LM for every pair; returns the per-pair results."""
        n = len(points0)
        assert len(points1) == n and n <= self.n_pairs
        pl0 = [np.ascontiguousarray(p, dtype=np.float32).reshape(-1, 2) for p in points0]
        pl1 = [np.ascontiguousarray(p, dtype=np.float32).reshape(-1, 2) for p in points1]
        cap = max(1, max((len(p) for p in pl0), default=1))
        p0 = np.zeros((n, cap, 2), dtype=np.float32)
        p1 = np.zeros((n, cap, 2), dtype=np.float32)
        counts = np.zeros(n, dtype=np.int32)
        for i in range(n):
            assert len(pl0[i]) == len(pl1[i])
            counts[i] = len(pl0[i])
            p0[i, :counts[i]] = pl0[i]
            p1[i, :counts[i]] = pl1[i]
        if out is None:
            out = np.zeros(n, dtype=RESULT_DTYPE)
        assert out.dtype == RESULT_DTYPE and out.shape[0] >= n
        self.ctx.check(self.ctx.lib.epivo_seq_process_points(self.h, C.byref(params), n, _p(p0), _p(p1), _p(counts), cap, _p(out)))
        return out

    def process_frames(self, params: PipelineParams, images, fastThreshold: int = 40, maps=None, corners: bool = False):
        """The optical-flow loop body of kitti_E.cpp:54-201 / euroc_E.cpp:169-208 from frames, without leaving the device:
        images (n, rows, cols) uint8 -> [remap with maps = (map_xy (h, w, 2) int16, map_frac (h, w) uint16)] -> FAST
        (fastThreshold, non-maximum suppression) -> 21 x 21 pyramidal LK into the pair's second frame -> the tracks with
        status 1 -> findEssentialMat -> recoverPose -> fallbacks -> LM, for the consecutive pairs or the pair list.
        Returns the per-pair results, and with corners=True also the corners FAST found per frame."""
        im = np.ascontiguousarray(images, dtype=np.uint8)
        if im.ndim != 3:
            raise ValueError("images must be (n, rows, cols) uint8")
        n, rows, cols = im.shape
        m1 = m2 = None
        drows = dcols = 0
        if maps is not None:
            m1 = np.ascontiguousarray(maps[0], dtype=np.int16)
            m2 = np.ascontiguousarray(maps[1], dtype=np.uint16)
            if m1.ndim != 3 or m1.shape[2] != 2 or m2.shape != m1.shape[:2]:
                raise ValueError("maps: (map_xy (h, w, 2) int16, map_frac (h, w) uint16)")
            drows, dcols = m2.shape
        n_out = self.n_pairs if self._pair_list else n - 1
        out = np.zeros(max(n_out, 1), dtype=RESULT_DTYPE)
        cnt = np.zeros(max(n, 1), dtype=np.int32)
        self.ctx.check(self.ctx.lib.epivo_seq_process_frames(self.h, C.byref(params), n, _p(im), rows, cols, _p(m1), _p(m2),
                                                              drows, dcols, int(fastThreshold), _p(cnt), _p(out)))
        self._frames = n
        return (out[:n_out], cnt[:n]) if corners else out[:n_out]

    def points(self, pair: int):
        """After process_frames: the kept tracks of one pair in pixels -> (p0 (k, 2), p1 (k, 2)) float32."""
        p0 = np.zeros((self.kp, 2), dtype=np.float32)
        p1 = np.zeros((self.kp, 2), dtype=np.float32)
        n = C.c_int(0)
        self.ctx.check(self.ctx.lib.epivo_seq_get_points(self.h, int(pair), _p(p0), _p(p1), C.byref(n)))
        return p0[:n.value], p1[:n.value]

    def bundle_adjust(self, window, stride: int, K, num_frames: int | None = None, huber_delta: float = 1e-5,
                      chains: bool = False):
        """kitti_ba.cpp:757-905 (mono) over the pairs of the last run (`process`, `run` or `process_frames` over a pair list
        that holds every window pair, e.g. `ba.window_pairs`), without the per-pair downloads: the same result as
        `ba.match_kp` followed by `ba.bundle_adjustment(..., stereo=False)`.  window: the (first, second) offsets; K: the
        intrinsics (inverted as `ba.assemble` does); num_frames: default the frames of the last process / process_frames.
        Returns (opt_T (num_frames, 4, 4), lm (B, 3) [H_norm, r_norm, lambda], reverted (B,) bool, starts), and with
        chains=True also the LM's per-window chains (B, n_zeta, 4, 4) and iteration counts (B,)."""
        F = self._frames if num_frames is None else int(num_frames)
        return self._bundle_adjust(False, window, stride, K, F, None, huber_delta, chains)

    def bundle_adjust_stereo(self, window, stride: int, K, pair_weights=None, num_frames: int | None = None,
                             huber_delta: float = 1e-5, chains: bool = False):
        """kitti_ba.cpp:908-1068 (bundle_adjustment_stereo) over the pairs of the last run: the same result as `ba.match_kp`
        with each reprojection's `w` set from pair_weights, followed by `ba.bundle_adjustment(..., stereo=True)`.  Frame f is
        node 2f (left) and 2f + 1 (right), and the frame slots of the sequence are the nodes.  The pair list the call needs
        is `ba.window_pairs(ba.expand_stereo_window(window), 2 * stride, 2 * num_frames)`.  window: the driver's frame
        offsets, expanded as `ba.expand_stereo_window`; stride: in frames; pair_weights: one weight per pair of the current
        list (the driver's reproj.w: 0 on the left -> right pairs (2f, 2f+1) freezes the rig extrinsics), None = 1.0;
        num_frames: default half the frames of the last process / process_frames.  Returns (opt_T (2 * num_frames, 4, 4),
        lm (B, 3), reverted (B,) bool, starts in frames), and with chains=True also the chains and iteration counts."""
        F = self._frames // 2 if num_frames is None else int(num_frames)
        pw = None
        if pair_weights is not None:
            pw = np.ascontiguousarray(pair_weights, dtype=np.float64).reshape(-1)
            if pw.shape[0] != self.n_pairs:
                raise ValueError(f"pair_weights has {pw.shape[0]} entries for {self.n_pairs} pairs")
        return self._bundle_adjust(True, window, stride, K, F, pw, huber_delta, chains)

    def _bundle_adjust(self, stereo, window, stride, K, F, pw, huber_delta, chains):
        from .ba import expand_stereo_window
        win = [(int(a), int(b)) for a, b in window]
        if not win:
            raise ValueError("empty window")
        first = np.array([a for a, _ in win], dtype=np.int32)
        second = np.array([b for _, b in win], dtype=np.int32)
        Kinv = np.ascontiguousarray(np.linalg.inv(np.asarray(K, dtype=np.float64)))
        nodes = expand_stereo_window(win) if stereo else win
        nz = max(max(a, b) for a, b in nodes) - min(min(a, b) for a, b in nodes)
        n_opt = 2 * F if stereo else F
        cap = max(1, (F + int(stride) - 1) // max(int(stride), 1))
        opt = np.zeros((max(n_opt, 1), 16), dtype=np.float64)
        win_T = np.zeros((cap, max(nz, 1), 16), dtype=np.float64)
        lm = np.zeros((cap, 3), dtype=np.float64)
        its = np.zeros(cap, dtype=np.int32)
        rev = np.zeros(cap, dtype=np.uint8)
        nw = C.c_int32(0)
        tail = (_p(Kinv), float(huber_delta), _p(opt), _p(win_T), _p(lm), _p(its), _p(rev), C.byref(nw))
        if stereo:
            self.ctx.check(self.ctx.lib.epivo_seq_bundle_adjust_stereo(self.h, len(win), _p(first), _p(second), int(stride),
                                                                       F, _p(pw), *tail))
        else:
            self.ctx.check(self.ctx.lib.epivo_seq_bundle_adjust(self.h, len(win), _p(first), _p(second), int(stride), F,
                                                                *tail))
        B = nw.value
        starts = list(range(0, B * int(stride), int(stride)))
        out = (opt[:n_opt].reshape(n_opt, 4, 4), lm[:B], rev[:B].astype(bool), starts)
        if chains:
            out += (win_T[:B].reshape(B, nz, 4, 4), its[:B])
        return out

    def download(self, first_pair: int, n_pairs: int, out=None):
        if out is None:
            out = np.zeros(n_pairs, dtype=RESULT_DTYPE)
        assert out.dtype == RESULT_DTYPE and out.shape[0] >= n_pairs
        self.ctx.check(self.ctx.lib.epivo_seq_download(self.h, _p(out), int(first_pair), int(n_pairs)))
        return out

    def set_overlap(self, on):
        """Scheduling of the geometry relative to the matcher (epivo_seq_set_overlap): False / 0 = default (after the
        matcher), True / 1 = two-stream pipelining across pair groups for resident data, 2 = the geometry between the
        matcher pieces of the host-buffer path.  Results do not depend on it; both options measured slower."""
        self.ctx.check(self.ctx.lib.epivo_seq_set_overlap(self.h, int(on)))

    def stage_ms(self):
        ms = np.zeros(16, dtype=np.float32)
        self.ctx.check(self.ctx.lib.epivo_seq_stage_ms(self.h, _p(ms), 16))
        return ms

    def cloud(self, scales=None, first_pair: int = 0, n_pairs: int | None = None, with_points: bool = True):
        """Pose chain + depth / point cloud of the last run (kitti_E.cpp:203-254).

        Returns (poses (n+1, 4, 4) -- the reference's all_T plus the final pose, points (m, 3),
        limits (n,) -- cloud points before each pair).  scales: GT step lengths (kitti_E.cpp:220)."""
        n = (self.max_frames - 1 - first_pair) if n_pairs is None else int(n_pairs)
        poses = np.zeros((n + 1, 4, 4), dtype=np.float64)
        limits = np.zeros(max(n, 1), dtype=np.int64)
        total = C.c_int64(0)
        sc = None
        if scales is not None:
            sc = np.ascontiguousarray(scales, dtype=np.float64)
            assert sc.shape == (n,)
        lib = self.ctx.lib
        self.ctx.check(lib.epivo_seq_cloud(self.h, _p(sc) if sc is not None else None, int(first_pair), n,
                                           _p(poses), None, 0, _p(limits), C.byref(total)))
        points = np.zeros((total.value, 3), dtype=np.float64)
        if with_points and total.value > 0:
            self.ctx.check(lib.epivo_seq_cloud(self.h, _p(sc) if sc is not None else None, int(first_pair), n,
                                               _p(poses), _p(points), total.value, _p(limits), C.byref(total)))
        return poses, points, limits[:n]

    def matches(self, pair: int):
        qi = np.zeros(self.kp, dtype=np.int32)
        ti = np.zeros(self.kp, dtype=np.int32)
        d = np.zeros(self.kp, dtype=np.int32)
        n = C.c_int(0)
        self.ctx.check(self.ctx.lib.epivo_seq_get_matches(self.h, int(pair), _p(qi), _p(ti), _p(d), C.byref(n)))
        return qi[:n.value], ti[:n.value], d[:n.value]

    def masks(self, pair: int):
        em = np.zeros(self.kp, dtype=np.uint8)
        pm = np.zeros(self.kp, dtype=np.uint8)
        ne, np_ = C.c_int(0), C.c_int(0)
        self.ctx.check(self.ctx.lib.epivo_seq_get_masks(self.h, int(pair), _p(em), C.byref(ne), _p(pm),
                                                        C.byref(np_)))
        return em[:ne.value], pm[:np_.value]


RESULT_DTYPE = np.dtype([("E", "f8", (3, 3)), ("R", "f8", (3, 3)), ("t", "f8", (3,)), ("T0", "f8", (4, 4)),
                         ("T", "f8", (4, 4)), ("H_norm", "f8"), ("r_norm", "f8"), ("lambda", "f8"),
                         ("n_matches", "i4"), ("n_inliers", "i4"), ("n_good", "i4"), ("ransac_iters", "i4"),
                         ("n_models", "i4"), ("lm_iters", "i4"), ("lm_ran", "i4"), ("lm_reverted", "i4")])
assert RESULT_DTYPE.itemsize == C.sizeof(PairResult), (RESULT_DTYPE.itemsize, C.sizeof(PairResult))
