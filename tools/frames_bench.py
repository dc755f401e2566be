"""The optical-flow loop body from frames, two ways, alternating in one process (one JSON line):
  composed  fastDetect -> trackSequenceLK -> status filter on the host -> process_points (bench.py's front_end_measure)
  fused     SequencePipeline.process_frames (frames in, results out; nothing goes back to the host between stages)
KITTI: bench.py's 128 synthetic 1241 x 376 frames, FAST(40), findEssentialMat(LMEDS, .99, .01).  EuRoC: 128 synthetic
752 x 480 frames undistorted with the cam0 maps, FAST(10), RANSAC(.99, .3).  Rates are pairs per second of wall clock over
whole calls (host buffers in, results on the host); the results of the two routes are compared byte for byte.
    python tools/frames_bench.py [frames] [reps]"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from epivo_b200 import api, synth  # noqa: E402
from epivo_b200 import datasets as D  # noqa: E402


def texture(rows, cols, seed):
    rng = np.random.default_rng(seed)
    tex = rng.integers(0, 256, (rows, cols)).astype(np.float32)
    for _ in range(4):                # four 3 x 3 box filters, as bench.py's front_end_measure
        tex = sum(np.roll(np.roll(tex, dy, 0), dx, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1)) / 9.0
    return ((tex - tex.min()) / (tex.max() - tex.min()) * 255).astype(np.uint8)


def composed(ctx, pipe, prm, frames, kp, thr, maps):
    if maps is not None:
        frames = api.remap(frames, maps[0], maps[1], ctx=ctx)
    det = api.fastDetect(frames, thr, True, max_keypoints=kp, ctx=ctx)
    n = len(frames)
    nxt, st = api.trackSequenceLK(frames, [d[0] for d in det[:-1]], ctx=ctx)
    p0 = [det[i][0][st[i] == 1] for i in range(n - 1)]                 # kitti_E.cpp:86-95
    p1 = [nxt[i][st[i] == 1] for i in range(n - 1)]
    return pipe.process_points(prm, p0, p1)


def measure(ctx, name, frames, prm, kp, thr, reps, maps=None):
    n = len(frames)
    pa = api.SequencePipeline(n, kp, ctx=ctx)
    pb = api.SequencePipeline(n, kp, ctx=ctx)
    ta, tb, same = [], [], True
    for _ in range(reps + 1):                          # the first round is the warm-up
        t0 = time.perf_counter()
        ra = composed(ctx, pa, prm, frames, kp, thr, maps)
        t1 = time.perf_counter()
        rb, corners = pb.process_frames(prm, frames, thr, maps=maps, corners=True)
        t2 = time.perf_counter()
        ta.append(t1 - t0)
        tb.append(t2 - t1)
        same &= ra.tobytes() == rb.tobytes()
    ta, tb = np.array(ta[1:]), np.array(tb[1:])
    pa.close()
    pb.close()
    return {"workload": name, "frames": n, "size": [int(frames.shape[2]), int(frames.shape[1])], "fast_threshold": thr,
            "kp_per_frame": kp, "mean_corners": float(corners.mean()), "max_corners": int(corners.max()),
            "mean_tracks_kept": float(rb["n_matches"].mean()),
            "composed_pairs_per_s": (n - 1) / float(np.median(ta)), "fused_pairs_per_s": (n - 1) / float(np.median(tb)),
            "composed_ms_median": float(np.median(ta)) * 1e3, "fused_ms_median": float(np.median(tb)) * 1e3,
            "composed_ms_min": float(ta.min()) * 1e3, "fused_ms_min": float(tb.min()) * 1e3,
            "speedup_median": float(np.median(ta) / np.median(tb)), "results_identical": bool(same)}


def device_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                  # reported, not guessed
        q = "nvidia-smi unavailable: %s" % e
    return q


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 128
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 7
    ctx = api.Context(0)
    tex = texture(376 + 64, 1241 + 64, 12)                 # bench.py's front_end_measure frames
    kitti = np.stack([tex[32 + (k % 5):32 + (k % 5) + 376, 32 + 2 * (k % 7):32 + 2 * (k % 7) + 1241] for k in range(n)])
    prm_k = api.default_params(synth.KITTI_K.astype(np.float32), method=api.LMEDS, prob=0.99, threshold=0.01)
    tex = texture(480 + 16, 752 + 2 * n + 8, 5)
    euroc = np.stack([tex[4 + (k % 5):4 + (k % 5) + 480, 2 * k:2 * k + 752] for k in range(n)])
    maps = D.undistort_rectify_maps(D.EUROC_CAM0_K, D.EUROC_CAM0_DIST, D.EUROC_CAM0_RECT, D.EUROC_CAM0_PROJ, (752, 480))
    prm_e = api.default_params(synth.EUROC_K.astype(np.float32), method=api.RANSAC, prob=0.99, threshold=0.3)
    out = {"device": device_info(),
           "method": "wall clock of whole calls (host frames in, results on the host), median of %d alternating rounds "
                     "after one warm-up round" % reps,
           "kitti_E": measure(ctx, "kitti_E.cpp:54-201, FAST(40), LMEDS(.99, .01)", kitti, prm_k, 4096, 40, reps),
           "euroc_E": measure(ctx, "euroc_E.cpp:169-208, remap + FAST(10), RANSAC(.99, .3)", euroc, prm_e, 12288, 10, reps,
                              maps=maps)}
    ctx.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
