"""The windowed bundle adjustment of kitti_ba.cpp over a drive, two ways, alternating in one process (one JSON line):
  composed  ba.match_kp (set_pairs -> process -> per-pair downloads and a numpy selection) -> ba.bundle_adjustment
            (ba.assemble on the host, one epivo_lm_rt_batch, ba.finish)
  resident  SequencePipeline: set_pairs -> process -> bundle_adjust / bundle_adjust_stereo (assembly and LM on the device,
            the tail on the host)
Both routes create their own pipeline, as ba.match_kp does.  Workload: window {(0,1),(0,2),(1,2)}, stride 2,
findEssentialMat(LMEDS, .99, .1), on
  mono      synth.make_sequence(1009 frames, 2000 keypoints): 1512 pairs, 504 windows;
  --stereo  synth.make_sequence(2 * 1009 nodes, 2000 keypoints), node 2f the left and 2f + 1 the right image of frame f:
            the window expands to 9 node reps over 4 nodes, 4032 node pairs, 504 windows, and every left -> right pair
            (2f, 2f+1) has weight 0 as the driver sets it (kitti_ba.cpp:1000-1008).
Times are wall clock of whole calls (each ends in a stream synchronise); medians over the rounds after one warm-up round.
The outputs of the two routes are compared with test_gpu_ba's tolerances (rotation 1e-4 rad, translation direction 1e-3
rad, r_norm rtol 1e-4, the same reverted windows).
    python tools/ba_seq_bench.py [--stereo] [frames] [reps]"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from epivo_b200 import api, ba, synth  # noqa: E402

WINDOW = [(0, 1), (0, 2), (1, 2)]
STRIDE = 2


def device_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                  # reported, not guessed
        q = "nvidia-smi unavailable: %s" % e
    return q


def rig_weight(a, b):
    """The stereo driver's reproj.w: 0 on the left -> right pairs (2f, 2f+1), which freezes the rig extrinsics."""
    return 0.0 if a % 2 == 0 and b == a + 1 else 1.0


def composed(ctx, seq, F, stereo):
    t0 = time.perf_counter()
    if stereo:
        reprojs = ba.match_kp(seq.kps, seq.descs, ba.expand_stereo_window(WINDOW), 2 * STRIDE, seq.K, ctx=ctx)
        for (a, b), r in reprojs.items():
            r.w = rig_weight(a, b)
    else:
        reprojs = ba.match_kp(seq.kps, seq.descs, WINDOW, STRIDE, seq.K, ctx=ctx)
    t1 = time.perf_counter()
    out = ba.bundle_adjustment(reprojs, WINDOW, STRIDE, F, seq.K, stereo, 1e-5, ctx=ctx)
    t2 = time.perf_counter()
    return out, {"total": t2 - t0, "match_kp": t1 - t0, "bundle_adjustment": t2 - t1}


def resident(ctx, seq, pairs, prm, pair_w):
    t0 = time.perf_counter()
    n = seq.kps.shape[0]
    pipe = api.SequencePipeline(n, seq.kps.shape[1], ctx=ctx, max_pairs=max(len(pairs), n - 1))
    pipe.set_pairs([p[0] for p in pairs], [p[1] for p in pairs])
    pipe.process(prm, seq.kps, seq.descs)
    t1 = time.perf_counter()
    if pair_w is None:
        out = pipe.bundle_adjust(WINDOW, STRIDE, seq.K, huber_delta=1e-5)
    else:
        out = pipe.bundle_adjust_stereo(WINDOW, STRIDE, seq.K, pair_weights=pair_w, huber_delta=1e-5)
    t2 = time.perf_counter()
    pipe.close()
    return out, {"total": t2 - t0, "process": t1 - t0, "bundle_adjust": t2 - t1}


def agree(a, b):
    """test_gpu_ba._compare's tolerances; returns a list of what differs (empty: the routes agree)."""
    opt, lm, rev, starts = a
    o_opt, o_lm, o_rev, o_starts = b
    bad = []
    if starts != o_starts:
        bad.append("starts")
    if not np.array_equal(rev, o_rev):
        bad.append("reverted")
    for k in range(len(opt)):
        Rg, Ro, tg, to = opt[k][:3, :3], o_opt[k][:3, :3], opt[k][:3, 3], o_opt[k][:3, 3]
        if np.arccos(np.clip((np.trace(Rg.T @ Ro) - 1) / 2, -1, 1)) >= 1e-4:
            bad.append("R %d" % k)
        if np.linalg.norm(to) > 0:
            c = tg @ to / (np.linalg.norm(tg) * np.linalg.norm(to))
            if np.arccos(np.clip(c, -1, 1)) >= 1e-3 or abs(np.linalg.norm(tg) / np.linalg.norm(to) - 1) >= 5e-3:
                bad.append("t %d" % k)
        elif np.linalg.norm(tg) != 0:
            bad.append("t %d" % k)
    ok = np.isfinite(o_lm[:, 1])
    if not np.allclose(lm[ok, 1], o_lm[ok, 1], rtol=1e-4, atol=1e-15):
        bad.append("r_norm")
    return bad


def main():
    args = [a for a in sys.argv[1:] if a != "--stereo"]
    stereo = len(args) < len(sys.argv) - 1
    F = int(args[0]) if len(args) > 0 else 1009
    reps = int(args[1]) if len(args) > 1 else 10
    os.environ.pop("EPIVO_LM_SHAPE", None)
    if stereo:
        seq = synth.make_sequence(n_frames=2 * F, n=2000)
        pairs = ba.window_pairs(ba.expand_stereo_window(WINDOW), 2 * STRIDE, 2 * F)
        pair_w = np.array([rig_weight(a, b) for a, b in pairs])
        workload = ("make_sequence(%d nodes = %d stereo frames, 2000), window %s expanded to %d node reps, stride %d "
                    "frames, weight 0 on (2f, 2f+1): %d pairs, %%d windows, LMEDS(.99, .1)"
                    % (2 * F, F, WINDOW, len(ba.expand_stereo_window(WINDOW)), STRIDE, len(pairs)))
    else:
        seq = synth.make_sequence(n_frames=F, n=2000)
        pairs = ba.window_pairs(WINDOW, STRIDE, F)
        pair_w = None
        workload = ("make_sequence(%d, 2000), window %s, stride %d: %d pairs, %%d windows, LMEDS(.99, .1)"
                    % (F, WINDOW, STRIDE, len(pairs)))
    prm = api.default_params(np.asarray(seq.K, dtype=np.float32), method=api.LMEDS, prob=0.99, threshold=0.1)
    ctx = api.Context(0)
    info = device_info()
    tc, tr, diffs = [], [], []
    for _ in range(reps + 1):                          # the first round is the warm-up
        a, ta = composed(ctx, seq, F, stereo)
        b, tb = resident(ctx, seq, pairs, prm, pair_w)
        tc.append(ta)
        tr.append(tb)
        diffs.append(agree(b, a))
    tc, tr = tc[1:], tr[1:]
    med = lambda rows, k: float(np.median([r[k] for r in rows])) * 1e3          # noqa: E731
    out = {"device": info,
           "workload": workload % len(b[3]),
           "method": "wall clock of whole calls, median of %d alternating rounds after one warm-up round" % reps,
           "composed_ms_median": {k: med(tc, k) for k in tc[0]},
           "resident_ms_median": {k: med(tr, k) for k in tr[0]},
           "speedup_total_median": med(tc, "total") / med(tr, "total"),
           # the composed route's BA step is the part of match_kp after its process call plus bundle_adjustment; match_kp
           # times its pipeline and process together, so that part is derived as match_kp - (resident) process
           "composed_ba_step_ms_derived": med(tc, "match_kp") - med(tr, "process") + med(tc, "bundle_adjustment"),
           "windows_reverted": int(np.asarray(b[2]).sum()),
           "outputs_agree": all(not d for d in diffs),
           "differences": sorted({x for d in diffs for x in d})}
    ctx.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
