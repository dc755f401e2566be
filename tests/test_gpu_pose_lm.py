"""P1 (recoverPose) and L4 (Levenberg_Marquardt) parity through the C ABI."""
import numpy as np
import pytest

from epivo_b200 import api, synth
from oracle import oracle as O

pytestmark = pytest.mark.gpu
CASES = ["kitti", "kitti_b", "euroc"]
CALLS = ["ransac10", "ransac03", "ransac005", "lmeds"]
ROT_TOL, T_TOL = 1e-4, 1e-3          # north_star: rotation <= 1e-4 rad, unit-t angle <= 1e-3 rad


def rot_angle(Ra, Rb):
    return float(np.arccos(np.clip((np.trace(Ra.T @ Rb) - 1) / 2, -1, 1)))


def vec_angle(a, b):
    a, b = a / np.linalg.norm(a), b / np.linalg.norm(b)
    return float(np.arccos(np.clip(a @ b, -1, 1)))


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("cname", CALLS)
def test_recover_pose_vs_cv2(ctx, golden_ess, case, cname):
    p0, p1, K = golden_ess[f"{case}_p0"], golden_ess[f"{case}_p1"], golden_ess[f"{case}_K"]
    E, m = golden_ess[f"{case}_{cname}_E"], golden_ess[f"{case}_{cname}_mask"] == 1
    n, R, t, mask = api.recoverPose(E, p0[m], p1[m], K, ctx=ctx)
    assert rot_angle(R, golden_ess[f"{case}_{cname}_R"]) < ROT_TOL
    assert vec_angle(t, golden_ess[f"{case}_{cname}_t"]) < T_TOL
    assert np.array_equal(mask, golden_ess[f"{case}_{cname}_pose_mask"])     # {0,255}, identical
    assert n == int(golden_ess[f"{case}_{cname}_pose_n"])
    assert abs(np.linalg.det(R) - 1) < 1e-12 and abs(np.linalg.norm(t) - 1) < 1e-12


def test_recover_pose_input_mask_and_sign(ctx, golden_ess):
    p0, p1, K = golden_ess["kitti_p0"], golden_ess["kitti_p1"], golden_ess["kitti_K"]
    E, m = golden_ess["kitti_ransac10_E"], golden_ess["kitti_ransac10_mask"] == 1
    c0, c1 = p0[m], p1[m]
    im = (np.arange(len(c0)) % 3 != 0).astype(np.uint8)
    n, R, t, mask = api.recoverPose(E, c0, c1, K, mask=im, ctx=ctx)
    no, Ro, to, mo = O.recover_pose(E, c0, c1, K, in_mask=im)
    assert n == no and np.array_equal(mask, mo) and not mask[im == 0].any()
    # -E decomposes into the same four candidates: same winner
    n2, R2, t2, mask2 = api.recoverPose(-E, c0, c1, K, ctx=ctx)
    n1, R1, t1, mask1 = api.recoverPose(E, c0, c1, K, ctx=ctx)
    assert n1 == n2 and np.abs(R1 - R2).max() < 1e-9 and np.abs(t1 - t2).max() < 1e-9 and np.array_equal(mask1, mask2)
    # empty input
    n0, R0, t0, m0 = api.recoverPose(E, np.zeros((0, 2), np.float32), np.zeros((0, 2), np.float32), K, ctx=ctx)
    assert n0 == 0 and len(m0) == 0


REPS10 = [(i, i) for i in range(10)] + [(0, i) for i in range(10)]    # test_jac_Rt_gen.cpp:294-297


def _check_lm(ctx, n_zeta, reps, N, seed, delta, iters, w=None, tol=1e-5):
    Ts, T0s, pr, p_r = synth.gen_scene_sequence(seed, N, n_zeta, reps)
    w = [1.0] * len(reps) if w is None else w
    To, lo = O.levenberg_marquardt(n_zeta, 1e-8, reps, w, 1e-2, T0s, pr, p_r, huber_delta=delta, max_iters=iters)
    Tg, lg = api.Levenberg_Marquardt(n_zeta, 1e-8, reps, w, 1e-2, T0s, pr, p_r, huber_delta=delta,
                                     max_iters=iters, ctx=ctx)
    assert lg["iters"] == lo["iters"]
    for k in range(n_zeta):
        assert rot_angle(Tg[k][:3, :3], To[k][:3, :3]) < ROT_TOL
        assert np.abs(Tg[k][:3, 3] - To[k][:3, 3]).max() < 1e-6 * max(1.0, np.abs(To[k][:3, 3]).max())
    assert abs(lg["r_norm"] - lo["r_norm"]) <= tol * max(lo["r_norm"], 1e-12) + 1e-15   # relative residual <= 1e-5
    assert abs(lg["lambda"] - lo["lambda"]) <= 1e-9 * lo["lambda"]
    assert abs(lg["H_norm"] - lo["H_norm"]) <= 1e-5 * max(lo["H_norm"], 1e-12) + 1e-15
    return Ts, Tg, lg


def test_lm_single_pair_shipped_delta(ctx):
    """kitti_E.cpp:196 shape: n_zeta = 1, reps = {(0,0)}, N = 48, delta = 1e-5 (as shipped)."""
    for seed in (1, 2, 3):
        _check_lm(ctx, 1, [(0, 0)], 48, seed, 1e-5, 30)


def test_lm_single_pair_converges(ctx):
    Ts, Tg, lg = _check_lm(ctx, 1, [(0, 0)], 48, 11, 1.0, 60)
    assert lg["r_norm"] < 1e-12
    assert np.linalg.norm(Tg[0][:3, :3] - Ts[0][:3, :3]) < 1e-6
    ratio = Ts[0][:3, 3] / Tg[0][:3, 3]                       # scale is unobservable: constant ratio
    assert np.ptp(ratio) < 1e-5 * abs(ratio.mean())


def test_lm_window_demo_shape(ctx):
    """test_jac_Rt_gen.cpp:280-513: n_zeta = 10, 20 reps, N = 15, delta = 1.0, 60 iterations."""
    Ts, Tg, lg = _check_lm(ctx, 10, REPS10, 15, 21, 1.0, 60)
    for k in range(10):
        assert np.linalg.norm(Tg[k][:3, :3] - Ts[k][:3, :3]) < 1e-5


def test_lm_reverse_reps_and_weights(ctx):
    reps = [(0, 0), (1, 1), (2, 2), (0, 2), (2, 0), (1, 0), (2, 1)]
    _check_lm(ctx, 3, reps, 32, 31, 1.0, 30, w=[1.0, 1.0, 1.0, 0.5, 1.0, 2.0, 1.0])
    _check_lm(ctx, 3, reps, 32, 32, 1e-5, 30)


def test_lm_zero_weight_rep_gives_nan_stop(ctx):
    """kitti_ba.cpp:821-826: a '<32 points' rep gets weight 0 and all-ones dummy points; if a zeta
    is covered by nothing else H is singular, delta has NaN and the loop stops (jac_Rt_gen_.cpp:407)."""
    reps = [(0, 0), (1, 1)]
    Ts, T0s, pr, p_r = synth.gen_scene_sequence(5, 32, 2, reps)
    pr[1][:] = 1.0
    p_r[1][:] = 1.0
    To, lo = O.levenberg_marquardt(2, 1e-8, reps, [1.0, 0.0], 1e-2, T0s, pr, p_r)
    Tg, lg = api.Levenberg_Marquardt(2, 1e-8, reps, [1.0, 0.0], 1e-2, T0s, pr, p_r, ctx=ctx)
    assert lo["iters"] == lg["iters"] == 1
    assert np.allclose(Tg, T0s) and np.allclose(To, T0s)


def test_lm_batch_and_errors(ctx):
    reps = [(0, 0), (0, 1), (1, 1)]
    B = 6
    T0b, prb, p_rb = [], [], []
    for b in range(B):
        _, T0s, pr, p_r = synth.gen_scene_sequence(100 + b, 32, 2, reps)
        T0b.append(T0s); prb.append(pr); p_rb.append(p_r)
    Tb, res, its = api.Levenberg_Marquardt_batch(2, 1e-8, reps, [1.0, 1.0, 1.0], 1e-2, np.stack(T0b), np.stack(prb),
                                                 np.stack(p_rb), huber_delta=1.0, ctx=ctx)
    for b in range(B):
        To, lo = O.levenberg_marquardt(2, 1e-8, reps, [1.0] * 3, 1e-2, T0b[b], prb[b], p_rb[b], huber_delta=1.0)
        assert its[b] == lo["iters"]
        assert np.abs(Tb[b] - To).max() < 1e-6
        assert abs(res[b][1] - lo["r_norm"]) <= 1e-5 * lo["r_norm"] + 1e-15
    with pytest.raises(api.EpivoError):
        api.Levenberg_Marquardt(2, 1e-8, [(0, 2)], [1.0], 1e-2, T0b[0], prb[0][:1], p_rb[0][:1], ctx=ctx)
    with pytest.raises(ValueError):
        api.Levenberg_Marquardt(2, 1e-8, reps, [1.0], 1e-2, T0b[0], prb[0], p_rb[0], ctx=ctx)


def _sms():
    """The SM count epivo_create reads: the LM launcher compares the batch size with it to pick a kernel shape."""
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _check_vs_c(ctx, n_zeta, reps, N, seed, delta, iters, w=None, copies=1):
    """One window against the plain-C restatement; copies > 1 runs that many copies of it in one batch (the batch size
    picks the kernel shape), and every copy must equal the first bit for bit."""
    from oracle import clib
    Ts, T0s, pr, p_r = synth.gen_scene_sequence(seed, N, n_zeta, reps)
    w = [1.0] * len(reps) if w is None else w
    To, lo = clib.levenberg_marquardt(n_zeta, 1e-8, reps, w, 1e-2, T0s, pr, p_r, huber_delta=delta, max_iters=iters)
    if copies == 1:
        Tg, lg = api.Levenberg_Marquardt(n_zeta, 1e-8, reps, w, 1e-2, T0s, pr, p_r, huber_delta=delta,
                                         max_iters=iters, ctx=ctx)
    else:
        Tb, res, its = api.Levenberg_Marquardt_batch(n_zeta, 1e-8, reps, w, 1e-2, np.stack([T0s] * copies),
                                                     np.stack([pr] * copies), np.stack([p_r] * copies),
                                                     huber_delta=delta, max_iters=iters, ctx=ctx)
        assert (Tb == Tb[0]).all() and (res == res[0]).all() and (its == its[0]).all()
        Tg, lg = Tb[0], {"iters": its[0], "r_norm": res[0][1]}
    assert lg["iters"] == lo["iters"]
    for k in range(n_zeta):
        assert rot_angle(Tg[k][:3, :3], To[k][:3, :3]) < ROT_TOL
        assert np.abs(Tg[k][:3, 3] - To[k][:3, 3]).max() < 1e-6 * max(1.0, np.abs(To[k][:3, 3]).max())
    assert abs(lg["r_norm"] - lo["r_norm"]) <= 1e-5 * max(lo["r_norm"], 1e-12) + 1e-15
    return Ts, Tg, lg


def test_lm_cfg5_window_full_size(ctx):
    """BASELINE config 5: n_zeta = 10, reps {(i,i),(0,i)} (test_jac_Rt_gen.cpp:294-297) x N = 250
    = 5000 correspondences, J 5000 x 60, H 60 x 60; against the plain-C restatement."""
    Ts, Tg, lg = _check_vs_c(ctx, 10, REPS10, 250, 51, 1.0, 30)
    for k in range(10):
        assert np.linalg.norm(Tg[k][:3, :3] - Ts[k][:3, :3]) < 1e-5
    _check_vs_c(ctx, 10, REPS10, 250, 52, 1e-5, 30)


def test_lm_kitti_ba_stereo_window_shape(ctx):
    """The shape kitti_ba.cpp ships: ws = 3 stereo -> 9 reps x 32 points, n_zeta = 4
    (kitti_ba.cpp:931-938,969-975,1038): reps below are what those lines build."""
    reps = [(0, 1), (1, 1), (0, 0), (0, 3), (1, 3), (0, 0), (2, 3), (3, 3), (2, 2)]
    _check_vs_c(ctx, 4, reps, 32, 61, 1.0, 30)
    _check_vs_c(ctx, 4, reps, 32, 62, 1e-5, 30)
    # a '<32 points' rep: weight 0 and all-ones dummy points (kitti_ba.cpp:983-987)
    from oracle import clib
    Ts, T0s, pr, p_r = synth.gen_scene_sequence(63, 32, 4, reps)
    pr[4][:] = 1.0
    p_r[4][:] = 1.0
    w = [1.0] * 9
    w[4] = 0.0
    To, lo = clib.levenberg_marquardt(4, 1e-8, reps, w, 1e-2, T0s, pr, p_r, huber_delta=1.0)
    Tg, lg = api.Levenberg_Marquardt(4, 1e-8, reps, w, 1e-2, T0s, pr, p_r, huber_delta=1.0, ctx=ctx)
    assert lg["iters"] == lo["iters"] and np.abs(Tg - To).max() < 1e-6


def test_lm_window_batch_sharded_like_8_gpus(ctx):
    """kitti_ba windows are independent: a rank's block of windows is one batched launch."""
    from epivo_b200 import shard
    from oracle import clib
    reps = [(0, 0), (1, 1), (2, 2), (0, 2), (0, 1), (1, 2)]
    B = 10
    data = [synth.gen_scene_sequence(200 + b, 32, 3, reps) for b in range(B)]
    a, b_ = shard.shard_range(B, 8, 1)            # rank 1 of 8
    Tb, res, its = api.Levenberg_Marquardt_batch(3, 1e-8, reps, [1.0] * 6, 1e-2, np.stack([d[1] for d in data[a:b_]]),
                                                 np.stack([d[2] for d in data[a:b_]]),
                                                 np.stack([d[3] for d in data[a:b_]]), huber_delta=1.0, ctx=ctx)
    for k, d in enumerate(data[a:b_]):
        To, lo = clib.levenberg_marquardt(3, 1e-8, reps, [1.0] * 6, 1e-2, d[1], d[2], d[3], huber_delta=1.0)
        assert its[k] == lo["iters"] and np.abs(Tb[k] - To).max() < 1e-6


def _lm_batch(ctx, data, delta):
    return api.Levenberg_Marquardt_batch(10, 1e-8, REPS10, [1.0] * 20, 1e-2, np.stack([d[1] for d in data]),
                                         np.stack([d[2] for d in data]), np.stack([d[3] for d in data]),
                                         huber_delta=delta, ctx=ctx)


def _check_batch_vs_c(data, Tb, res, its, delta, tol=1e-6):
    """The first len(data) windows of a REPS10 batch against the plain-C restatement, window by window."""
    from oracle import clib
    for k, d in enumerate(data):
        To, lo = clib.levenberg_marquardt(10, 1e-8, REPS10, [1.0] * 20, 1e-2, d[1], d[2], d[3], huber_delta=delta)
        assert its[k] == lo["iters"] and np.abs(Tb[k] - To).max() < tol
        for z in range(10):
            assert rot_angle(Tb[k][z][:3, :3], To[z][:3, :3]) < ROT_TOL
        assert abs(res[k][1] - lo["r_norm"]) <= 1e-5 * max(lo["r_norm"], 1e-12) + 1e-15


@pytest.mark.parametrize("shape", ["384x64x4", "384x128x2"])
def test_lm_cfg5_window_on_a_cluster(ctx, shape):
    """Small batches share a window between the CTAs of a thread-block cluster (partial H | b summed over DSMEM): the
    launcher takes clusters of four CTAs for one window (4 B <= SMs) and of two for SMs / 2 windows (2 B <= SMs).
    Same parity bar as the one-CTA kernel, against the plain-C restatement, both Huber settings, plus a batch whose
    windows differ (every cluster must keep to its own window)."""
    B = 1 if shape == "384x64x4" else _sms() // 2
    Ts, Tg, lg = _check_vs_c(ctx, 10, REPS10, 250, 51, 1.0, 30, copies=B)
    for k in range(10):
        assert np.linalg.norm(Tg[k][:3, :3] - Ts[k][:3, :3]) < 1e-5
    _check_vs_c(ctx, 10, REPS10, 250, 52, 1e-5, 30, copies=B)
    _check_vs_c(ctx, 10, REPS10, 97, 53, 1.0, 30, copies=B)   # ragged last tile, tiles not a multiple of the cluster
    data = [synth.gen_scene_sequence(s, 130, 10, REPS10) for s in range(300, 300 + max(B, 5))]
    Tb, res, its = _lm_batch(ctx, data, 1.0)
    # the first five windows against the C code (one is still descending after 30 iterations: its translation scale, a
    # gauge freedom of the reprojection error, is pinned to ~2e-6 only, for the one-CTA kernel as well).  The others
    # include windows that the C code itself moves by up to 0.1 under a 1-ulp change of the input, so every window is
    # checked for isolation instead: the batch rolled by one returns the same bytes, rolled.
    _check_batch_vs_c(data[:5], Tb, res, its, 1.0, tol=1e-5)
    Tr, rr, ir = _lm_batch(ctx, data[1:] + data[:1], 1.0)
    assert (np.roll(Tr, 1, 0) == Tb).all() and (np.roll(rr, 1, 0) == res).all() and (np.roll(ir, 1, 0) == its).all()


def test_lm_window_of_64_points(ctx):
    """Windows of 33..95 points per rep run on 128-thread CTAs with 64-point tiles whatever the batch size: REPS10 with
    N = 64 alone and in a batch of four distinct windows, both Huber settings, against the plain-C restatement."""
    for delta in (1.0, 1e-5):
        _check_vs_c(ctx, 10, REPS10, 64, 80, delta, 30)
        data = [synth.gen_scene_sequence(s, 64, 10, REPS10) for s in range(81, 85)]
        _check_batch_vs_c(data, *_lm_batch(ctx, data, delta), delta)


def test_lm_long_chain_uses_the_small_tile_shape(ctx):
    """Chain length: the reference's bound is rep_max = 128 (jac_Rt_gen_.cpp:18); a window lives in shared memory here,
    which fits up to n_zeta = 19 on the smallest tile shape (chosen automatically).  n_zeta = 18 against the C
    restatement; n_zeta = 24 is refused with an error, never truncated."""
    nz = 18
    reps = [(i, i) for i in range(nz)] + [(0, i) for i in range(1, nz, 4)] + [(nz - 1, nz - 3)]
    _check_vs_c(ctx, nz, reps, 24, 91, 1.0, 30)
    nz = 24
    reps = [(i, i) for i in range(nz)]
    Ts, T0s, pr, p_r = synth.gen_scene_sequence(92, 8, nz, reps)
    with pytest.raises(api.EpivoError):
        api.Levenberg_Marquardt(nz, 1e-8, reps, [1.0] * nz, 1e-2, T0s, pr, p_r, ctx=ctx)
