"""The fused sequence pipeline (epivo_seq_*) against the oracle pipeline, pair by pair."""
import numpy as np
import pytest

from conftest import esame
from epivo_b200 import api, synth
from oracle import oracle as O
from oracle import pipeline as OP

pytestmark = pytest.mark.gpu


def rot_angle(Ra, Rb):
    return float(np.arccos(np.clip((np.trace(Ra.T @ Rb) - 1) / 2, -1, 1)))


@pytest.fixture(scope="module")
def seq():
    return synth.make_sequence(n_frames=7, n=2000, seed=synth.seed_for(3, 1))


@pytest.mark.parametrize("method,thr", [(api.RANSAC, 1.0), (api.LMEDS, 0.01)])
def test_sequence_vs_oracle(ctx, seq, method, thr):
    P = seq.n_pairs
    pipe = api.SequencePipeline(seq.n_frames, 2000, ctx=ctx)
    pipe.upload(seq.kps, seq.descs)
    prm = api.default_params(seq.K.astype(np.float32), method=method, threshold=thr)   # cam is a float Mat (kitti_E.cpp:38)
    pipe.run(prm, 0, P)
    res = pipe.download(0, P)
    for i in range(P):
        o = OP.pair_pipeline(seq.kps[i], seq.descs[i], seq.kps[i + 1], seq.descs[i + 1], seq.K, method, 0.99, thr)
        qi, ti, d = pipe.matches(i)
        for g, w in zip((qi, ti, d), o["matches"]):
            assert np.array_equal(g, w)                       # bit-exact match indices
        em, pm = pipe.masks(i)
        assert np.array_equal(em, o["e_mask"])                # bit-exact inlier mask
        assert np.array_equal(pm, o["pose_mask"])
        r = res[i]
        assert r["n_matches"] == len(qi) and r["n_inliers"] == int(o["e_mask"].sum())
        assert r["n_good"] == o["n_good"] and r["ransac_iters"] == o["e_info"]["iters"]
        assert esame(r["E"], o["E"]) < 1e-9
        assert rot_angle(r["R"], o["R"]) < 1e-4
        assert np.arccos(np.clip(r["t"] @ o["t"], -1, 1)) < 1e-3
        assert bool(r["lm_ran"]) == o["lm_ran"]
        assert np.abs(r["T0"] - o["T0"]).max() < 1e-7
        if o["lm_ran"]:
            assert bool(r["lm_reverted"]) == o["lm_reverted"]
            assert abs(r["r_norm"] - o["lm"]["r_norm"]) <= 1e-5 * o["lm"]["r_norm"]
        assert rot_angle(r["T"][:3, :3], o["T"][:3, :3]) < 1e-4
        # and the estimate is close to the synthetic ground truth
        assert rot_angle(r["R"], seq.R[i]) < 5e-3
    ms = pipe.stage_ms()
    assert ms[0] > 0 and ms[7] > 0
    pipe.close()


def test_sequence_chunking_and_subranges(ctx, seq):
    """Running a sub-range, or the same range twice, gives identical results (idempotence)."""
    pipe = api.SequencePipeline(seq.n_frames, 2000, ctx=ctx)
    pipe.upload(seq.kps, seq.descs)
    prm = api.default_params(seq.K.astype(np.float32))
    pipe.run(prm, 0, seq.n_pairs)
    a = pipe.download(0, seq.n_pairs).copy()
    pipe.run(prm, 2, 3)
    b = pipe.download(2, 3).copy()
    assert a[2:5].tobytes() == b.tobytes()
    pipe.run(prm, 0, seq.n_pairs)
    c = pipe.download(0, seq.n_pairs)
    assert a.tobytes() == c.tobytes()
    pipe.close()


def test_run_split_into_groups_identical(ctx):
    """More pairs than one group of 8192 holds: the run takes two matcher and two geometry groups, and its bytes are
    those of the same pairs run as two sub-ranges of one group each."""
    s = synth.make_sequence(n_frames=8201, n=256, seed=synth.seed_for(3, 2))
    P = s.n_pairs
    assert P >= 8193
    pipe = api.SequencePipeline(s.n_frames, 256, ctx=ctx)
    pipe.upload(s.kps, s.descs)
    prm = api.default_params(s.K.astype(np.float32))
    pipe.run(prm, 0, P)
    a = pipe.download(0, P).copy()
    assert pipe.stage_ms()[8] == 2
    h = P // 2
    pipe.run(prm, 0, h)
    b0 = pipe.download(0, h).copy()
    pipe.run(prm, h, P - h)
    b1 = pipe.download(h, P - h).copy()
    assert a.tobytes() == b0.tobytes() + b1.tobytes()
    assert (a["n_matches"] > 50).all()
    pipe.close()


def test_process_host_buffers_equals_upload_run_download(ctx):
    s = synth.make_sequence(n_frames=1201, n=256, seed=synth.seed_for(3, 3))
    pipe = api.SequencePipeline(s.n_frames, 256, ctx=ctx)
    prm = api.default_params(s.K.astype(np.float32))
    a = pipe.process(prm, s.kps, s.descs).copy()
    pipe2 = api.SequencePipeline(s.n_frames, 256, ctx=ctx)
    pipe2.upload(s.kps, s.descs)
    pipe2.run(prm, 0, s.n_pairs)
    b = pipe2.download(0, s.n_pairs)
    assert a.tobytes() == b.tobytes()
    pipe.close()
    pipe2.close()


def test_process_many_pieces_identical(ctx):
    """Host-buffer path with the default upload plan cut into many pieces (at least 8, checked), over repeated calls on
    one object, and for LMedS and the ratio matcher with plain Hamming (no planes on the copy stream): every call gives
    the bytes of upload + run + download."""
    s = synth.make_sequence(n_frames=5001, n=256, seed=synth.seed_for(3, 5))
    ref_pipe = api.SequencePipeline(s.n_frames, 256, ctx=ctx)
    ref_pipe.upload(s.kps, s.descs)
    pipe = api.SequencePipeline(s.n_frames, 256, ctx=ctx)
    for i, kw in enumerate((dict(), dict(method=api.LMEDS, threshold=0.01),
                            dict(norm=api.NORM_HAMMING, match_mode=api.MATCH_RATIO))):
        prm = api.default_params(s.K.astype(np.float32), **kw)
        ref_pipe.run(prm, 0, s.n_pairs)
        ref = ref_pipe.download(0, s.n_pairs).tobytes()
        for _ in range(3 if i == 0 else 1):
            assert pipe.process(prm, s.kps, s.descs).tobytes() == ref, kw
            ms = pipe.stage_ms()
            assert ms[0] > 0 and ms[8] >= 8, (kw, ms[8])
    ref_pipe.close()
    pipe.close()


def test_ratio_mode_pipeline(ctx, seq):
    pipe = api.SequencePipeline(seq.n_frames, 2000, ctx=ctx)
    pipe.upload(seq.kps, seq.descs)
    prm = api.default_params(seq.K.astype(np.float32), norm=api.NORM_HAMMING, match_mode=api.MATCH_RATIO)
    pipe.run(prm, 0, 2)
    res = pipe.download(0, 2)
    for i in range(2):
        qi, ti, d = pipe.matches(i)
        w = O.ratio_match(seq.descs[i], seq.descs[i + 1], 0.8, O.NORM_HAMMING)
        assert np.array_equal(qi, w[0]) and np.array_equal(ti, w[1]) and np.array_equal(d, w[2])
        assert rot_angle(res[i]["R"], seq.R[i]) < 5e-3
    pipe.close()
