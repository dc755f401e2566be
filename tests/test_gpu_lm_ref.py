"""GPU LM (epivo_lm_rt / epivo_lm_rt_batch through the C ABI) against the reference's OWN Levenberg_Marquardt:
tests/golden/lm_ref.npz holds the outputs of /root/reference/jac_Rt_gen_.cpp compiled unmodified (oracle/_ref,
tests/golden/make_golden_lm_ref.py) for the shapes the drivers and the demo run -- kitti_E.cpp:196 (1 zeta, 48
points), euroc_E.cpp:283-299, the demo's 10-zeta chain (test_jac_Rt_gen.cpp:282-297) on scenes drawn by the
reference's own generator, BASELINE config 5 (20 reps x 250), the kitti_ba stereo window (ws = 3), reverse reps,
a w = 0 rep, a singular H.  Comparison rule and tolerances: tests/lm_ref_util.py."""
import numpy as np
import pytest

from lm_ref_util import DELTAS, EPSILON, LAMBDA0, NAMES, case, check, gold

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from epivo_b200 import api
    c = api.Context(0)
    yield c
    c.close()


@pytest.mark.parametrize("tag", ["ref", "d1"])
@pytest.mark.parametrize("name", NAMES)
def test_gpu_lm_equals_reference_build(ctx, name, tag):
    from epivo_b200 import api
    c = case(name)
    T, info = api.Levenberg_Marquardt(c["n_zeta"], EPSILON, c["reps"], c["wreps"], LAMBDA0, c["T0s"], c["pr"], c["p_r"],
                                      huber_delta=DELTAS[tag], ctx=ctx)
    check(name, tag, T, info["r_norm"], info["lambda"], info["H_norm"])
    if gold(name, tag)["nan_break"]:
        assert np.array_equal(T, c["T0s"])                    # "delta has Nan" before any update (:407)


# epv_lm_launch picks the shape of a window with N >= 96 points per rep from the batch size B against the SM count
# (the value epivo_create reads): a cluster of 4 CTAs while 4 B <= SMs, of 2 while 2 B <= SMs, one 384-thread CTA
# while B <= SMs, else a 192-thread CTA
WIDE_SHAPE_BATCH = {"384x64x4": lambda sms: 1, "384x128x2": lambda sms: sms // 2, "384x128": lambda sms: sms,
                    "192x96": lambda sms: sms + 1}


@pytest.mark.parametrize("shape", list(WIDE_SHAPE_BATCH))
def test_gpu_lm_cfg5_on_every_launched_shape_equals_reference_build(ctx, shape):
    """The window kernel's shapes differ in summation order only: B copies of BASELINE config 5 in one batch, with B
    chosen so that the launcher picks `shape`, must meet the reference at both Huber settings, and every copy must
    equal the first bit for bit (one shape, one summation order).  The demo chain (N = 15) runs the 64 x 32 shape in
    test_gpu_lm_equals_reference_build."""
    import torch
    from epivo_b200 import api
    B = WIDE_SHAPE_BATCH[shape](torch.cuda.get_device_properties(0).multi_processor_count)
    c = case("cfg5_51")
    for tag in ("ref", "d1"):
        Tb, res, its = api.Levenberg_Marquardt_batch(c["n_zeta"], EPSILON, c["reps"], c["wreps"], LAMBDA0,
                                                     np.stack([c["T0s"]] * B), np.stack([c["pr"]] * B),
                                                     np.stack([c["p_r"]] * B), huber_delta=DELTAS[tag], ctx=ctx)
        check("cfg5_51", tag, Tb[0], res[0][1], res[0][2], res[0][0])
        assert (Tb == Tb[0]).all() and (res == res[0]).all() and (its == its[0]).all()


def test_gpu_lm_batch_of_kitti_e_pairs_equals_reference_build(ctx):
    """The single-pair kernel (8 lanes per problem) on a batch: the three kitti_E goldens side by side."""
    from epivo_b200 import api
    names = [n for n in NAMES if n.startswith("kitti_E")]
    cs = [case(n) for n in names]
    for tag in ("ref", "d1"):
        Tb, res, its = api.Levenberg_Marquardt_batch(1, EPSILON, [(0, 0)], [1.0], LAMBDA0, np.stack([c["T0s"] for c in cs]),
                                                     np.stack([c["pr"] for c in cs]), np.stack([c["p_r"] for c in cs]),
                                                     huber_delta=DELTAS[tag], ctx=ctx)
        for k, n in enumerate(names):
            check(n, tag, Tb[k], res[k][1], res[k][2], res[k][0])
