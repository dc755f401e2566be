"""Pins the LM oracle (numpy restatement oracle/oracle.py and plain-C restatement oracle/lm_c.c) against
the reference's OWN code: /root/reference/jac_Rt_gen_.cpp compiled unmodified into oracle/_ref
(oracle/Makefile, oracle/ref_lm_tu.cpp, Eigen/Sophus stand-ins in oracle/ref_shim/), and against
tests/golden/lm_ref.npz, the outputs of that build committed as fixtures
(tests/golden/make_golden_lm_ref.py).  The live-library tests skip where oracle/_ref is absent;
the golden tests, and the stand-in's SE3::exp compiled on its own, always run."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from epivo_b200 import synth
from oracle import clib, reflib
from oracle import oracle as O

from lm_ref_util import DELTAS, NAMES, case, check, check_trace, gold

SMALL = [n for n in NAMES if not n.startswith("cfg5")]          # numpy restatement: seconds per case

needs_ref = pytest.mark.skipif(not (reflib.available() or os.path.exists(reflib.REFERENCE_SRC)),
                               reason="oracle/_ref not built and /root/reference absent")


@pytest.mark.parametrize("tag", ["ref", "d1"])
@pytest.mark.parametrize("name", NAMES)
def test_c_restatement_equals_reference_build(name, tag):
    c = case(name)
    T, info = clib.levenberg_marquardt(c["n_zeta"], 1e-8, c["reps"], c["wreps"], 1e-2, c["T0s"], c["pr"], c["p_r"],
                                       huber_delta=DELTAS[tag])
    check(name, tag, T, info["r_norm"], info["lambda"], info["H_norm"])
    n = check_trace(name, tag, info["trace"])
    assert n >= min(14, len(gold(name, tag)["trace"]) - 1) or gold(name, tag)["nan_break"], n


@pytest.mark.parametrize("tag", ["ref", "d1"])
@pytest.mark.parametrize("name", SMALL)
def test_numpy_restatement_equals_reference_build(name, tag):
    c = case(name)
    T, info = O.levenberg_marquardt(c["n_zeta"], 1e-8, [tuple(r) for r in c["reps"]], list(c["wreps"]), 1e-2,
                                    c["T0s"], c["pr"], c["p_r"], huber_delta=DELTAS[tag])
    check(name, tag, T, info["r_norm"], info["lambda"], info["H_norm"])
    check_trace(name, tag, info["trace"])


@needs_ref
def test_reference_build_reproduces_its_goldens():
    """The committed fixtures are what oracle/_ref computes (same compiler, same machine class: exact)."""
    libs = {"ref": reflib.ref(), "d1": reflib.ref_d1()}
    assert libs["ref"].huber_delta == 1e-5 and libs["d1"].huber_delta == 1.0      # jac_Rt_gen_.cpp:17 / patched
    for name in SMALL:
        c = case(name)
        for tag, lib in libs.items():
            T, info = lib.levenberg_marquardt(c["n_zeta"], 1e-8, c["reps"], c["wreps"], 1e-2, c["T0s"], c["pr"], c["p_r"])
            g = gold(name, tag)
            assert (info["accepts"], info["rejects"], info["nan_break"]) == (g["acc"], g["rej"], g["nan_break"])
            assert np.abs(T - g["T"]).max() < 1e-12 and abs(info["r_norm"] - g["r_norm"]) <= 1e-10 * g["r_norm"] + 1e-20


@needs_ref
def test_res_and_jacobian_equal_reference_functions():
    """res (:212-259), Dr_Deps (:23-209, both `reverse` settings) and RepJacobian::compute (:262-284: forward,
    reverse, first / middle / last zeta) of the reference build vs the numpy restatement, at both deltas and for
    residuals on both sides of the Huber switch."""
    reps = [(0, 0), (0, 3), (3, 0), (2, 1), (1, 3)]
    for seed, noise in ((7, 1e-1), (8, 1e-3), (9, 1e-5)):
        Ts, T0s, pr, p_r = synth.gen_scene_sequence(seed, 40, 4, reps, noise_rot=noise, noise_tr=noise)
        mem = O.chain_memo(list(T0s))
        for tag, lib in (("ref", reflib.ref()), ("d1", reflib.ref_d1())):
            d = DELTAS[tag]
            for j, (s, t) in enumerate(reps):
                T = synth.compose_rep(T0s, s, t)
                a = lib.res(T[:3, :3], T[:3, 3], pr[j], p_r[j])
                b = O.res(T[:3, :3], T[:3, 3], pr[j], p_r[j], d)
                assert np.abs(a - b).max() <= 1e-9 * max(np.abs(b).max(), 1e-30) + 1e-22      # e = p' - X'/z cancels ~1e-4
                for z in range(min(s, t), max(s, t) + 1):
                    Ja = lib.rep_jacobian(T0s, z, s, t, pr[j], p_r[j])
                    Jb = O.rep_jacobian(mem, z, s, t, pr[j], p_r[j], d)
                    assert np.abs(Ja - Jb).max() <= 1e-8 * max(np.abs(Jb).max(), 1e-30)
            for rev in (False, True):
                Ja = lib.dr_deps(T0s[1], T0s[0], pr[1], p_r[1], rev)
                Jb = O.dr_deps(T0s[1], T0s[0], pr[1], p_r[1], rev, d)
                assert np.abs(Ja - Jb).max() <= 1e-8 * np.abs(Jb).max()
    # the demo translation unit (test_jac_Rt_gen.cpp, delta = 1.0, no `reverse`) agrees with the restatement too
    dm = reflib.demo()
    assert dm.huber_delta == 1.0
    Ja = dm.rep_jacobian(T0s, 2, 1, 3, pr[4], p_r[4])
    assert np.abs(Ja - O.rep_jacobian(mem, 2, 1, 3, pr[4], p_r[4], 1.0)).max() <= 1e-10 * np.abs(Ja).max()


def _standin_se3_exp(tmp_dir):
    """SE3::exp of the Sophus stand-in the reference build links, compiled on its own (tests/cpp/se3_exp_standin.cpp)
    with the flags oracle/Makefile gives the stand-in."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    shim = os.path.join(root, "oracle", "ref_shim")
    so = os.path.join(str(tmp_dir), "se3_exp_standin.so")
    p = subprocess.run(["g++", "-O2", "-fPIC", "-ffp-contract=off", "-DNDEBUG", "-I", shim, "-shared",
                        os.path.join(root, "tests", "cpp", "se3_exp_standin.cpp"), os.path.join(shim, "standin_impl.cpp"),
                        "-o", so], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    fn = C.CDLL(so).standin_se3_exp
    fn.restype, fn.argtypes = None, [C.c_void_p, C.c_void_p]

    def se3_exp(a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        T = np.zeros((4, 4))
        fn(a.ctypes.data, T.ctypes.data)
        return T
    return se3_exp


def test_se3_exp_equals_sophus_standin(tmp_path):
    """The numpy restatement against the stand-in's SE3::exp, and against the reference build's export of it where
    that build is present."""
    rng = np.random.default_rng(3)
    impls = [_standin_se3_exp(tmp_path)]
    if reflib.available() or os.path.exists(reflib.REFERENCE_SRC):
        impls.append(reflib.ref().se3_exp)
    for scale in (1.0, 1e-3, 1e-8, 1e-12, 0.0):
        for _ in range(5):
            a = rng.normal(size=6) * np.array([1, 1, 1, scale, scale, scale])
            for se3_exp in impls:
                assert np.abs(se3_exp(a) - O.se3_exp(a)).max() < 1e-14


@needs_ref
def test_reference_generator_matches_synth_contract():
    """sequence.hpp:64-104 through the reference build: p = X / X_z, p' = (T X) / (T X)_z with depth > 10 in
    view 1, noiseless -- the contract epivo_b200/synth.py's generator restates."""
    reps = [(0, 0), (0, 2), (2, 1)]
    Ts, T0s, Xr, pr, p_r = reflib.ref().gen_scene_sequence(17, 12, 3, reps)
    for j, (s, t) in enumerate(reps):
        T = synth.compose_rep(Ts, s, t)
        Xp = Xr[j] @ T[:3, :3].T + T[:3, 3]
        assert (Xr[j][:, 2] > 0).all() and (Xp[:, 2] > 10.0).all()
        assert np.allclose(pr[j], Xr[j] / Xr[j][:, 2:3], atol=1e-14)
        assert np.allclose(p_r[j], Xp / Xp[:, 2:3], atol=1e-12)
    for k in range(3):
        assert np.allclose(Ts[k][:3, :3] @ Ts[k][:3, :3].T, np.eye(3), atol=1e-14) and Ts[k][2, 3] >= 0


@needs_ref
def test_reference_demo_converges(tmp_path):
    """test_jac_Rt_gen.cpp's main(), unmodified (seeded): after its 60 LM iterations it prints, per zeta,
    ||R - R0|| and the three t / t0 ratios -- rotation recovered, translation up to ONE common scale."""
    log = reflib.demo().demo(3, cwd=str(tmp_path))
    nums = [[float(x) for x in ln.split()] for ln in log.splitlines() if ln.strip()]
    head, body = nums[0], nums[1:]
    assert len(head) == 4 and head[1] < 1e-12                    # " |H| |r0| |delta| lambda"
    assert len(body) == 40
    ratios = []
    for z in range(10):
        rot_err, t, t0, ratio = body[4 * z: 4 * z + 4]
        assert len(rot_err) == 1 and rot_err[0] < 1e-8
        ratios += ratio
    assert np.ptp(ratios) < 1e-5 * abs(ratios[0])
    assert (tmp_path / "est.pose").exists() and (tmp_path / "gt.pose").exists()
