"""ctypes binding of libepivo_b200.so (the C ABI in include/epivo_b200.h).

The library is loaded from the package directory (built in-tree by epivo_b200/build.py).
There is no fallback: if the shared object is missing, or no CUDA device can be opened,
the product path raises.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# EPIVO_VARIANT selects a tuning build made by build.py with the same variable (default: the product library)
_VARIANT = os.environ.get("EPIVO_VARIANT", "")
LIB_PATH = os.path.join(HERE, "libepivo_b200" + ("_" + _VARIANT if _VARIANT else "") + ".so")

OK, ERR_INVALID, ERR_CUDA, ERR_UNSUPPORTED, ERR_NOMODEL = 0, -1, -2, -3, -4
NORM_HAMMING, NORM_HAMMING2 = 6, 7
LMEDS, RANSAC = 4, 8
MATCH_NN, MATCH_CROSSCHECK, MATCH_RATIO = 0, 1, 2


class EpivoError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"epivo_b200 error {code}: {msg}")
        self.code = code


class LmRes(C.Structure):
    _fields_ = [("H_norm", C.c_double), ("r_norm", C.c_double), ("lambda_", C.c_double)]


class PipelineParams(C.Structure):
    _fields_ = [("norm", C.c_int), ("match_mode", C.c_int), ("ratio", C.c_float),
                ("K", C.c_double * 9), ("method", C.c_int), ("prob", C.c_double),
                ("threshold", C.c_double), ("max_iters", C.c_int), ("dist_thresh", C.c_double),
                ("min_trace", C.c_double), ("fallback_t", C.c_double * 3), ("min_t_norm", C.c_double),
                ("lm_points", C.c_int), ("lm_lambda0", C.c_double), ("lm_epsilon", C.c_double),
                ("lm_max_iters", C.c_int), ("huber_delta", C.c_double), ("lm_revert", C.c_double)]


class PairResult(C.Structure):
    _fields_ = [("E", C.c_double * 9), ("R", C.c_double * 9), ("t", C.c_double * 3),
                ("T0", C.c_double * 16), ("T", C.c_double * 16), ("lm", LmRes),
                ("n_matches", C.c_int32), ("n_inliers", C.c_int32), ("n_good", C.c_int32),
                ("ransac_iters", C.c_int32), ("n_models", C.c_int32), ("lm_iters", C.c_int32),
                ("lm_ran", C.c_int32), ("lm_reverted", C.c_int32)]


_vp, _i, _d, _f = C.c_void_p, C.c_int, C.c_double, C.c_float
_pi = C.POINTER(C.c_int)

# name -> (restype, argtypes); every symbol include/epivo_b200.h declares
SIGNATURES = {
    "epivo_create": (_i, [C.POINTER(_vp), _i]),
    "epivo_destroy": (None, [_vp]),
    "epivo_last_error": (C.c_char_p, [_vp]),
    "epivo_version": (C.c_char_p, []),
    "epivo_stream": (_vp, [_vp]),
    "epivo_launch_count": (C.c_int64, [_vp]),
    "epivo_sync": (_i, [_vp]),
    "epivo_match_hamming": (_i, [_vp, _vp, _i, _vp, _i, _i, _i, _i, _f, _vp, _vp, _vp, _vp, _pi]),
    "epivo_knn2_hamming": (_i, [_vp, _vp, _i, _vp, _i, _i, _i, _vp, _vp]),
    "epivo_find_essential": (_i, [_vp, _vp, _vp, _i, _vp, _i, _d, _d, _i, _vp, _i, _vp, _vp, _pi, _pi]),
    "epivo_five_point": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "epivo_score_sampson": (_i, [_vp, _vp, _i, _vp, _vp, _i, _vp, _d, _vp, _vp, _pi, _vp]),
    "epivo_recover_pose": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _d, _vp, _vp, _vp, _vp, _pi]),
    "epivo_lm_rt": (_i, [_vp, _i, _d, _vp, _vp, _i, _d, _i, _d, _vp, _vp, _vp, _i, C.POINTER(LmRes), _pi]),
    "epivo_lm_rt_batch": (_i, [_vp, _i, _i, _d, _vp, _vp, _i, _d, _i, _d, _vp, _vp, _vp, _i, _vp, _vp]),
    "epivo_pipeline_params_default": (None, [C.POINTER(PipelineParams)]),
    "epivo_seq_create": (_i, [_vp, C.POINTER(_vp), _i, _i]),
    "epivo_seq_destroy": (None, [_vp]),
    "epivo_seq_upload": (_i, [_vp, _i, _i, _vp, _vp]),
    "epivo_last_kernel_ms": (_i, [_vp, _vp]),
    "epivo_seq_set_counts": (_i, [_vp, _i, _i, _vp]),
    "epivo_seq_extract_orb": (_i, [_vp, _i, _i, _vp, _i, _i, _i, C.c_float, _i, _i, _i, _vp]),
    "epivo_seq_create_pairs": (_i, [_vp, C.POINTER(_vp), _i, _i, _i]),
    "epivo_seq_set_pairs": (_i, [_vp, _i, _vp, _vp]),
    "epivo_seq_run": (_i, [_vp, C.POINTER(PipelineParams), _i, _i]),
    "epivo_seq_download": (_i, [_vp, _vp, _i, _i]),
    "epivo_seq_process": (_i, [_vp, C.POINTER(PipelineParams), _i, _vp, _vp, _vp]),
    "epivo_seq_stage_ms": (_i, [_vp, _vp, _i]),
    "epivo_seq_set_overlap": (_i, [_vp, _i]),
    "epivo_seq_get_matches": (_i, [_vp, _i, _vp, _vp, _vp, _pi]),
    "epivo_seq_get_masks": (_i, [_vp, _i, _vp, _pi, _vp, _pi]),
    "epivo_seq_cloud": (_i, [_vp, _vp, _i, _i, _vp, _vp, C.c_int64, _vp, C.POINTER(C.c_int64)]),
    "epivo_chain_poses": (_i, [_vp, _vp, _vp, _i, _vp]),
    "epivo_eight_point": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "epivo_fast_detect": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "epivo_lk_track": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i, _i, _i, _d, _d, _vp, _vp, _vp]),
    "epivo_orb_detect_and_compute": (_i, [_vp, _vp, _i, _i, _i, _i, C.c_float, _i, _i, _i, _i, _vp, _vp, _vp]),
    "epivo_orb_level_geometry": (_i, [_i, _i, _i, C.c_float, _i, _vp, _vp, _vp]),
    "epivo_remap": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i, _i, _i, _vp]),
    "epivo_seq_process_points": (_i, [_vp, C.POINTER(PipelineParams), _i, _vp, _vp, _vp, _i, _vp]),
    "epivo_seq_process_frames": (_i, [_vp, C.POINTER(PipelineParams), _i, _vp, _i, _i, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "epivo_seq_get_points": (_i, [_vp, _i, _vp, _vp, _pi]),
    "epivo_seq_bundle_adjust": (_i, [_vp, _i, _vp, _vp, _i, _i, _vp, _d, _vp, _vp, _vp, _vp, _vp, _vp]),
    "epivo_seq_bundle_adjust_stereo": (_i, [_vp, _i, _vp, _vp, _i, _i, _vp, _vp, _d, _vp, _vp, _vp, _vp, _vp, _vp]),
    "epivo_microbench": (_i, [_vp, _i, C.POINTER(_d)]),
}

_lib = None


def load() -> C.CDLL:
    """Load the shared library and bind every declared symbol (raises if any is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EpivoError(ERR_CUDA, f"{LIB_PATH} is missing: run `python epivo_b200/build.py` "
                                   "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
