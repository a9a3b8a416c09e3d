"""ctypes loader of libcvgraft.so (the C ABI in include/cvgraft.h).  There is no fallback: a missing
library or a missing GPU is an error the caller sees."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("CVGRAFT_SO") or os.path.join(HERE, "libcvgraft.so")      # CVGRAFT_SO: A/B builds of experiments


class RansacParams(C.Structure):
    _fields_ = [("size", C.c_uint32), ("flags", C.c_uint32), ("threshold", C.c_double),
                ("confidence", C.c_double), ("max_iters", C.c_int32), ("reserved", C.c_int32)]


class AffineParams(C.Structure):
    _fields_ = [("size", C.c_uint32), ("flags", C.c_uint32), ("threshold", C.c_double),
                ("confidence", C.c_double), ("max_iters", C.c_int32), ("refine_iters", C.c_int32)]


class DetectParams(C.Structure):
    _fields_ = [("size", C.c_uint32), ("ratio", C.c_float), ("min_inliers", C.c_int32), ("det_lo", C.c_float),
                ("det_hi", C.c_float), ("reserved", C.c_int32), ("ransac", RansacParams),
                ("method", C.c_int32), ("refine_iters", C.c_int32)]


class PairResult(C.Structure):
    _fields_ = [("status", C.c_int32), ("n_good", C.c_int32), ("n_inliers", C.c_int32),
                ("ransac_iters", C.c_int32), ("H", C.c_double * 9), ("det", C.c_double)]


# every symbol include/cvgraft.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "cvg_ransac_params_default": (None, [C.POINTER(RansacParams)]),
    "cvg_detect_params_default": (None, [C.POINTER(DetectParams)]),
    "cvg_affine_params_default": (None, [C.POINTER(AffineParams)]),
    "cvg_create": (C.c_int, [C.POINTER(_P), C.c_int, C.c_uint]),
    "cvg_create_multi": (C.c_int, [C.POINTER(_P), C.POINTER(C.c_int), C.c_int, C.c_uint]),
    "cvg_num_devices": (C.c_int, [_P]),
    "cvg_exchange_kind": (C.c_char_p, [_P]),
    "cvg_set_lanes": (C.c_int, [_P, C.c_int]),
    "cvg_detect_scenes_submit": (C.c_int, [_P, _P, _P, _P, C.POINTER(DetectParams), _P, _P, _P, C.POINTER(_P)]),
    "cvg_job_wait": (C.c_int, [_P, _P]),
    "cvg_match_knn2_sharded": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_float, _P, _P, _P]),
    "cvg_find_homography_sharded": (C.c_int, [_P, _P, _P, C.c_int, C.POINTER(RansacParams), _P, _P, C.POINTER(C.c_int), _P, _P]),
    "cvg_last_exchange": (C.c_int, [_P, C.POINTER(C.c_int), C.POINTER(C.c_float)]),
    "cvg_last_match_guard_rows": (C.c_int, [_P]),
    "cvg_destroy": (None, [_P]),
    "cvg_last_error": (C.c_char_p, []),
    "cvg_host_alloc": (C.c_void_p, [C.c_size_t]),
    "cvg_host_free": (None, [_P]),
    "cvg_version": (C.c_char_p, []),
    "cvg_models_upload": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.POINTER(_P)]),
    "cvg_models_free": (None, [_P, _P]),
    "cvg_models_num_views": (C.c_int, [_P]),
    "cvg_models_num_rows": (C.c_int, [_P]),
    "cvg_match_knn2": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_float, _P, _P, _P]),
    "cvg_match_knn2_raw": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_float, _P, _P, _P]),
    "cvg_match_cross_check": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, _P]),
    "cvg_match_cross_check_raw": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, _P]),
    "cvg_find_homography": (C.c_int, [_P, _P, _P, C.c_int, C.POINTER(RansacParams), _P, _P, C.POINTER(C.c_int), _P]),
    "cvg_find_homography_batch": (C.c_int, [_P, _P, _P, _P, C.c_int, C.POINTER(RansacParams), _P, _P, _P, _P, _P]),
    "cvg_estimate_affine2d": (C.c_int, [_P, _P, _P, C.c_int, C.POINTER(AffineParams), _P, _P, C.POINTER(C.c_int)]),
    "cvg_estimate_affine2d_batch": (C.c_int, [_P, _P, _P, _P, C.c_int, C.POINTER(AffineParams), _P, _P, _P, _P]),
    "cvg_estimate_affine_partial2d": (C.c_int, [_P, _P, _P, C.c_int, C.POINTER(AffineParams), _P, _P, C.POINTER(C.c_int)]),
    "cvg_estimate_affine_partial2d_batch": (C.c_int, [_P, _P, _P, _P, C.c_int, C.POINTER(AffineParams), _P, _P, _P, _P]),
    "cvg_detect_pairs": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_float, C.POINTER(DetectParams), _P, _P, _P]),
    "cvg_scenes_upload": (C.c_int, [_P, _P, _P, _P, C.c_int, C.POINTER(_P)]),
    "cvg_scenes_free": (None, [_P, _P]),
    "cvg_scenes_upload_async": (C.c_int, [_P, _P, _P, _P, C.c_int, C.POINTER(_P)]),
    "cvg_scenes_wait": (C.c_int, [_P, _P]),
    "cvg_scenes_upload_u8_async": (C.c_int, [_P, _P, _P, _P, C.c_int, C.POINTER(_P)]),
    "cvg_detect_scenes": (C.c_int, [_P, _P, _P, _P, C.POINTER(DetectParams), _P]),
    "cvg_detect_scenes_inliers": (C.c_int, [_P, _P, _P, _P, C.POINTER(DetectParams), _P, _P, _P]),
    "cvg_dev_match_top2": (C.c_int, [_P, _P, _P, C.c_int, _P, C.c_int, C.c_int32, _P, _P]),
    "cvg_dev_merge_top2": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_float, _P, _P, _P]),
    "cvg_last_match_path": (C.c_int, [_P]),
    "cvg_last_match_fallback_rows": (C.c_int, [_P]),
    "cvg_last_sampler_serial_sets": (C.c_int, [_P]),
    "cvg_stream": (C.c_void_p, [_P]),
    "cvg_launch_count": (C.c_int64, [_P]),
    "cvg_set_timing": (C.c_int, [_P, C.c_int]),
    "cvg_last_timing": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "cvg_last_hyp_stats": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_uint64)]),
    "cvg_last_score_ms": (C.c_int, [_P, C.POINTER(C.c_float)]),
    "cvg_selftest": (C.c_int, [_P, C.c_int, C.POINTER(C.c_uint64)]),
    "cvg_trace_dump": (None, []),
    "cvg_debug_words": (C.c_int, [_P, C.POINTER(C.c_int), C.c_int]),
    "cvg_device_reset": (C.c_int, [C.c_int]),
}

_lib = None


def load():
    """Load libcvgraft.so; raises if it has not been built (python -m ..._b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError(f"{SO_PATH} is missing: build it with "
                               "`python -m computervision_objectdetection_featurematching_b200.build` "
                               "(libcvgraft has no CPU fallback)")
        lib = C.CDLL(SO_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
