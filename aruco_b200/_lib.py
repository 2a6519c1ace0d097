"""ctypes binding of libaruco_b200.so (the C ABI of include/aruco_b200.h).

There is no fallback: importing the detector on a machine where the CUDA library is missing, or creating a
context where no GPU is visible, raises.  `load(require_gpu=False)` exists so CPU-only CI can still check
that the library loads and exports every declared symbol.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# ARUCO_B200_LIB selects an alternative build of the same library (kernel-variant experiments)
LIB_PATH = os.environ.get("ARUCO_B200_LIB") or os.path.join(_HERE, "lib", "libaruco_b200.so")

AB_OK, AB_E_INVALID, AB_E_CUDA, AB_E_CAPACITY, AB_E_NO_DEVICE, AB_E_STATE = 0, -1, -2, -3, -4, -5


class ab_params(C.Structure):
    _fields_ = [("thres_method", C.c_int32), ("thres_param1", C.c_double), ("thres_param2", C.c_double),
                ("corner_method", C.c_int32), ("min_size", C.c_float), ("max_size", C.c_float),
                ("warp_size", C.c_int32), ("border_dist", C.c_float), ("locked_corners", C.c_int32),
                ("erosion", C.c_int32), ("decoder", C.c_int32), ("set_y_perpendicular", C.c_int32),
                ("thres_param1_range", C.c_int32)]


class ab_board_config(C.Structure):
    _fields_ = [("n_markers", C.c_int32), ("info_type", C.c_int32), ("ids", C.c_void_p), ("corners", C.c_void_p)]


class ab_board(C.Structure):
    _fields_ = [("n_markers", C.c_int32), ("has_pose", C.c_int32), ("prob", C.c_float), ("ssize", C.c_float),
                ("rvec", C.c_double * 3), ("tvec", C.c_double * 3)]


class ab_marker(C.Structure):
    _fields_ = [("id", C.c_int32), ("has_pose", C.c_int32), ("corners", C.c_float * 8), ("ssize", C.c_float),
                ("pad_", C.c_float), ("rvec", C.c_double * 3), ("tvec", C.c_double * 3)]


class ab_calib_camera(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("n_views", C.c_int32), ("n_points", C.c_void_p), ("obj", C.c_void_p),
                ("img", C.c_void_p)]


class ab_calib_result(C.Structure):
    _fields_ = [("K", C.c_double * 9), ("D", C.c_double * 5), ("rms", C.c_double), ("iterations", C.c_int32), ("status", C.c_int32)]


DECODER_FN = C.CFUNCTYPE(C.c_int, C.POINTER(C.c_uint8), C.c_int, C.POINTER(C.c_int), C.c_void_p)

# every symbol include/aruco_b200.h declares: name -> (restype, argtypes)
_vp, _i, _sz, _f, _d, _i64 = C.c_void_p, C.c_int, C.c_size_t, C.c_float, C.c_double, C.c_int64
SYMBOLS = {
    "ab_create": (_i, [_i, C.POINTER(_vp)]),
    "ab_destroy": (None, [_vp]),
    "ab_last_error": (C.c_char_p, [_vp]),
    "ab_version": (C.c_char_p, []),
    "ab_default_params": (_i, [C.POINTER(ab_params)]),
    "ab_set_params": (_i, [_vp, C.POINTER(ab_params)]),
    "ab_get_params": (_i, [_vp, C.POINTER(ab_params)]),
    "ab_load_hrm_dictionary": (_i, [_vp, _i, _i, _vp, _i, _f]),
    "ab_set_decoder_callback": (_i, [_vp, DECODER_FN, _vp]),
    "ab_reserve": (_i, [_vp, _i, _i, _i, _i, _i, _i64, _i64]),
    "ab_set_stream": (_i, [_vp, _vp]),
    "ab_detect_batch": (_i, [_vp, _vp, _i, _i, _sz, _sz, _i, _vp, _vp, _f, _vp, _i, _vp]),
    "ab_enqueue_batch_device": (_i, [_vp, _vp, _i, _i, _sz, _sz, _i, _vp, _vp, _f]),
    "ab_fetch_results": (_i, [_vp, _vp, _i, _vp]),
    "ab_detect_batch_bgr": (_i, [_vp, _vp, _i, _i, _sz, _sz, _i, _vp, _vp, _f, _vp, _i, _vp]),
    "ab_get_thresholded": (_i, [_vp, _i, _vp, _sz]),
    "ab_get_grey": (_i, [_vp, _i, _vp, _sz]),
    "ab_get_candidates": (_i, [_vp, _i, _vp, _vp, _vp, _i, C.POINTER(C.c_int32)]),
    "ab_get_canonical": (_i, [_vp, _i, _i, _vp]),
    "ab_get_canonical_size": (_i, [_vp, C.POINTER(C.c_int32)]),
    "ab_get_contour": (_i, [_vp, _i, _i, _vp, _i, C.POINTER(C.c_int32)]),
    "ab_get_counters": (_i, [_vp, _vp, _i]),
    "ab_enable_timing": (_i, [_vp, _i]),
    "ab_get_stage_ms": (_i, [_vp, _vp, _i]),
    "ab_get_kernel_ms": (_i, [_vp, _vp, _i]),
    "ab_threshold": (_i, [_vp, _vp, _i, _i, _sz, _i, _d, _d, _vp, _sz]),
    "ab_detect_rectangles": (_i, [_vp, _vp, _i, _i, _sz, _vp, _i, C.POINTER(C.c_int32)]),
    "ab_warp": (_i, [_vp, _vp, _i, _i, _sz, _vp, _i, _vp]),
    "ab_refine_candidate_lines": (_i, [_vp, _vp, _i, _vp, _vp, _vp]),
    "ab_calculate_extrinsics": (_i, [_vp, _vp, _i, _vp, _vp, _f, _i]),
    "ab_detect_board": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _f, _f, _i, _vp, _vp]),
    "ab_set_board": (_i, [_vp, _vp, _vp, _vp, _f, _f, _i]),
    "ab_get_boards": (_i, [_vp, _i, _vp, _vp, _i]),
    "ab_calibrate_cameras": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "ab_create_marker_image": (_i, [_vp, _i, _i, _i, _vp, _sz, C.POINTER(C.c_int)]),
    "ab_create_board_image": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _i, _vp, _sz, C.POINTER(C.c_int), C.POINTER(C.c_int), _vp, _vp, _i,
                                   C.POINTER(C.c_int)]),
    "ab_create_hrm_marker_image": (_i, [_vp, _i, _vp, _i, _vp, _sz, C.POINTER(C.c_int)]),
    "ab_create_hrm_board_image": (_i, [_vp, _i, _i, _i, _vp, _i, _vp, _sz, C.POINTER(C.c_int), C.POINTER(C.c_int), _vp, _vp, _i,
                                       C.POINTER(C.c_int)]),
    "ab_host_alloc": (_i, [C.POINTER(_vp), _sz]),
    "ab_host_free": (_i, [_vp]),
}

_lib = None


def load():
    """Loads the shared library and binds every declared symbol (raises if any is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("aruco_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "or `make`; there is no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class ArucoError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("aruco_b200 error %d: %s" % (code, msg))
        self.code = code
