"""ctypes binding of libapse_b200.so (include/apse_b200.h).  There is NO CPU fallback: if the CUDA library
is missing or no B200 is visible, every hot call raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("APSE_LIB") or os.path.join(_HERE, "libapse_b200.so")   # APSE_LIB: another build of the library (make decprof)


# candidate quads per frame the library handles (APSE_MAX_QUADS, csrc/common.cuh): no frame can yield more markers or rejects
MAX_QUADS = 4096


# apse_yuv_layout: YUV 4:2:0 layouts of apse_cvt_yuv420_bgr (cv2's single-array form [h*3/2][w])
YUV_LAYOUTS = {"nv12": 0, "nv21": 1, "i420": 2, "yv12": 3}


class ApseError(RuntimeError):
    """Raised for every non-zero apse_status (mirrors cv2.error in the drop-in API)."""

    def __init__(self, code, msg):
        super().__init__(f"apse_b200 error {code}: {msg}")
        self.code = code


class Params(C.Structure):
    """POD mirror of apse_params == cv2.aruco.DetectorParameters (aruco_detect.py:190-236)."""
    _fields_ = [
        ("adaptiveThreshWinSizeMin", C.c_int), ("adaptiveThreshWinSizeMax", C.c_int),
        ("adaptiveThreshWinSizeStep", C.c_int), ("adaptiveThreshConstant", C.c_double),
        ("minMarkerPerimeterRate", C.c_double), ("maxMarkerPerimeterRate", C.c_double),
        ("polygonalApproxAccuracyRate", C.c_double), ("minCornerDistanceRate", C.c_double),
        ("minDistanceToBorder", C.c_int), ("minMarkerDistanceRate", C.c_double), ("minGroupDistance", C.c_float),
        ("cornerRefinementMethod", C.c_int), ("cornerRefinementWinSize", C.c_int),
        ("relativeCornerRefinmentWinSize", C.c_float), ("cornerRefinementMaxIterations", C.c_int),
        ("cornerRefinementMinAccuracy", C.c_double), ("markerBorderBits", C.c_int),
        ("perspectiveRemovePixelPerCell", C.c_int), ("perspectiveRemoveIgnoredMarginPerCell", C.c_double),
        ("maxErroneousBitsInBorderRate", C.c_double), ("minOtsuStdDev", C.c_double),
        ("errorCorrectionRate", C.c_double), ("aprilTagQuadDecimate", C.c_float), ("aprilTagQuadSigma", C.c_float),
        ("aprilTagMinClusterPixels", C.c_int), ("aprilTagMaxNmaxima", C.c_int), ("aprilTagCriticalRad", C.c_float),
        ("aprilTagMaxLineFitMse", C.c_float), ("aprilTagMinWhiteBlackDiff", C.c_int), ("aprilTagDeglitch", C.c_int),
        ("detectInvertedMarker", C.c_int), ("useAruco3Detection", C.c_int), ("minSideLengthCanonicalImg", C.c_int),
        ("minMarkerLengthRatioOriginalImg", C.c_float),
    ]


class Detections(C.Structure):
    _fields_ = [("max_markers", C.c_int), ("corners", C.c_void_p), ("ids", C.c_void_p), ("n_markers", C.c_void_p),
                ("rejected", C.c_void_p), ("n_rejected", C.c_void_p), ("status", C.c_void_p)]


class SeqConfig(C.Structure):
    """apse_seq_config: constants of the reference's frame loop (aruco_detect.py:13-18,36,519-524)."""
    _fields_ = [("start_frame", C.c_int), ("step_frame", C.c_int), ("marker_length_org", C.c_double), ("marker_div", C.c_double),
                ("div", C.c_double), ("width", C.c_int), ("height", C.c_int), ("leds_threshold", C.c_int), ("leds", C.c_int)]


# numpy views of the sequence post-pass structs (apse_seq_job / apse_seq_job_result / apse_seq_row)
SEQ_JOB_DTYPE = [("frame", "<i4"), ("kind", "<i4"), ("rvec", "<f8", 3), ("tvec", "<f8", 3), ("dim", "<f8", 4), ("src", "<f4", 2),
                 ("tgt", "<f4", 2), ("scale", "<f8"), ("led_threshold", "<i4"), ("pad_", "<i4")]
SEQ_RESULT_DTYPE = [("dist_aruco", "<f8"), ("dist_bbox", "<f8"), ("leds", "<i4"), ("valid", "<i4"), ("nearest_px", "<i4", 2),
                    ("outline_px", "<i4", (4, 2))]
OVERLAY_PRIM_DTYPE = [("frame", "<i4"), ("kind", "<i4"), ("x0", "<i4"), ("y0", "<i4"), ("x1", "<i4"), ("y1", "<i4"), ("thickness", "<i4"),
                      ("bgr", "u1", 4)]
SEQ_ROW_DTYPE = [("frame_id", "<i4"), ("detected", "<i4", 4), ("host_fields", "<i4"), ("leds", "<i4"), ("job_led", "<i4"),
                 ("job_dist", "<i4", 3), ("accepted_mask", "<i4"), ("marker_length", "<f8"), ("altitude", "<f8"), ("fov_width", "<f8"),
                 ("fov_height", "<f8"), ("dist_aruco", "<f8", 3), ("dist_bbox", "<f8", 3)]

_vp, _i, _i64, _f = C.c_void_p, C.c_int, C.c_int64, C.c_float
_dp = C.POINTER(C.c_double)
_u8p = C.POINTER(C.c_uint8)

# name -> argtypes (restype is int unless listed in _RESTYPES); must list every symbol of include/apse_b200.h
SIGNATURES = {
    "apse_abi_version": [],
    "apse_params_default": [C.POINTER(Params)],
    "apse_create": [C.POINTER(_vp), _i, _i, _i, _i],
    "apse_destroy": [_vp],
    "apse_last_error": [_vp],
    "apse_set_camera": [_vp, _dp, _dp, _i, _i, _vp],
    "apse_set_lut": [_vp, _u8p, _vp],
    "apse_set_dictionary": [_vp, _u8p, _i, _i, _i, _vp],
    "apse_set_params": [_vp, C.POINTER(Params)],
    "apse_init_undistort_map": [_vp, _dp, _dp, _i, _i, _vp, _vp, _vp],
    "apse_remap": [_vp, _vp, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp],
    "apse_undistort": [_vp, _vp, _i, _i, _i, _dp, _dp, _dp, _vp, _vp],
    "apse_cvt_rgb2lab": [_vp, _vp, _i64, _vp, _vp],
    "apse_cvt_lab2rgb": [_vp, _vp, _i64, _vp, _vp],
    "apse_cvt_bgr2gray": [_vp, _vp, _i64, _vp, _vp],
    "apse_lut": [_vp, _vp, _i64, _i, _vp, _vp, _i, _vp],
    "apse_cvt_yuv420_bgr": [_vp, _vp, _i, _i, _i, _i, _vp, _vp],
    "apse_preprocess": [_vp, _vp, _vp, _vp, _i, _vp],
    "apse_detect": [_vp, _vp, _i, _i, _i, C.POINTER(Detections), _vp],
    "apse_pose": [_vp, _vp, _i, _vp, _f, _dp, _dp, _vp, _vp, _vp],
    "apse_pose_frames": [_vp, _vp, _vp, _i, _i, _vp, _f, _dp, _dp, _vp, _vp, _vp],
    "apse_process_frames": [_vp, _vp, _vp, _i, C.POINTER(Detections), _vp, _f, _vp, _vp, _vp],
    "apse_preprocess_tiles": [_vp, _vp, _vp, _i, _vp],
    "apse_preprocess_tiles_sparse": [_vp, _vp, _vp, _i, _vp],
    "apse_detect_pose_frames": [_vp, _vp, _i, C.POINTER(Detections), _vp, _f, _vp, _vp, _vp],
    "apse_project_points": [_vp, _vp, _i, _vp, _vp, _dp, _dp, _vp, _vp],
    "apse_project_points_multi": [_vp, _vp, _i, _vp, _vp, _vp, _dp, _dp, _vp, _vp],
    "apse_debug_apriltag": [_vp, _vp, _i, _i, _vp, _vp, _vp, _i, C.POINTER(C.c_int64), _vp],
    "apse_patch_sums": [_vp, _vp, _i, _i, _vp, _i, _i, _vp, _vp],
    "apse_adaptive_threshold": [_vp, _vp, _i, _i, _i, _i, C.c_double, _vp, _vp],
    "apse_debug_classic": [_vp, _vp, _i, _i, _vp, _vp, _i, C.POINTER(C.c_int64), _vp],
    "apse_seq_config_default": [C.POINTER(SeqConfig)],
    "apse_py_round": [C.c_double, _i],
    "apse_sequence_scan": [C.POINTER(SeqConfig), _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i, C.POINTER(C.c_int)],
    "apse_sequence_jobs": [_vp, _vp, _i, _vp, _i, _i, _i, _i, _dp, _dp, _vp, _vp],
    "apse_sequence_finish": [_i, _vp, _vp, _i],
    "apse_sequence_scan_chunk": [C.POINTER(SeqConfig), _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i, C.POINTER(C.c_int)],
    "apse_sequence_finish_chunk": [_vp, _i, _vp, _vp, _i],
    "apse_sequence_csv": [_vp, _i, _i, _vp, _i64],
    "apse_debug_sparse": [_vp, _vp, _vp, _i, C.POINTER(C.c_int), _vp],
    "apse_debug_tile_bounds": [_vp, _vp, _i, _vp],
    "apse_debug_tile_extrema": [_vp, _vp, _i, _vp],
    "apse_debug_decode": [_vp, _vp, _i, _i, _vp, _i, _vp, _vp, _vp, _vp],
    "apse_draw_overlay": [_vp, _vp, _i, _i, _i, _vp, _i, _vp],
    "apse_launch_count": [_vp],
    "apse_kernel_count": [],
    "apse_kernel_name": [_i],
    "apse_timing_enable": [_vp, _i],
    "apse_timing_collect": [_vp, _dp, C.POINTER(C.c_int64), _i],
    "apse_timing_trace": [_vp, _dp, _i],
}
_RESTYPES = {"apse_destroy": None, "apse_params_default": None, "apse_seq_config_default": None, "apse_py_round": C.c_double, "apse_sequence_csv": C.c_int64, "apse_last_error": C.c_char_p,
             "apse_launch_count": C.c_int64, "apse_kernel_name": C.c_char_p}

_lib = None


def load():
    """Load the shared library (no CUDA call is made here)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ApseError(-2, f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; "
                                "g.build()'` (nvcc, sm_100a); there is no CPU fallback")
        lib = C.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = _RESTYPES.get(name, C.c_int)
        _lib = lib
    return _lib


def darr(a):
    import numpy as np
    a = np.ascontiguousarray(a, np.float64).ravel()
    return a, a.ctypes.data_as(_dp)


def dist14(D):
    import numpy as np
    k = np.zeros(14, np.float64)
    if D is not None:
        d = np.asarray(D, np.float64).ravel()
        if d.size not in (4, 5, 8, 12, 14):
            raise ApseError(-1, f"distortion vector must have 4, 5, 8, 12 or 14 coefficients, got {d.size}")
        k[:d.size] = d
    return k
