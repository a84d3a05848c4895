"""apse_uav_b200 -- drop-in, B200-native (sm_100a CUDA) replacement for the cv2 calls on the hot path of
vision-agh/apse_uav's aruco_detect.py.  Usage = an import swap at aruco_detect.py:1-2:

    import apse_uav_b200 as cv2
    from apse_uav_b200 import aruco

Hot functions (re-implemented as hand-written CUDA kernels behind libapse_b200.so, same signatures and
return conventions as cv2): initUndistortRectifyMap (:568), remap (:252), cvtColor for COLOR_RGB2LAB /
COLOR_LAB2RGB / COLOR_BGR2GRAY (:255,257,592) and for decoder output in YUV 4:2:0 (COLOR_YUV2BGR_NV12 / _NV21 / _I420 /
_IYUV / _YV12), LUT (:256), undistort, projectPoints (:344,377,424,468),
aruco.detectMarkers (:267), aruco.estimatePoseSingleMarkers (:601).  Everything else the script touches
(VideoCapture, imread, imshow, putText, ...) is passed through to the installed cv2 when it is importable.

numpy in -> numpy out (host<->device copies inside the call); torch CUDA tensors in -> torch CUDA tensors out.
There is no CPU fallback: without the built library or without a GPU every hot call raises ApseError.
"""
from __future__ import annotations

import numpy as np

from ._lib import ApseError, load as _load_library, LIB_PATH  # noqa: F401
from . import engine as _engine
from .engine import Engine, default_engine  # noqa: F401
from . import aruco  # noqa: F401
from .pipeline import Pipeline  # noqa: F401
from . import postpass, shard  # noqa: F401

error = ApseError

# constants (values identical to cv2's)
INTER_NEAREST, INTER_LINEAR = 0, 1
BORDER_CONSTANT = 0
COLOR_BGR2GRAY, COLOR_RGB2GRAY = 6, 7
COLOR_BGR2LAB, COLOR_RGB2LAB, COLOR_LAB2BGR, COLOR_LAB2RGB = 44, 45, 56, 57
COLOR_BGR2Lab, COLOR_RGB2Lab, COLOR_Lab2BGR, COLOR_Lab2RGB = 44, 45, 56, 57
COLOR_YUV2BGR_NV12, COLOR_YUV2BGR_NV21, COLOR_YUV2BGR_YV12, COLOR_YUV2BGR_I420, COLOR_YUV2BGR_IYUV = 91, 93, 99, 101, 101
CV_32FC1, CV_16SC2 = 5, 11
_YUV_CODES = {COLOR_YUV2BGR_NV12: "nv12", COLOR_YUV2BGR_NV21: "nv21", COLOR_YUV2BGR_YV12: "yv12", COLOR_YUV2BGR_I420: "i420"}


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _out(t, like):
    return t if _is_torch(like) else t.cpu().numpy()


def initUndistortRectifyMap(cameraMatrix, distCoeffs, R, newCameraMatrix, size, m1type, map1=None, map2=None):
    """aruco_detect.py:568.  Only R = None/identity, newCameraMatrix == cameraMatrix and CV_32FC1 maps (the
    reference's call) are implemented."""
    K = np.asarray(cameraMatrix, np.float64).reshape(3, 3)
    if R is not None and not np.allclose(np.asarray(R, np.float64).reshape(3, 3), np.eye(3)):
        raise ApseError(-5, "initUndistortRectifyMap: rectification rotation is not supported")
    if newCameraMatrix is not None and not np.array_equal(np.asarray(newCameraMatrix, np.float64).reshape(3, 3), K):
        raise ApseError(-5, "initUndistortRectifyMap: newCameraMatrix must equal cameraMatrix")
    if m1type != CV_32FC1:
        raise ApseError(-5, "initUndistortRectifyMap: only m1type=CV_32FC1 (5) is supported")
    w, h = int(size[0]), int(size[1])
    e = default_engine(w, h)
    mx, my = e.init_undistort_map(K, distCoeffs, w, h)
    return mx.cpu().numpy(), my.cpu().numpy()


def remap(src, map1, map2, interpolation, dst=None, borderMode=BORDER_CONSTANT, borderValue=0):
    """aruco_detect.py:252 (INTER_LINEAR, BORDER_CONSTANT 0, float32 maps)."""
    if interpolation != INTER_LINEAR:
        raise ApseError(-5, "remap: only INTER_LINEAR is supported")
    if borderMode != BORDER_CONSTANT or np.any(np.asarray(borderValue) != 0):
        raise ApseError(-5, "remap: only BORDER_CONSTANT with value 0 is supported")
    if map2 is None or np.ndim(map1) != 2:
        raise ApseError(-5, "remap: two CV_32FC1 maps expected")
    e = default_engine(max(src.shape[1], map1.shape[1]), max(src.shape[0], map1.shape[0]))
    return _out(e.remap(src, map1, map2), src)


def cvtColor(src, code, dst=None, dstCn=0):
    """aruco_detect.py:255,257,592, and YUV 4:2:0 [H*3/2, W] -> BGR [H, W, 3] (COLOR_YUV2BGR_NV12 / _NV21 / _I420 / _YV12)."""
    if code in _YUV_CODES:
        e = default_engine(src.shape[-1], src.shape[-2] * 2 // 3)   # sized for the output frame, not the source's rows
        return _out(e.cvt_yuv420(src, _YUV_CODES[code]), src)
    kinds = {COLOR_RGB2LAB: "rgb2lab", COLOR_LAB2RGB: "lab2rgb", COLOR_BGR2GRAY: "bgr2gray"}
    if code not in kinds:
        raise ApseError(-5, f"cvtColor: conversion code {code} is not on the hot path (RGB2LAB, LAB2RGB, BGR2GRAY, YUV2BGR_NV12 / NV21 / I420 / YV12 only)")
    e = default_engine(src.shape[1], src.shape[0])
    return _out(e.cvt(src, kinds[code]), src)


def LUT(src, lut, dst=None):
    """aruco_detect.py:256 (accepts the strided lab[...,0] view)."""
    shape = src.shape
    e = default_engine(max(shape[1], 64) if len(shape) > 1 else 64, max(shape[0], 64))
    if _is_torch(src):
        return e.lut(src, lut)
    import torch
    t = torch.from_numpy(np.ascontiguousarray(src))
    return e.lut(t, lut).cpu().numpy()


def undistort(src, cameraMatrix, distCoeffs, dst=None, newCameraMatrix=None):
    """cv2.undistort (dcnn/scripts/tests/visualize_uav.py:62): bit-exact with the dependency, which rounds the FP64 source
    coordinate to the Q5 grid directly -- NOT the same pixels as initUndistortRectifyMap(CV_32FC1) + remap
    (aruco_detect.py:568,252), which go through float32 maps (SURVEY.md A.1); both variants are provided."""
    h, w = src.shape[:2]
    e = default_engine(w, h)
    return _out(e.undistort(src, cameraMatrix, distCoeffs, newCameraMatrix), src)


def projectPoints(objectPoints, rvec, tvec, cameraMatrix, distCoeffs, imagePoints=None, jacobian=None, aspectRatio=0):
    """aruco_detect.py:344,377,424,468 -> (imagePoints (n,1,2) float64, None).  The Jacobian output is not
    produced (the reference discards it)."""
    e = default_engine()
    img = e.project_points(objectPoints, rvec, tvec, np.asarray(cameraMatrix, np.float64), distCoeffs)
    return img.cpu().numpy().reshape(-1, 1, 2), None


def __getattr__(name):
    """Non-hot names (VideoCapture, imread, imshow, putText, circle, FONT_*, ...) pass through to cv2."""
    try:
        import cv2 as _cv2
    except ImportError as exc:  # pragma: no cover
        raise AttributeError(f"apse_uav_b200 has no attribute {name!r} and cv2 is not importable") from exc
    return getattr(_cv2, name)
