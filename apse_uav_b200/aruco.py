"""aruco submodule of the drop-in: same names the reference uses from `cv2.aruco` (legacy 4.2 free functions,
aruco_detect.py:191,263,266,267,601) plus the 4.13 object API, all backed by libapse_b200.so."""
from __future__ import annotations

import base64
import zlib
import numpy as np

from ._dict_data import DICTS as _DICTS
from . import _lib
from ._lib import ApseError
from . import engine as _engine

CORNER_REFINE_NONE, CORNER_REFINE_SUBPIX, CORNER_REFINE_CONTOUR, CORNER_REFINE_APRILTAG = 0, 1, 2, 3

for _name, _v in _DICTS.items():
    globals()[_name] = _v[0]
_BY_ID = {v[0]: k for k, v in _DICTS.items()}


class Dictionary:
    """bytesList uint8 (n, nbytes, 4) with rotation-major row memory, markerSize, maxCorrectionBits (as cv2)."""

    def __init__(self, bytesList=None, markerSize=0, maxCorrectionBits=0):
        self.bytesList = np.ascontiguousarray(bytesList, np.uint8) if bytesList is not None else np.zeros((0, 0, 4), np.uint8)
        self.markerSize = int(markerSize)
        self.maxCorrectionBits = int(maxCorrectionBits)

    @property
    def raw(self):
        return self.bytesList.reshape(self.bytesList.shape[0], -1)


def getPredefinedDictionary(dict_id) -> Dictionary:
    if dict_id not in _BY_ID:
        raise ApseError(-5, f"predefined dictionary {dict_id} is not embedded; pass a cv2 Dictionary object instead")
    _, ms, mc, n, blob = _DICTS[_BY_ID[dict_id]]
    raw = np.frombuffer(zlib.decompress(base64.b64decode(blob)), np.uint8).reshape(n, -1)
    nbytes = raw.shape[1] // 4
    return Dictionary(raw.reshape(n, nbytes, 4).copy(), ms, mc)


Dictionary_get = getPredefinedDictionary  # aruco_detect.py:263


class DetectorParameters:
    """Attribute bag with the cv2 4.13 defaults (SURVEY.md Appendix D); aruco_detect.py:190-236 sets 9 of them."""

    def __init__(self):
        self.adaptiveThreshWinSizeMin = 3
        self.adaptiveThreshWinSizeMax = 23
        self.adaptiveThreshWinSizeStep = 10
        self.adaptiveThreshConstant = 7.0
        self.minMarkerPerimeterRate = 0.03
        self.maxMarkerPerimeterRate = 4.0
        self.polygonalApproxAccuracyRate = 0.03
        self.minCornerDistanceRate = 0.05
        self.minDistanceToBorder = 3
        self.minMarkerDistanceRate = 0.125
        self.minGroupDistance = 0.21
        self.cornerRefinementMethod = CORNER_REFINE_NONE
        self.cornerRefinementWinSize = 5
        self.relativeCornerRefinmentWinSize = 0.3
        self.cornerRefinementMaxIterations = 30
        self.cornerRefinementMinAccuracy = 0.1
        self.markerBorderBits = 1
        self.perspectiveRemovePixelPerCell = 4
        self.perspectiveRemoveIgnoredMarginPerCell = 0.13
        self.maxErroneousBitsInBorderRate = 0.35
        self.minOtsuStdDev = 5.0
        self.errorCorrectionRate = 0.6
        self.aprilTagQuadDecimate = 0.0
        self.aprilTagQuadSigma = 0.0
        self.aprilTagMinClusterPixels = 5
        self.aprilTagMaxNmaxima = 10
        self.aprilTagCriticalRad = float(np.float32(10 * np.pi / 180))
        self.aprilTagMaxLineFitMse = 10.0
        self.aprilTagMinWhiteBlackDiff = 5
        self.aprilTagDeglitch = 0
        self.detectInvertedMarker = False
        self.useAruco3Detection = False
        self.minSideLengthCanonicalImg = 32
        self.minMarkerLengthRatioOriginalImg = 0.0


def DetectorParameters_create():  # aruco_detect.py:191
    return DetectorParameters()


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _dict_fields(dictionary):
    bl = np.ascontiguousarray(dictionary.bytesList, np.uint8)
    return bl.reshape(bl.shape[0], -1), int(dictionary.markerSize), int(dictionary.maxCorrectionBits)


def detectMarkers(image, dictionary, corners=None, ids=None, parameters=None, rejectedImgPoints=None,
                  cameraMatrix=None, distCoeff=None):
    """aruco_detect.py:267 -> (corners: tuple of (1,4,2) float32, ids: (N,1) int32 or None, rejected: tuple).
    cameraMatrix / distCoeff are accepted and ignored exactly as OpenCV ignores them outside CORNER_REFINE_CONTOUR."""
    if image is None or np.size(image) == 0:
        raise ApseError(-1, "detectMarkers: empty image")
    shape = image.shape
    e = _engine.default_engine(shape[1], shape[0])
    img = e._u8(image, "detectMarkers")
    if img.dim() == 3:
        if img.shape[2] != 3:
            raise ApseError(-1, "detectMarkers: 1- or 3-channel 8-bit image expected")
        img = e.cvt(img, "bgr2gray")
    raw, ms, mc = _dict_fields(dictionary)
    e.set_dictionary(raw, ms, mc)
    e.set_params(parameters if parameters is not None else DetectorParameters())
    res = e.detect(img, max_markers=_lib.MAX_QUADS, want_rejected=True)   # room for every candidate: cv2 returns them all
    status = int(res["status"][0])
    if status != 0:
        raise ApseError(status, "detectMarkers: work-buffer capacity exceeded for this frame")
    n, nr = int(res["n"][0]), int(res["n_rejected"][0])
    if _is_torch(image):
        c = tuple(res["corners"][0, i].reshape(1, 4, 2) for i in range(n))
        r = tuple(res["rejected"][0, i].reshape(1, 4, 2) for i in range(nr))
        return c, (res["ids"][0, :n].reshape(n, 1) if n else None), r
    cc = res["corners"][0, :n].cpu().numpy()
    rr = res["rejected"][0, :nr].cpu().numpy()
    ii = res["ids"][0, :n].cpu().numpy().reshape(n, 1).astype(np.int32)
    return (tuple(cc[i].reshape(1, 4, 2) for i in range(n)), ii if n else None,
            tuple(rr[i].reshape(1, 4, 2) for i in range(nr)))


def estimatePoseSingleMarkers(corners, markerLength, cameraMatrix, distCoeffs, rvecs=None, tvecs=None, objPoints=None):
    """aruco_detect.py:601 -> (rvecs (N,1,3) float64, tvecs (N,1,3) float64, objPoints (4,1,3) float32)."""
    e = _engine.default_engine()
    if _is_torch(corners):
        c = corners.reshape(-1, 4, 2)
    else:
        c = np.asarray([np.asarray(x, np.float32).reshape(4, 2) for x in corners], np.float32).reshape(-1, 4, 2)
        if c.shape[0] == 0:
            c = np.zeros((0, 4, 2), np.float32)
    n = c.shape[0]
    rv, tv = e.pose(c, float(markerLength), np.asarray(cameraMatrix, np.float64), distCoeffs)
    h = np.float32(np.float32(markerLength) / np.float32(2.0))
    obj = np.array([[-h, h, 0], [h, h, 0], [h, -h, 0], [-h, -h, 0]], np.float32).reshape(4, 1, 3)
    if _is_torch(corners):
        return rv.reshape(n, 1, 3), tv.reshape(n, 1, 3), obj
    return rv.cpu().numpy().reshape(n, 1, 3), tv.cpu().numpy().reshape(n, 1, 3), obj


class ArucoDetector:
    """cv2 4.13 object API: ArucoDetector(dictionary, parameters).detectMarkers(image)."""

    def __init__(self, dictionary=None, detectorParams=None, refineParams=None):
        self.dictionary = dictionary if dictionary is not None else getPredefinedDictionary(globals()["DICT_4X4_50"])
        self.params = detectorParams if detectorParams is not None else DetectorParameters()

    def detectMarkers(self, image, corners=None, ids=None, rejectedImgPoints=None):
        return detectMarkers(image, self.dictionary, parameters=self.params)

    def getDetectorParameters(self):
        return self.params

    def getDictionary(self):
        return self.dictionary


def __getattr__(name):
    """drawAxis / drawDetectedMarkers / generateImageMarker ... pass through to cv2.aruco (visualisation only)."""
    import cv2 as _cv2
    if name == "drawAxis":
        return lambda img, K, D, rvec, tvec, length: _cv2.drawFrameAxes(img, K, D, rvec, tvec, length)
    if name == "drawMarker":
        return lambda d, i, s: _cv2.aruco.generateImageMarker(_cv2.aruco.getPredefinedDictionary(_cv2.aruco.DICT_4X4_50)
                                                              if isinstance(d, Dictionary) else d, i, s)
    return getattr(_cv2.aruco, name)
