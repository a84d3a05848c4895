"""Engine: one apse_ctx (one GPU, one process) + torch device buffers around the C ABI.

torch is plumbing only (device memory, streams); every computation is a hand-written sm_100a kernel in
libapse_b200.so.  All methods take / return torch CUDA tensors and enqueue on torch's current stream.
"""
from __future__ import annotations

import ctypes as C
import numpy as np

from . import _lib
from ._lib import ApseError, Params, Detections

CORNER_REFINE_NONE, CORNER_REFINE_SUBPIX, CORNER_REFINE_CONTOUR, CORNER_REFINE_APRILTAG = 0, 1, 2, 3


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise ApseError(-2, "no CUDA device visible: apse_uav_b200 has no CPU fallback")
    return torch


def params_from_object(obj) -> Params:
    """Marshal a DetectorParameters-like attribute bag (ours or cv2's) into the POD struct."""
    p = Params()
    _lib.load().apse_params_default(C.byref(p))
    if obj is None:
        return p
    for name, ctype in Params._fields_:
        if hasattr(obj, name):
            v = getattr(obj, name)
            setattr(p, name, int(v) if ctype in (C.c_int,) else float(v))
    return p


class Engine:
    def __init__(self, device: int = 0, max_w: int = 3840, max_h: int = 2160, max_batch: int = 1):
        self.torch = _torch()
        self.lib = _lib.load()
        self.device = device
        self.max_w, self.max_h, self.max_batch = max_w, max_h, max_batch
        h = C.c_void_p()
        rc = self.lib.apse_create(C.byref(h), device, max_w, max_h, max_batch)
        if rc != 0:
            raise ApseError(rc, "apse_create failed (is a B200 visible and is there enough free HBM?)")
        self.h = h
        self.tdev = self.torch.device("cuda", device)
        self._lut_dev = None
        self.K = self.D = None
        self.size = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.apse_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------------------------------ helpers
    def _check(self, rc):
        if rc != 0:
            raise ApseError(rc, self.lib.apse_last_error(self.h).decode())

    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.tdev).cuda_stream)

    def _u8(self, t, name):
        torch = self.torch
        if not isinstance(t, torch.Tensor):
            t = torch.from_numpy(np.ascontiguousarray(t))
        if t.dtype != torch.uint8:
            raise ApseError(-1, f"{name}: 8-bit unsigned image expected, got {t.dtype}")
        return t.to(self.tdev, non_blocking=True).contiguous()

    @property
    def launches(self):
        return int(self.lib.apse_launch_count(self.h))

    def timing(self, on: bool):
        self._check(self.lib.apse_timing_enable(self.h, 1 if on else 0))

    def timing_collect(self, reset=True):
        """{kernel name: (total ms, launches)} accumulated since the last reset (synchronises)."""
        n = self.lib.apse_kernel_count()
        ms = (C.c_double * n)()
        cnt = (C.c_int64 * n)()
        self._check(self.lib.apse_timing_collect(self.h, ms, cnt, 1 if reset else 0))
        return {self.lib.apse_kernel_name(i).decode(): (float(ms[i]), int(cnt[i])) for i in range(n) if cnt[i]}

    # ------------------------------------------------------------------------------------ configuration
    def set_camera(self, K, D, w, h):
        self.K = np.ascontiguousarray(K, np.float64).reshape(3, 3)
        self.D = _lib.dist14(D)
        _, kp = _lib.darr(self.K)
        _, dp = _lib.darr(self.D)
        self._check(self.lib.apse_set_camera(self.h, kp, dp, int(w), int(h), self._stream()))
        self.size = (int(w), int(h))

    def set_lut(self, lut):
        lut = np.ascontiguousarray(lut, np.uint8).ravel()
        if lut.size != 256:
            raise ApseError(-1, "lut must have 256 entries")
        self._check(self.lib.apse_set_lut(self.h, lut.ctypes.data_as(C.POINTER(C.c_uint8)), self._stream()))

    def set_dictionary(self, bytes_list, marker_size, max_correction_bits):
        bl = np.ascontiguousarray(bytes_list, np.uint8)
        n = bl.shape[0]
        self._check(self.lib.apse_set_dictionary(self.h, bl.ctypes.data_as(C.POINTER(C.c_uint8)), n, int(marker_size),
                                                 int(max_correction_bits), self._stream()))

    def set_params(self, params):
        p = params if isinstance(params, Params) else params_from_object(params)
        self._check(self.lib.apse_set_params(self.h, C.byref(p)))

    # -------------------------------------------------------------------------------------------- stage 1
    def init_undistort_map(self, K, D, w, h):
        torch = self.torch
        mx = torch.empty((h, w), dtype=torch.float32, device=self.tdev)
        my = torch.empty((h, w), dtype=torch.float32, device=self.tdev)
        _, kp = _lib.darr(K)
        _, dp = _lib.darr(_lib.dist14(D))
        self._check(self.lib.apse_init_undistort_map(self.h, kp, dp, int(w), int(h), mx.data_ptr(), my.data_ptr(),
                                                     self._stream()))
        return mx, my

    def remap(self, src, mapx, mapy):
        torch = self.torch
        src = self._u8(src, "remap")
        mapx = torch.as_tensor(mapx, dtype=torch.float32, device=self.tdev).contiguous()
        mapy = torch.as_tensor(mapy, dtype=torch.float32, device=self.tdev).contiguous()
        cn = 1 if src.dim() == 2 else src.shape[2]
        dh, dw = mapx.shape
        dst = torch.empty((dh, dw) + (() if src.dim() == 2 else (cn,)), dtype=torch.uint8, device=self.tdev)
        self._check(self.lib.apse_remap(self.h, src.data_ptr(), src.shape[1], src.shape[0], cn, mapx.data_ptr(),
                                        mapy.data_ptr(), dw, dh, dst.data_ptr(), self._stream()))
        return dst

    def undistort(self, src, K, D, newK=None):
        """cv2.undistort(src, K, D, None, newK): FP64 coordinates rounded to Q5 directly, bilinear, BORDER_CONSTANT 0"""
        torch = self.torch
        src = self._u8(src, "undistort")
        cn = 1 if src.dim() == 2 else src.shape[2]
        h, w = src.shape[:2]
        dst = torch.empty_like(src)
        _, kp = _lib.darr(K)
        _, dp = _lib.darr(_lib.dist14(D))
        na, npp = _lib.darr(newK) if newK is not None else (None, None)
        self._check(self.lib.apse_undistort(self.h, src.data_ptr(), w, h, cn, kp, dp, npp, dst.data_ptr(), self._stream()))
        return dst

    def cvt(self, src, kind):
        torch = self.torch
        src = self._u8(src, "cvtColor")
        if src.dim() != 3 or src.shape[2] != 3:
            raise ApseError(-1, "cvtColor: HxWx3 8-bit image expected")
        npx = src.shape[0] * src.shape[1]
        if kind == "bgr2gray":
            dst = torch.empty(src.shape[:2], dtype=torch.uint8, device=self.tdev)
            self._check(self.lib.apse_cvt_bgr2gray(self.h, src.data_ptr(), npx, dst.data_ptr(), self._stream()))
        else:
            dst = torch.empty_like(src)
            fn = self.lib.apse_cvt_rgb2lab if kind == "rgb2lab" else self.lib.apse_cvt_lab2rgb
            self._check(fn(self.h, src.data_ptr(), npx, dst.data_ptr(), self._stream()))
        return dst

    def cvt_yuv420(self, src, layout, out=None, stream=None):
        """cv2.cvtColor(src, COLOR_YUV2BGR_<layout>) for layout nv12 / nv21 / i420 / yv12: src [H*3/2, W] or [B, H*3/2, W] uint8
        (numpy or tensor) -> [.., H, W, 3].  out: a contiguous uint8 CUDA tensor of that shape to write into; stream: torch stream
        of the launch (None = current)."""
        torch = self.torch
        if layout not in _lib.YUV_LAYOUTS:
            raise ApseError(-1, f"cvt_yuv420: unknown layout {layout!r} (one of {', '.join(_lib.YUV_LAYOUTS)})")
        src = self._u8(src, "cvtColor")
        if src.dim() not in (2, 3) or src.shape[-2] % 3:
            raise ApseError(-1, "cvtColor: YUV 4:2:0 source of shape [H*3/2, W] or [B, H*3/2, W] expected (rows divisible by 3)")
        rows, W = src.shape[-2:]
        H = rows * 2 // 3
        B = src.shape[0] if src.dim() == 3 else 1
        shape = tuple(src.shape[:-2]) + (H, W, 3)
        if out is None:
            out = torch.empty(shape, dtype=torch.uint8, device=self.tdev)
        elif tuple(out.shape) != shape or out.dtype != torch.uint8 or not out.is_contiguous() or out.device != self.tdev:
            raise ApseError(-1, f"cvt_yuv420: out must be a contiguous uint8 tensor of shape {shape} on {self.tdev}")
        st = C.c_void_p(stream.cuda_stream) if stream is not None else self._stream()
        self._check(self.lib.apse_cvt_yuv420_bgr(self.h, src.data_ptr(), W, H, B, _lib.YUV_LAYOUTS[layout], out.data_ptr(), st))
        return out

    def lut(self, src, lut):
        """cv2.LUT on an arbitrary (possibly strided channel view) uint8 tensor; returns a contiguous tensor."""
        torch = self.torch
        if not isinstance(src, torch.Tensor):
            src = torch.from_numpy(np.asarray(src))
        src = src.to(self.tdev)
        lut_t = torch.as_tensor(np.ascontiguousarray(lut, np.uint8).ravel(), device=self.tdev)
        if lut_t.numel() != 256:
            raise ApseError(-1, "LUT must have 256 entries")
        dst = torch.empty(src.shape, dtype=torch.uint8, device=self.tdev)
        if src.is_contiguous():
            sstride, base = 1, src
        elif src.dim() >= 1 and self._uniform_stride(src):
            sstride, base = src.stride(-1), src
        else:
            base, sstride = src.contiguous(), 1
        self._check(self.lib.apse_lut(self.h, base.data_ptr(), src.numel(), int(sstride), lut_t.data_ptr(),
                                      dst.data_ptr(), 1, self._stream()))
        return dst

    @staticmethod
    def _uniform_stride(t):
        # channel view of a contiguous interleaved image: element i lives at base + i*stride
        s, expect = t.stride(), t.stride(-1)
        for dim in range(t.dim() - 1, -1, -1):
            if s[dim] != expect:
                return False
            expect *= t.shape[dim]
        return True

    def preprocess(self, bgr, want_bgr=False):
        """aruco_detect.py:250-259 + :592 for a batch: bgr [B,H,W,3] u8 -> (corrected [B,H,W,3] | None, gray [B,H,W])."""
        torch = self.torch
        bgr = self._u8(bgr, "preprocess")
        single = bgr.dim() == 3
        if single:
            bgr = bgr[None]
        B, H, W, _ = bgr.shape
        if self.size != (W, H):
            raise ApseError(-3, f"preprocess: frames are {W}x{H} but the camera was set for {self.size}")
        gray = torch.empty((B, H, W), dtype=torch.uint8, device=self.tdev)
        out = torch.empty_like(bgr) if want_bgr else None
        self._check(self.lib.apse_preprocess(self.h, bgr.data_ptr(), out.data_ptr() if want_bgr else None,
                                             gray.data_ptr(), B, self._stream()))
        if single:
            return (out[0] if want_bgr else None), gray[0]
        return out, gray

    # -------------------------------------------------------------------------------------------- detect
    def alloc_detections(self, B, max_markers, want_rejected=True, pose=False):
        """Output buffers of detect() (and pose_frames()) for B frames; slices along dim 0 can be handed to several
        engines / streams."""
        torch, dev = self.torch, self.tdev
        res = dict(corners=torch.zeros((B, max_markers, 4, 2), dtype=torch.float32, device=dev),
                   ids=torch.full((B, max_markers), -1, dtype=torch.int32, device=dev),
                   n=torch.zeros(B, dtype=torch.int32, device=dev),
                   status=torch.zeros(B, dtype=torch.int32, device=dev))
        if want_rejected:
            res["rejected"] = torch.zeros((B, max_markers, 4, 2), dtype=torch.float32, device=dev)
            res["n_rejected"] = torch.zeros(B, dtype=torch.int32, device=dev)
        if pose:
            res["rvec"] = torch.zeros((B, max_markers, 3), dtype=torch.float64, device=dev)
            res["tvec"] = torch.zeros((B, max_markers, 3), dtype=torch.float64, device=dev)
        return res

    def detect(self, gray, max_markers=256, want_rejected=True, out=None):
        """aruco_detect.py:267 for a batch: gray [B,H,W] u8 -> dict of device tensors (written into `out` if given)."""
        gray = self._u8(gray, "detectMarkers")
        if gray.dim() == 2:
            gray = gray[None]
        B, H, W = gray.shape
        res = out if out is not None else self.alloc_detections(B, max_markers, want_rejected)
        want_rejected = "rejected" in res
        max_markers = res["corners"].shape[1]
        d = Detections(max_markers, res["corners"].data_ptr(), res["ids"].data_ptr(), res["n"].data_ptr(),
                       res["rejected"].data_ptr() if want_rejected else None,
                       res["n_rejected"].data_ptr() if want_rejected else None, res["status"].data_ptr())
        self._check(self.lib.apse_detect(self.h, gray.data_ptr(), W, H, B, C.byref(d), self._stream()))
        return res

    def process_frames(self, bgr, out, marker_length, gray=None):
        """aruco_detect.py:589-601 for a batch in ONE library call (apse_process_frames): preprocess -> detect -> pose.
        `out` is a dict from alloc_detections(..., pose=True); gray [B,H,W] is written if given, else context scratch."""
        torch = self.torch
        bgr = self._u8(bgr, "process_frames")
        B, H, W, _ = bgr.shape
        if self.size != (W, H):
            raise ApseError(-3, f"process_frames: frames are {W}x{H} but the camera was set for {self.size}")
        want_rejected = "rejected" in out
        d = Detections(out["corners"].shape[1], out["corners"].data_ptr(), out["ids"].data_ptr(), out["n"].data_ptr(),
                       out["rejected"].data_ptr() if want_rejected else None,
                       out["n_rejected"].data_ptr() if want_rejected else None, out["status"].data_ptr())
        ml = None
        if isinstance(marker_length, torch.Tensor) or np.ndim(marker_length) > 0:
            ml = torch.as_tensor(marker_length, dtype=torch.float32, device=self.tdev).contiguous()
        self._check(self.lib.apse_process_frames(self.h, bgr.data_ptr(), gray.data_ptr() if gray is not None else None, B,
                                                 C.byref(d), ml.data_ptr() if ml is not None else None,
                                                 float(marker_length) if ml is None else 0.0, out["rvec"].data_ptr(),
                                                 out["tvec"].data_ptr(), self._stream()))
        return out

    def preprocess_tiles(self, bgr, gray, stream=None, sparse=False):
        """first half of process_frames on `stream` (torch stream or None = current): K1t -> gray + tile extrema.
        sparse=True: `gray` is only a work buffer of the detect_pose_frames call that follows (apse_preprocess_tiles_sparse)."""
        B = bgr.shape[0]
        st = C.c_void_p(stream.cuda_stream) if stream is not None else self._stream()
        fn = self.lib.apse_preprocess_tiles_sparse if sparse else self.lib.apse_preprocess_tiles
        self._check(fn(self.h, bgr.data_ptr(), gray.data_ptr(), B, st))

    def detect_pose_frames(self, gray, out, marker_length, stream=None):
        """second half of process_frames on `stream`: candidates -> decode -> pose on the gray batch of preprocess_tiles"""
        torch = self.torch
        B = gray.shape[0]
        want_rejected = "rejected" in out
        d = Detections(out["corners"].shape[1], out["corners"].data_ptr(), out["ids"].data_ptr(), out["n"].data_ptr(),
                       out["rejected"].data_ptr() if want_rejected else None,
                       out["n_rejected"].data_ptr() if want_rejected else None, out["status"].data_ptr())
        ml = None
        if isinstance(marker_length, torch.Tensor) or np.ndim(marker_length) > 0:
            ml = torch.as_tensor(marker_length, dtype=torch.float32, device=self.tdev).contiguous()
        st = C.c_void_p(stream.cuda_stream) if stream is not None else self._stream()
        self._check(self.lib.apse_detect_pose_frames(self.h, gray.data_ptr(), B, C.byref(d), ml.data_ptr() if ml is not None else None,
                                                     float(marker_length) if ml is None else 0.0, out["rvec"].data_ptr(),
                                                     out["tvec"].data_ptr(), st))
        return out

    def debug_apriltag(self, gray, max_quads=512):
        torch = self.torch
        gray = self._u8(gray, "debug_apriltag")
        H, W = gray.shape
        thresh = torch.empty((H, W), dtype=torch.uint8, device=self.tdev)
        labels = torch.empty((H, W), dtype=torch.int32, device=self.tdev)
        quads = torch.zeros((max_quads, 4, 2), dtype=torch.float32, device=self.tdev)
        stats = (C.c_int64 * 4)()
        self._check(self.lib.apse_debug_apriltag(self.h, gray.data_ptr(), W, H, thresh.data_ptr(), labels.data_ptr(),
                                                 quads.data_ptr(), max_quads, stats, self._stream()))
        nq = min(int(stats[3]), max_quads)
        return dict(thresh=thresh, labels=labels, quads=quads[:nq], points=int(stats[0]), clusters=int(stats[1]),
                    fitted=int(stats[2]), n_quads=int(stats[3]))

    def patch_sums(self, gray, pts, half=2):
        """Sums of gray[f][y-half:y+half+1, x-half:x+half+1] (numpy slicing rules) for pts = [(f, x, y), ...] -> int64 numpy."""
        torch = self.torch
        gray = self._u8(gray, "patch_sums")
        if gray.dim() == 2:
            gray = gray[None]
        _, H, W = gray.shape
        p = torch.as_tensor(np.asarray(pts, np.int32).reshape(-1, 3), device=self.tdev).contiguous()
        n = p.shape[0]
        out = torch.zeros(n, dtype=torch.int64, device=self.tdev)
        if n:
            self._check(self.lib.apse_patch_sums(self.h, gray.data_ptr(), W, H, p.data_ptr(), n, int(half), out.data_ptr(), self._stream()))
        return out.cpu().numpy()

    def adaptive_threshold(self, gray, win, c):
        """cv2.adaptiveThreshold(gray, 255, ADAPTIVE_THRESH_MEAN_C, THRESH_BINARY_INV, win, c) on [H,W] or [B,H,W]."""
        torch = self.torch
        gray = self._u8(gray, "adaptiveThreshold")
        single = gray.dim() == 2
        g = gray[None] if single else gray
        B, H, W = g.shape
        out = torch.empty_like(g)
        self._check(self.lib.apse_adaptive_threshold(self.h, g.data_ptr(), W, H, B, int(win), float(c), out.data_ptr(), self._stream()))
        return out[0] if single else out

    def debug_classic(self, gray, max_quads=4096):
        """Raw candidate quads of the classic path for one frame, in the dependency's candidate order."""
        torch = self.torch
        gray = self._u8(gray, "debug_classic")
        H, W = gray.shape
        quads = torch.zeros((max_quads, 4, 2), dtype=torch.float32, device=self.tdev)
        order = torch.zeros(max_quads, dtype=torch.int32, device=self.tdev)
        stats = (C.c_int64 * 4)()
        self._check(self.lib.apse_debug_classic(self.h, gray.data_ptr(), W, H, quads.data_ptr(), order.data_ptr(), max_quads,
                                                stats, self._stream()))
        n = min(int(stats[0]), max_quads)
        res = torch.empty((n, 4, 2), dtype=torch.float32, device=self.tdev)
        res[order[:n].long()] = quads[:n]
        return res

    # ---------------------------------------------------------------------------------------------- pose
    def _cam(self, K, D):
        K = self.K if K is None else np.ascontiguousarray(K, np.float64)
        D = self.D if D is None else _lib.dist14(D)
        if K is None:
            raise ApseError(-3, "camera matrix not set")
        return _lib.darr(K), _lib.darr(_lib.dist14(D) if np.size(D) != 14 else D)

    def pose(self, corners, marker_length, K=None, D=None):
        torch = self.torch
        c = torch.as_tensor(corners, dtype=torch.float32, device=self.tdev).reshape(-1, 4, 2).contiguous()
        n = c.shape[0]
        rv = torch.zeros((n, 3), dtype=torch.float64, device=self.tdev)
        tv = torch.zeros((n, 3), dtype=torch.float64, device=self.tdev)
        if n == 0:
            return rv, tv
        (ka, kp), (da, dp) = self._cam(K, D)
        ml = None
        if isinstance(marker_length, torch.Tensor) or np.ndim(marker_length) > 0:
            ml = torch.as_tensor(marker_length, dtype=torch.float32, device=self.tdev).contiguous()
        self._check(self.lib.apse_pose(self.h, c.data_ptr(), n, ml.data_ptr() if ml is not None else None,
                                       float(marker_length) if ml is None else 0.0, kp, dp, rv.data_ptr(), tv.data_ptr(),
                                       self._stream()))
        return rv, tv

    def pose_frames(self, corners, n_markers, marker_length, K=None, D=None, out=None):
        torch = self.torch
        B, M = corners.shape[:2]
        rv = out[0] if out is not None else torch.zeros((B, M, 3), dtype=torch.float64, device=self.tdev)
        tv = out[1] if out is not None else torch.zeros((B, M, 3), dtype=torch.float64, device=self.tdev)
        (ka, kp), (da, dp) = self._cam(K, D)
        ml = None
        if isinstance(marker_length, torch.Tensor) or np.ndim(marker_length) > 0:
            ml = torch.as_tensor(marker_length, dtype=torch.float32, device=self.tdev).contiguous()
        self._check(self.lib.apse_pose_frames(self.h, corners.data_ptr(), n_markers.data_ptr(), B, M,
                                              ml.data_ptr() if ml is not None else None,
                                              float(marker_length) if ml is None else 0.0, kp, dp, rv.data_ptr(),
                                              tv.data_ptr(), self._stream()))
        return rv, tv

    def project_points(self, obj, rvec, tvec, K=None, D=None):
        torch = self.torch
        o = torch.as_tensor(np.asarray(obj, np.float64).reshape(-1, 3) if not isinstance(obj, torch.Tensor) else obj,
                            dtype=torch.float64, device=self.tdev).reshape(-1, 3).contiguous()
        r = torch.as_tensor(np.asarray(rvec, np.float64).ravel() if not isinstance(rvec, torch.Tensor) else rvec,
                            dtype=torch.float64, device=self.tdev).reshape(3).contiguous()
        t = torch.as_tensor(np.asarray(tvec, np.float64).ravel() if not isinstance(tvec, torch.Tensor) else tvec,
                            dtype=torch.float64, device=self.tdev).reshape(3).contiguous()
        img = torch.empty((o.shape[0], 2), dtype=torch.float64, device=self.tdev)
        (ka, kp), (da, dp) = self._cam(K, D)
        self._check(self.lib.apse_project_points(self.h, o.data_ptr(), o.shape[0], r.data_ptr(), t.data_ptr(), kp, dp,
                                                 img.data_ptr(), self._stream()))
        return img

    def project_points_multi(self, obj, pose_idx, rvecs, tvecs, K=None, D=None):
        torch = self.torch
        o = torch.as_tensor(obj, dtype=torch.float64, device=self.tdev).reshape(-1, 3).contiguous()
        idx = torch.as_tensor(pose_idx, dtype=torch.int32, device=self.tdev).contiguous()
        r = torch.as_tensor(rvecs, dtype=torch.float64, device=self.tdev).reshape(-1, 3).contiguous()
        t = torch.as_tensor(tvecs, dtype=torch.float64, device=self.tdev).reshape(-1, 3).contiguous()
        img = torch.empty((o.shape[0], 2), dtype=torch.float64, device=self.tdev)
        (ka, kp), (da, dp) = self._cam(K, D)
        self._check(self.lib.apse_project_points_multi(self.h, o.data_ptr(), o.shape[0], idx.data_ptr(), r.data_ptr(),
                                                       t.data_ptr(), kp, dp, img.data_ptr(), self._stream()))
        return img


_default = {}


def default_engine(w=3840, h=2160, device=None) -> Engine:
    """Process-wide single-frame engine used by the cv2-shaped drop-in functions (grown on demand)."""
    torch = _torch()
    if device is None:
        device = torch.cuda.current_device()
    e = _default.get(device)
    if e is None or e.max_w < w or e.max_h < h:
        if e is not None:
            e.close()
        e = Engine(device, max(w, 64), max(h, 64), 1)
        _default[device] = e
    return e
