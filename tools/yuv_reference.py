"""CPU restatement of cv2.cvtColor(yuv, COLOR_YUV2BGR_NV12 / _NV21 / _I420 / _YV12) for the tests (numpy, independent of the
GPU kernel and of cv2): BT.601 limited range in 20-bit fixed point, as OpenCV's YUV420sp2RGB / YUV420p2RGB converters compute
it; the four pixels of a 2x2 block share one (U, V) pair.  Pinned to cv2 by tests/test_oracle_yuv.py."""
from __future__ import annotations

import numpy as np

LAYOUTS = ("nv12", "nv21", "i420", "yv12")


def yuv420_planes(yuv: np.ndarray, layout: str):
    """[h*3/2, w] single-array frame -> (Y [h, w], U [h/2, w/2], V [h/2, w/2]).  Planar chroma planes are contiguous
    (h/2)*(w/2)-byte runs: byte offsets, not row offsets (with odd h/2 a plane starts in the middle of a w-wide row)."""
    if layout not in LAYOUTS:
        raise ValueError(f"unknown YUV 4:2:0 layout {layout!r}")
    yuv = np.ascontiguousarray(yuv, np.uint8)
    rows, w = yuv.shape
    h = rows * 2 // 3
    flat = yuv.reshape(-1)
    ysz, q = h * w, (h // 2) * (w // 2)
    Y = flat[:ysz].reshape(h, w)
    if layout in ("nv12", "nv21"):
        c = flat[ysz:].reshape(h // 2, w // 2, 2)
        a, b = c[..., 0], c[..., 1]
        return (Y, a, b) if layout == "nv12" else (Y, b, a)
    a, b = flat[ysz:ysz + q].reshape(h // 2, w // 2), flat[ysz + q:ysz + 2 * q].reshape(h // 2, w // 2)
    return (Y, a, b) if layout == "i420" else (Y, b, a)


def yuv420_to_bgr(yuv: np.ndarray, layout: str) -> np.ndarray:
    """cv2.cvtColor(yuv, COLOR_YUV2BGR_<layout>) for one [h*3/2, w] uint8 frame -> [h, w, 3] uint8"""
    Y, U, V = yuv420_planes(yuv, layout)
    uu, vv, half = U.astype(np.int32) - 128, V.astype(np.int32) - 128, np.int32(1 << 19)
    terms = (half + 2116026 * uu, half - 852492 * vv - 409993 * uu, half + 1673527 * vv)   # B, G, R: |sum| < 5.7e8 fits int32
    y = np.maximum(Y.astype(np.int32) - 16, 0) * np.int32(1220542)
    out = np.empty(Y.shape + (3,), np.uint8)
    for ch, t in enumerate(terms):
        full = np.repeat(np.repeat(t, 2, axis=0), 2, axis=1)
        out[..., ch] = np.clip((y + full) >> 20, 0, 255)   # >> on int32 is an arithmetic shift: it floors, as in cv2
    return out
