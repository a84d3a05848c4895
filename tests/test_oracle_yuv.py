"""CPU: the reference restatement of YUV 4:2:0 -> BGR (tools/yuv_reference.py, what tests/test_gpu_yuv.py checks the kernel
against besides cv2) pinned to cv2.cvtColor for the four layouts the library accepts, on every (Y, U, V) triple and on frame
sizes with odd h/2 and widths that are no multiple of 16."""
import os

import numpy as np
import pytest

from conftest import needs_cv2

LAYOUTS = ("nv12", "nv21", "i420", "yv12")
SIZES = ((3840, 2160), (1920, 1082), (66, 6), (2, 2))


def _codes(cv2):
    return {"nv12": cv2.COLOR_YUV2BGR_NV12, "nv21": cv2.COLOR_YUV2BGR_NV21, "i420": cv2.COLOR_YUV2BGR_I420,
            "yv12": cv2.COLOR_YUV2BGR_YV12}


@pytest.fixture(params=[1, os.cpu_count() or 1], ids=["1thread", "allthreads"])
def cv2_threads(request):
    import cv2
    old = cv2.getNumThreads()
    cv2.setNumThreads(request.param)
    yield cv2
    cv2.setNumThreads(old)


@needs_cv2
@pytest.mark.parametrize("layout", LAYOUTS)
def test_all_triples(cv2_threads, layout):
    """2^24 (Y, U, V) triples in one 4096 x 4096 frame: 0 differing bytes"""
    from tools import synth, yuv_reference
    cv2 = cv2_threads
    yuv = synth.yuv420_all_triples(layout)
    assert np.array_equal(yuv_reference.yuv420_to_bgr(yuv, layout), cv2.cvtColor(yuv, _codes(cv2)[layout]))


@needs_cv2
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("size", SIZES, ids=[f"{w}x{h}" for w, h in SIZES])
def test_frame_sizes(cv2_threads, layout, size):
    from tools import yuv_reference
    cv2 = cv2_threads
    w, h = size
    yuv = np.random.default_rng(w * 7 + h).integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)
    assert np.array_equal(yuv_reference.yuv420_to_bgr(yuv, layout), cv2.cvtColor(yuv, _codes(cv2)[layout]))


@needs_cv2
@pytest.mark.parametrize("layout", LAYOUTS)
def test_layouts_from_bgr(layout):
    """tools.synth.bgr_to_yuv420 derives NV12 / NV21 / YV12 from cv2's BGR -> I420 planes: every layout decodes to the I420 result"""
    import cv2
    from tools import synth
    bgr = np.random.default_rng(3).integers(0, 256, (1082, 1920, 3), dtype=np.uint8)
    want = cv2.cvtColor(synth.bgr_to_yuv420(bgr, "i420"), cv2.COLOR_YUV2BGR_I420)
    assert np.array_equal(cv2.cvtColor(synth.bgr_to_yuv420(bgr, layout), _codes(cv2)[layout]), want)
