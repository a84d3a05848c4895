"""CPU: the frame geometries that send the preprocess stage down its edge-size code paths, and the frames that test them.

apse_preprocess_ex and apse_preprocess_sparse (csrc/preprocess.cu) choose a kernel from the frame size and the alignment of the
buffers.  dense_kernel() and sparse_kernel() restate those choices; GEOMETRIES lists frame sizes, each with the kernels it is
meant to reach, and test_geometry_table_reaches_its_kernels keeps the table honest if a tile constant or a condition changes.
tests/test_gpu_batch_geometry.py runs every entry on the GPU against the oracle.

tools.synth.make_edge_frame puts markers across the edges of the last CTA column and row; here the oracle chain must find
markers there, so that the GPU comparison covers detections in the partial CTAs and not only their pixels.
"""
import numpy as np
import pytest
from conftest import needs_cv2

P2_TW, P2_TH = 64, 24           # output pixels of one k_preprocess_tma CTA (csrc/preprocess.cu)
W4K, H4K = 3840, 2160


def tma_ok(w, h, bgr_offset=0):
    """k_preprocess_tma can take the frame: bulk tensor copies need 16-byte row strides and a 16-byte aligned source, a thread owns
    4 rows, and the frame holds at least one whole CTA"""
    return w % 4 == 0 and h % 4 == 0 and (w * 3) % 16 == 0 and w >= P2_TW and h >= P2_TH and bgr_offset % 16 == 0


def full_ctas(w, h):
    """every thread of every CTA has pixels (the FULL template argument)"""
    return w % P2_TW == 0 and h % P2_TH == 0


def dense_kernel(w, h, want_bgr=False, bgr_offset=0):
    """the kernel apse_preprocess_ex launches"""
    if not tma_ok(w, h, bgr_offset):
        return "fused"
    if want_bgr:
        return "tma<true,64,0>"
    if w == 3840:
        return "tma<false,48,3840,true>" if h % P2_TH == 0 else "tma<false,48,3840>"
    return "tma<false,64,0>"


def sparse_kernel(w, h, batch=1, bgr_offset=0, gray_offset=0):
    """the bounds pass apse_preprocess_sparse launches, or None when the sparse evaluation falls back to the dense kernel
    (k_sparse_flags takes 8 tiles per thread: w % 32 == 0; k_sparse_exact stores 4 gray bytes at once: 4-byte aligned gray)"""
    if not (tma_ok(w, h, bgr_offset) and batch <= 64 and w % 32 == 0 and gray_offset % 4 == 0):
        return None
    return "bounds<false,40,3840,true,1,3>" if w == 3840 and h % P2_TH == 0 else "bounds<false,48,0,false,1>"


# (w, h) -> (dense kernel, bounds pass of the sparse evaluation or None, every CTA full)
GEOMETRIES = {
    (3840, 2160): ("tma<false,48,3840,true>", "bounds<false,40,3840,true,1,3>", True),   # the footage: control
    (3840, 2152): ("tma<false,48,3840>", "bounds<false,48,0,false,1>", False),          # 4K width, partial last CTA row
    (1952, 1100): ("tma<false,64,0>", "bounds<false,48,0,false,1>", False),             # w % 64 = 32, h % 24 = 20, partial SFL_ROWS group
    (1936, 1096): ("tma<false,64,0>", None, False),                                     # w % 32 = 16: sparse falls back
    (1920, 1082): ("fused", None, False),                                               # h % 4 = 2: no TMA, no tile extrema
    (64, 24): ("tma<false,64,0>", "bounds<false,48,0,false,1>", True),                  # the TMA minimum: one CTA
    (80, 44): ("tma<false,64,0>", None, False),                                         # one full and one partial CTA per row
    (60, 40): ("fused", None, False),                                                   # narrower than a CTA
}
GEOMETRY_IDS = [f"{w}x{h}" for w, h in GEOMETRIES]


def scaled_camera(K, w):
    """the camera matrix of a frame `w` px wide taken with the 4K test lens (the same distortion)"""
    Ks = np.array(K, np.float64).copy()
    Ks[:2] *= w / W4K
    return Ks


def last_cta_edges(w, h):
    """left edge of the last CTA column and top edge of the last CTA row"""
    return w - (w % P2_TW or P2_TW), h - (h % P2_TH or P2_TH)


def test_geometry_table_reaches_its_kernels():
    for (w, h), (dense, sparse, full) in GEOMETRIES.items():
        assert dense_kernel(w, h) == dense, (w, h)
        assert sparse_kernel(w, h) == sparse, (w, h)
        assert full_ctas(w, h) == full, (w, h)
        if dense != "fused":
            assert dense_kernel(w, h, want_bgr=True) == "tma<true,64,0>"
    # TMA geometries with partial CTAs: in both directions, and in the row direction alone
    partial = [(w % P2_TW, h % P2_TH) for (w, h), (d, s, f) in GEOMETRIES.items() if d != "fused" and not f]
    assert any(px and py for px, py in partial) and any(py and not px for px, py in partial)
    # the sparse entry with partial CTAs also ends in a partial group of k_sparse_flags' tile rows (SFL_ROWS = 6)
    assert (1100 // 4) % 6 != 0


def test_misaligned_buffers_leave_the_fast_paths():
    assert dense_kernel(W4K, H4K, bgr_offset=1) == "fused"
    assert sparse_kernel(W4K, H4K, bgr_offset=1) is None
    assert sparse_kernel(W4K, H4K, gray_offset=1) is None
    assert sparse_kernel(W4K, H4K, gray_offset=4) == GEOMETRIES[(W4K, H4K)][1]
    assert sparse_kernel(W4K, H4K, batch=65) is None


@needs_cv2
@pytest.mark.parametrize("geom", list(GEOMETRIES), ids=GEOMETRY_IDS)
def test_edge_frame_puts_detections_in_the_last_ctas(oracle, camera, lut, dictionary, ref_params, geom):
    """At every geometry of at least 640 px the oracle chain finds at least 2 markers whose quads reach into the last CTA column
    or row; below that the frame has contrast everywhere and no marker, and the chain returns nothing."""
    from tools import synth
    w, h = geom
    K, D = camera
    frame = synth.make_edge_frame(dictionary.bytesList, 3, w, h)
    assert frame.shape == (h, w, 3) and frame.dtype == np.uint8
    assert np.array_equal(frame, synth.make_edge_frame(dictionary.bytesList, 3, w, h))
    mx, my = oracle.init_undistort_map(scaled_camera(K, w), D, w, h)
    _, gray = oracle.preprocess(frame, mx, my, lut)
    oc, oi, _ = oracle.detect_markers_apriltag(gray, dictionary.raw, ref_params)
    if w < 640:
        assert len(oi) == 0
        assert int(gray.max()) - int(gray.min()) >= ref_params.aprilTagMinWhiteBlackDiff
        assert len(np.unique(gray)) > 32
        return
    x0, y0 = last_cta_edges(w, h)
    at_edge = [bool(q[:, 0].max() >= x0 or q[:, 1].max() >= y0) for q in oc]
    print(f"{w}x{h}: {len(oi)} markers, {sum(at_edge)} in the last CTA column or row")
    assert sum(at_edge) >= 2
    assert len(oi) >= 8
