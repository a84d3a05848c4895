"""GPU: the hand-off of tile extrema (and, for a sparse batch, tile flags) from apse_preprocess_tiles[_sparse] to
apse_detect_pose_frames.

The library keeps two slots, so that the preprocess of one sub-batch can run while the detector chain of the previous one is
still in flight (Pipeline).  Checked here:
  * two sparse batches preprocessed into two gray buffers are each detected with their own slot, in either order, and give
    what process_frames gives on the same frames, without recomputing any extrema;
  * a detect call on other data between the preprocess and its detect_pose_frames drops the hand-off: a dense gray batch is
    then detected from its pixels (extrema recomputed, the same detections), a sparse one is refused;
  * the kernels each entry point launches, per kernel, at 4K and at a geometry without the TMA kernels.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ML = 0.55
MAX_MARKERS = 256
KEYS = ("status", "n", "ids", "corners", "n_rejected", "rejected", "rvec", "tvec")
GENERIC = (1920, 1082)   # h % 4 = 2: the generic preprocess kernel, no tile extrema, no sparse evaluation


def _engine(K, D, lut, dictionary, params, w, h, batch):
    from apse_uav_b200.engine import Engine
    e = Engine(0, w, h, batch)
    e.set_camera(K, D, w, h)
    e.set_lut(lut)
    bl = np.ascontiguousarray(dictionary.bytesList, np.uint8)
    e.set_dictionary(bl.reshape(bl.shape[0], -1), dictionary.markerSize, dictionary.maxCorrectionBits)
    e.set_params(params)
    return e


@pytest.fixture
def engine4k(camera, lut, dictionary, ref_params):
    e = _engine(camera[0], camera[1], lut, dictionary, ref_params, 3840, 2160, 2)
    yield e
    e.close()


@pytest.fixture(scope="module")
def batches4k(frames4k):
    """two 4K batches holding the same two frames in opposite order"""
    import torch
    a = torch.from_numpy(np.stack([frames4k["sparse"], frames4k["dense"]])).cuda()
    return a, a.flip(0).contiguous()


def _host(det):
    import torch
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in det.items()}


def _same(a, b, what):
    assert (a["status"] == 0).all() and (b["status"] == 0).all(), what
    for k in KEYS:
        assert np.array_equal(a[k], b[k]), (what, k)


def _process(e, frames, gray=None):
    det = e.alloc_detections(frames.shape[0], MAX_MARKERS, True, pose=True)
    e.process_frames(frames, det, ML, gray=gray)
    return _host(det)


def _detect(e, gray):
    det = e.alloc_detections(gray.shape[0], MAX_MARKERS, True, pose=True)
    e.detect_pose_frames(gray, det, ML)
    return _host(det)


def _timed(e, fn):
    """fn() with per-kernel timing on: (its result, {kernel name: launches})"""
    e.timing(True)
    e.timing_collect(reset=True)
    r = fn()
    launched = {k: n for k, (_, n) in e.timing_collect(reset=True).items()}
    e.timing(False)
    return r, launched


def test_two_sparse_batches_detected_in_reverse_order(engine4k, batches4k):
    import torch
    e = engine4k
    a, b = batches4k
    ref = [_process(e, a), _process(e, b)]
    assert ref[0]["n"].min() >= 4 and not np.array_equal(ref[0]["ids"], ref[1]["ids"])
    ga, gb = (torch.empty(f.shape[:3], dtype=torch.uint8, device="cuda") for f in (a, b))
    e.preprocess_tiles(a, ga, sparse=True)
    e.preprocess_tiles(b, gb, sparse=True)
    (rb, ra), launched = _timed(e, lambda: (_detect(e, gb), _detect(e, ga)))
    _same(ra, ref[0], "first batch")
    _same(rb, ref[1], "second batch")
    assert "k_tile_minmax" not in launched, launched   # both batches came with their extrema
    assert launched["k_decode"] == 2


@pytest.mark.parametrize("sparse", [False, True], ids=["dense", "sparse"])
def test_detect_in_between_drops_the_handoff(engine4k, batches4k, sparse):
    import torch
    from apse_uav_b200._lib import ApseError
    e = engine4k
    a, b = batches4k
    ga = torch.empty(a.shape[:3], dtype=torch.uint8, device="cuda")
    ref = _process(e, a, gray=ga)
    _, other = e.preprocess(b)
    e.preprocess_tiles(a, ga, sparse=sparse)
    e.detect(other, MAX_MARKERS)
    torch.cuda.synchronize()
    n0 = e.launches
    if sparse:   # the gray batch is only complete together with its flags, which are gone
        with pytest.raises(ApseError):
            _detect(e, ga)
        assert e.launches == n0
        return
    r, launched = _timed(e, lambda: _detect(e, ga))
    _same(r, ref, "dense gray after a detect call in between")
    assert launched["k_tile_minmax"] == 1, launched


# per-kernel launches of one call of each entry point (after one call of the same kind), recorded before the hand-off state of
# the library was restructured: which kernels run must not depend on how that state is kept.  (k_preprocess_fused counts every
# dense or bounds preprocess kernel, k_threshold every kernel of the threshold stage.)
MODES = ("process", "process_gray", "tiles", "tiles_sparse")
_CHAIN = {"k_preprocess_fused": 1, "k_threshold": 4, "k_ccl_local": 1, "k_ccl_merge": 1, "k_emit_points": 2, "k_cluster_scan": 1,
          "k_scatter_points": 1, "k_fit_quads": 2, "k_decode_bits": 1, "k_decode": 1, "k_pose": 1}
_SPARSE = {**_CHAIN, "k_sparse_flags": 1, "k_sparse_exact": 1}
LAUNCHES = {
    ("3840x2160", "process"): _SPARSE,
    ("3840x2160", "process_gray"): _CHAIN,
    ("3840x2160", "tiles"): _CHAIN,
    ("3840x2160", "tiles_sparse"): _SPARSE,
    # no tile extrema from the generic preprocess kernel, a partial tile row for the edge threshold kernel
    **{("1920x1082", m): {**_CHAIN, "k_tile_minmax": 1, "k_threshold": 5} for m in MODES},
}


def _launches(e, frames, mode):
    import torch
    gray = torch.empty(frames.shape[:3], dtype=torch.uint8, device="cuda")

    def once():
        if mode in ("process", "process_gray"):
            _process(e, frames, gray=gray if mode == "process_gray" else None)
        else:
            e.preprocess_tiles(frames, gray, sparse=mode == "tiles_sparse")
            _detect(e, gray)
    once()
    return _timed(e, once)[1]


def _frames(dictionary, geom):
    import torch
    from tools import synth
    w, h = geom
    return torch.from_numpy(np.stack([synth.make_edge_frame(dictionary.bytesList, 11 + i, w, h) for i in range(2)])).cuda()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("geom", [(3840, 2160), GENERIC], ids=["3840x2160", "generic"])
def test_launches_per_entry_point(camera, lut, dictionary, ref_params, geom, mode):
    from test_oracle_geometry import scaled_camera
    w, h = geom
    e = _engine(scaled_camera(camera[0], w), camera[1], lut, dictionary, ref_params, w, h, 2)
    try:
        launched = _launches(e, _frames(dictionary, geom), mode)
    finally:
        e.close()
    assert launched == LAUNCHES[f"{w}x{h}", mode]
