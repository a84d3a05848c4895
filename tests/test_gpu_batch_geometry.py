"""GPU: the frame pipeline against the oracle at the batch sizes the benchmark runs and at frame sizes that leave partial CTAs.

Batch axis (4K, the test camera, one context of 64 frames).  bench.py sends 60-frame batches as 3 sub-batches of 20; the API takes
up to 64 frames per call.  k_preprocess_tma runs at most 20 frames per CTA (grid z = div_up(batch, 20) slices), so B = 20 fills one
slice, 21 and 41 give uneven slices (11 + 10, 14 + 14 + 13), and every B here takes the staging rings of the bounds pass (3 and 4
buffers) round more than twice, where the mbarrier parity comes back to 0.  At B > 32 the exact-tile list entries
(tx | ty << 13 | f << 26) set bit 31.  Twelve distinct frames are arranged so that no frame equals any of the 4 before it: a
staging buffer or an output slice left from another frame shows.  For B in {20, 21, 41, 64}:
  * preprocess (gray, gray + corrected BGR) equals oracle.preprocess at every position;
  * process_frames with the sparse evaluation and with the dense kernel, and preprocess_tiles[_sparse] + detect_pose_frames:
    ids, order, corners and rejected candidates equal the oracle chain's, poses within 1e-4, sparse = dense bit for bit;
  * the 4x4-tile extrema K1 hands to the detector (apse_debug_tile_extrema) equal the oracle gray's, on the tiles the sparse
    evaluation flagged, and are (255, 0) on the others;
  * every position equals a one-frame call on the same frame.
The full-range colour noise frame has more boundary points than a frame's work buffers hold: its detections may end with the
status APSE_ERR_CAPACITY, which the same frame must then give on every path; the other frames must end with status 0.
The 60-frame, 3-stream Pipeline of the benchmark gives the same results twice and equals the oracle.

Geometry axis: every entry of test_oracle_geometry.GEOMETRIES with the test lens and with pincushion5 (whose map sends many CTAs,
the partial ones included, down the direct-gather path): gray and BGR, tile extrema, tile bounds and flags, detections, and which
kernels ran.  Misaligned source and gray buffers give the aligned results.  One context cycled through three frame sizes gives, at
each step, what a fresh context of that size gives.
"""
import ctypes as C

import numpy as np
import pytest
from test_oracle_geometry import GEOMETRIES, GEOMETRY_IDS, H4K, W4K, dense_kernel, scaled_camera, sparse_kernel
from test_oracle_lens_models import LENSES

pytestmark = pytest.mark.gpu

ML = 0.55
MAX_MARKERS = 1024
KEYS = ("status", "n", "ids", "corners", "n_rejected", "rejected", "rvec", "tvec")
BATCHES = (20, 21, 41, 64)
CAPACITY = -4                     # APSE_ERR_CAPACITY


def _engine(K, D, lut, dictionary, params, w, h, batch):
    from apse_uav_b200.engine import Engine
    e = Engine(0, w, h, batch)
    _configure(e, K, D, lut, dictionary, params, w, h)
    return e


def _configure(e, K, D, lut, dictionary, params, w, h):
    e.set_camera(K, D, w, h)
    e.set_lut(lut)
    bl = np.ascontiguousarray(dictionary.bytesList, np.uint8)
    e.set_dictionary(bl.reshape(bl.shape[0], -1), dictionary.markerSize, dictionary.maxCorrectionBits)
    e.set_params(params)


def _oracle(oracle, frames, K, D, lut, dictionary, params, noise=()):
    """per frame: corrected BGR, gray, detections and poses of the oracle chain; `noise`: indices of full-range colour noise
    frames, whose candidate stage may exceed the library's per-frame work buffers"""
    h, w = frames[0].shape[:2]
    mx, my = oracle.init_undistort_map(K, D, w, h)
    out = []
    for f in frames:
        bgr, gray = oracle.preprocess(f, mx, my, lut)
        oc, oi, orj = oracle.detect_markers_apriltag(gray, dictionary.raw, params)
        otv = oracle.estimate_pose_single_markers(oc, ML, K, D)[1][:, 0] if len(oi) else np.zeros((0, 3))
        out.append(dict(bgr=bgr, gray=gray, corners=oc, ids=oi, rejected=orj, tvec=otv, noise=len(out) in noise))
    return out


def _host(det):
    import torch
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in det.items()}


def _run(e, frames, mode):
    """detections of one batch: 'sparse' / 'dense' = process_frames without / with a gray output, 'tiles' / 'tiles_sparse' =
    preprocess_tiles[_sparse] + detect_pose_frames"""
    import torch
    det = e.alloc_detections(frames.shape[0], MAX_MARKERS, True, pose=True)
    gray = torch.empty(frames.shape[:3], dtype=torch.uint8, device="cuda")
    if mode in ("sparse", "dense"):
        e.process_frames(frames, det, ML, gray=None if mode == "sparse" else gray)
    else:
        e.preprocess_tiles(frames, gray, sparse=mode == "tiles_sparse")
        e.detect_pose_frames(gray, det, ML)
    return _host(det)


def _same(a, b, what, fa=None, fb=None):
    """equal status everywhere; every output equal on the frames without an error status (a frame whose work buffers
    overflowed has no defined detections)"""
    sa = a["status"] if fa is None else a["status"][fa:fa + 1]
    sb = b["status"] if fb is None else b["status"][fb:fb + 1]
    assert np.array_equal(sa, sb), (what, "status", sa, sb)
    ok = sa == 0
    for k in KEYS[1:]:
        x = a[k] if fa is None else a[k][fa:fa + 1]
        y = b[k] if fb is None else b[k][fb:fb + 1]
        assert np.array_equal(x[ok], y[ok]), (what, k)


def _vs_oracle(res, f, ref, what):
    n, nr = int(res["n"][f]), int(res["n_rejected"][f])
    if ref["noise"] and int(res["status"][f]) == CAPACITY:
        return                    # reported, not truncated silently (DESIGN.md §3)
    assert int(res["status"][f]) == 0, what
    assert n == len(ref["ids"]) and np.array_equal(res["ids"][f, :n], ref["ids"]), (what, n, len(ref["ids"]))
    assert np.array_equal(res["corners"][f, :n], ref["corners"]), what
    assert nr == len(ref["rejected"]) and np.array_equal(res["rejected"][f, :nr], ref["rejected"]), (what, nr, len(ref["rejected"]))
    if n:
        rel = np.linalg.norm(res["tvec"][f, :n] - ref["tvec"], axis=-1) / np.linalg.norm(ref["tvec"], axis=-1)
        assert rel.max() < 1e-4, what


def _extrema(e, batch):
    """apse_debug_tile_extrema of the last preprocess_tiles call: (min, max) int tensors [batch][h/4][w/4]"""
    import torch
    w, h = e.size
    t = torch.zeros((batch, h // 4, w // 4), dtype=torch.int16, device="cuda")
    e._check(e.lib.apse_debug_tile_extrema(e.h, t.data_ptr(), batch, e._stream()))
    t = t.to(torch.int32) & 0xffff
    return t & 255, t >> 8


def _flags(e, batch):
    import torch
    w, h = e.size
    fl = torch.zeros((batch, h // 4, w // 4), dtype=torch.uint8, device="cuda")
    e._check(e.lib.apse_debug_sparse(e.h, None, fl.data_ptr(), batch, None, e._stream()))
    return fl.bool()


def _tile_minmax(gray):
    """4x4-tile (min, max) of [B,H,W] uint8 gray (CUDA tensor), complete tiles only, as int32"""
    import torch
    B, H, W = gray.shape
    t = gray[:, :H // 4 * 4, :W // 4 * 4].to(torch.int32).reshape(B, H // 4, 4, W // 4, 4)
    return t.amin((2, 4)), t.amax((2, 4))


def _check_extrema(e, og, flags=None):
    """tile extrema of the last preprocess_tiles call against those of the oracle gray og [B,H,W] (CUDA); with the tile flags
    of the sparse evaluation: equal where flagged, (255, 0) elsewhere"""
    import torch
    mn, mx = _extrema(e, og.shape[0])
    emn, emx = _tile_minmax(og)
    if flags is not None:
        emn = torch.where(flags, emn, torch.full_like(emn, 255))
        emx = torch.where(flags, emx, torch.zeros_like(emx))
    bad = ((mn != emn) | (mx != emx)).flatten(1).sum(1)
    assert int(bad.sum()) == 0, f"tile extrema differ in {bad.tolist()} tiles per frame"


def _dil(a, f):
    p = np.pad(a, 1, mode="edge")
    out = a.copy()
    for dy in range(3):
        for dx in range(3):
            out = f(out, p[dy:dy + a.shape[0], dx:dx + a.shape[1]])
    return out


def _check_sparse_tiles(e, og, gray, mwbd):
    """after preprocess_tiles(sparse=True): bounds contain the oracle gray, every tile the threshold reads (and its ring) is
    flagged, flagged tiles hold the oracle gray, the extrema are those of the flagged tiles"""
    import torch
    B = og.shape[0]
    w, h = e.size
    tb = torch.zeros((B, h // 4, w // 4), dtype=torch.int16, device="cuda")
    e._check(e.lib.apse_debug_tile_bounds(e.h, tb.data_ptr(), B, e._stream()))
    flags = _flags(e, B)
    _check_extrema(e, og, flags)
    tb = tb.to(torch.int32) & 0xffff
    emn, emx = _tile_minmax(og)
    assert bool(((tb & 255) <= emn).all()) and bool(((tb >> 8) >= emx).all()), "tile bounds miss the gray"
    px = flags.repeat_interleave(4, 1).repeat_interleave(4, 2)
    assert torch.equal(gray[px], og[px]), "gray of a flagged tile differs from the oracle"
    fl, mn, mx = flags.cpu().numpy(), emn.cpu().numpy(), emx.cpu().numpy()
    for f in range(B):
        active = (_dil(mx[f], np.maximum) - _dil(mn[f], np.minimum)) >= mwbd
        assert not (_dil(active, np.logical_or) & ~fl[f]).any(), "a tile the detector reads was not evaluated"


# ------------------------------------------------------------------------------------------------------------- batch axis
N_DISTINCT = 12


def _order(B):
    """frame index of each batch position: period 12, step 5, so no frame repeats within 5 positions"""
    return [(5 * i + B) % N_DISTINCT for i in range(B)]


@pytest.fixture(scope="module")
def batch_set(oracle, camera, lut, dictionary, ref_params):
    """12 distinct 4K frames (7 sparse marker frames of different ids and sizes, 2 dense, textured background only, full-range
    colour noise, markers in the last CTA column and row) and the oracle chain's results"""
    pytest.importorskip("cv2")   # tools.synth renders the frames with cv2
    from tools import synth
    K, D = camera
    bl = dictionary.bytesList
    sides = ((40, 70), (60, 110), (30, 50), (80, 140), (45, 90), (35, 60), (100, 160))
    frames = [synth.make_frame(bl, 7100 + 17 * i, ids=tuple(range(1 + 5 * i, 5 + 5 * i + i % 3)), side_range=sides[i])
              for i in range(7)]
    frames += [synth.make_dense_frame(bl, 600), synth.make_dense_frame(bl, 601), synth.make_frame(bl, 7300, ids=()),
               np.random.default_rng(3).integers(0, 256, (H4K, W4K, 3), dtype=np.uint8), synth.make_edge_frame(bl, 5, W4K, H4K)]
    frames = np.stack(frames)
    ref = _oracle(oracle, frames, K, D, lut, dictionary, ref_params, noise=(10,))
    assert sum(len(r["ids"]) >= 3 for r in ref) >= 9
    return frames, ref


@pytest.fixture(scope="class")
def ctx(batch_set, camera, lut, dictionary, ref_params):
    """the 64-frame context, the frames and oracle gray / BGR on the device, and one-frame results of every frame"""
    import torch
    frames, ref = batch_set
    K, D = camera
    e = _engine(K, D, lut, dictionary, ref_params, W4K, H4K, 64)
    dev = torch.from_numpy(frames).cuda()
    og = torch.from_numpy(np.stack([r["gray"] for r in ref])).cuda()
    ob = torch.from_numpy(np.stack([r["bgr"] for r in ref])).cuda()
    single = [{m: _run(e, dev[i:i + 1], m) for m in ("sparse", "dense")} for i in range(N_DISTINCT)]
    yield e, dev, og, ob, single
    e.close()


class TestBatchAxis:
    @pytest.mark.parametrize("B", BATCHES)
    def test_preprocess_every_position(self, ctx, B):
        import torch
        e, dev, og, ob, _ = ctx
        idx = torch.tensor(_order(B), device="cuda")
        frames = dev[idx].contiguous()
        _, gray = e.preprocess(frames)
        bgr, gray2 = e.preprocess(frames, want_bgr=True)
        for what, got, want in (("gray", gray, og[idx]), ("gray with BGR", gray2, og[idx]), ("BGR", bgr, ob[idx])):
            bad = (got != want).flatten(1).any(1).nonzero().flatten().tolist()
            assert not bad, f"B={B}: {what} differs from the oracle at positions {bad}"

    @pytest.mark.parametrize("B", BATCHES)
    def test_detections_every_position(self, ctx, batch_set, ref_params, B):
        import torch
        e, dev, og, _, single = ctx
        _, ref = batch_set
        order = _order(B)
        idx = torch.tensor(order, device="cuda")
        frames = dev[idx].contiguous()
        res = {m: _run(e, frames, m) for m in ("sparse", "dense")}
        _same(res["sparse"], res["dense"], f"B={B} sparse vs dense")
        for f, i in enumerate(order):
            _vs_oracle(res["dense"], f, ref[i], f"B={B} position {f} (frame {i})")
            for m in ("sparse", "dense"):
                _same(res[m], single[i][m], f"B={B} position {f} (frame {i}) {m} vs one-frame call", fa=f, fb=0)
        # the two halves of process_frames, with the tile extrema K1 leaves for the detector checked on the way
        gray = torch.empty(frames.shape[:3], dtype=torch.uint8, device="cuda")
        e.preprocess_tiles(frames, gray)
        assert torch.equal(gray, og[idx])
        _check_extrema(e, og[idx])
        det = e.alloc_detections(B, MAX_MARKERS, True, pose=True)
        e.detect_pose_frames(gray, det, ML)
        _same(_host(det), res["dense"], f"B={B} preprocess_tiles + detect_pose_frames")
        gray.fill_(77)
        e.preprocess_tiles(frames, gray, sparse=True)
        _check_sparse_tiles(e, og[idx], gray, ref_params.aprilTagMinWhiteBlackDiff)
        det = e.alloc_detections(B, MAX_MARKERS, True, pose=True)
        e.detect_pose_frames(gray, det, ML)
        _same(_host(det), res["dense"], f"B={B} preprocess_tiles_sparse + detect_pose_frames")


def test_benchmark_pipeline_shape(batch_set, camera, lut, dictionary, ref_params):
    """Pipeline(max_batch=60, streams=3) as bench.py runs it: two runs identical, every frame equal to the oracle"""
    import torch
    import apse_uav_b200 as A
    frames, ref = batch_set
    K, D = camera
    order = _order(60)
    pipe = A.Pipeline(K, D, (W4K, H4K), lut, dictionary, ref_params, max_batch=60, max_markers=MAX_MARKERS, streams=3)
    dev = torch.from_numpy(frames).cuda()[torch.tensor(order, device="cuda")].contiguous()
    torch.cuda.synchronize()
    runs = [_host(A.Pipeline.wait(pipe.run_batch(dev, want_rejected=True, sync=False, input_ready=True))) for _ in range(2)]
    pipe.close()
    _same(runs[0], runs[1], "two runs")
    for f, i in enumerate(order):
        _vs_oracle(runs[0], f, ref[i], f"Pipeline position {f} (frame {i})")


# ---------------------------------------------------------------------------------------------------------- geometry axis
def _geometry_frames(dictionary, w, h):
    from tools import synth
    rng = np.random.default_rng(w * 7 + h)
    return np.stack([synth.make_edge_frame(dictionary.bytesList, 11, w, h), rng.integers(0, 256, (h, w, 3), dtype=np.uint8),
                     synth.make_edge_frame(dictionary.bytesList, 12, w, h)])


@pytest.mark.parametrize("lens", ["reference", "pincushion5"])
@pytest.mark.parametrize("geom", list(GEOMETRIES), ids=GEOMETRY_IDS)
def test_geometry(oracle, lut, dictionary, ref_params, geom, lens):
    pytest.importorskip("cv2")
    import torch
    from apse_uav_b200._lib import ApseError
    w, h = geom
    K, D = LENSES[lens]
    K = scaled_camera(K, w)
    frames = _geometry_frames(dictionary, w, h)
    B = len(frames)
    ref = _oracle(oracle, frames, K, D, lut, dictionary, ref_params, noise=(1,))
    og = torch.from_numpy(np.stack([r["gray"] for r in ref])).cuda()
    ob = torch.from_numpy(np.stack([r["bgr"] for r in ref])).cuda()
    e = _engine(K, D, lut, dictionary, ref_params, w, h, B)
    dev = torch.from_numpy(frames).cuda()
    _, gray = e.preprocess(dev)
    bgr, gray2 = e.preprocess(dev, want_bgr=True)
    assert torch.equal(gray, og) and torch.equal(gray2, og) and torch.equal(bgr, ob)

    tma = dense_kernel(w, h) != "fused"
    sparse_ok = sparse_kernel(w, h, B) is not None
    g = torch.empty_like(gray)
    e.preprocess_tiles(dev, g)
    assert torch.equal(g, og)
    if tma:
        _check_extrema(e, og)
    else:
        with pytest.raises(ApseError):
            _extrema(e, B)
    g.fill_(77)
    e.preprocess_tiles(dev, g, sparse=True)
    if sparse_ok:
        _check_sparse_tiles(e, og, g, ref_params.aprilTagMinWhiteBlackDiff)
    else:
        assert torch.equal(g, og)           # the dense kernel ran instead
        if tma:
            _check_extrema(e, og)

    e.timing(True)
    e.timing_collect(reset=True)
    res = {m: _run(e, dev, m) for m in ("sparse", "dense", "tiles", "tiles_sparse")}
    launched = e.timing_collect(reset=True)
    e.timing(False)
    e.close()
    for m in ("dense", "tiles", "tiles_sparse"):
        _same(res["sparse"], res[m], f"{w}x{h} {lens}: sparse vs {m}")
    for f in range(B):
        _vs_oracle(res["dense"], f, ref[f], f"{w}x{h} {lens} frame {f}")
    # process_frames and preprocess_tiles_sparse each ran the flag and exact kernels once, exactly where the sparse path is eligible
    for k in ("k_sparse_flags", "k_sparse_exact"):
        assert launched.get(k, (0, 0))[1] == (2 if sparse_ok else 0), (k, launched.get(k))
    if w >= 640 and lens == "reference":
        assert min(int(n) for n in res["dense"]["n"][[0, 2]]) >= 8


def test_misaligned_buffers(oracle, camera, lut, dictionary, ref_params):
    """4K with the source frames one byte off a 16-byte boundary (k_preprocess_fused instead of the TMA kernels, sparse falls
    back) and a gray buffer one byte off (the sparse path falls back to the dense kernel; the fused kernel and the detector's
    threshold kernels leave their 32-bit accesses): the results of the aligned calls"""
    pytest.importorskip("cv2")
    import torch
    K, D = camera
    frames = _geometry_frames(dictionary, W4K, H4K)
    B = len(frames)
    e = _engine(K, D, lut, dictionary, ref_params, W4K, H4K, B)
    dev = torch.from_numpy(frames).cuda()
    raw = torch.empty(dev.numel() + 16, dtype=torch.uint8, device="cuda")
    off = raw[1:1 + dev.numel()].view(dev.shape)
    off.copy_(dev)
    assert off.data_ptr() % 16 == 1
    _, g0 = e.preprocess(dev)
    b0, _ = e.preprocess(dev, want_bgr=True)
    _, g1 = e.preprocess(off)
    b1, _ = e.preprocess(off, want_bgr=True)
    assert torch.equal(g0, g1) and torch.equal(b0, b1)
    want = {m: _run(e, dev, m) for m in ("sparse", "dense")}
    _same(want["sparse"], want["dense"], "aligned sparse vs dense")
    for m in ("sparse", "dense"):
        _same(_run(e, off, m), want[m], f"misaligned source, {m}")
    graw = torch.empty(g0.numel() + 16, dtype=torch.uint8, device="cuda")
    goff = graw[1:1 + g0.numel()].view(g0.shape)
    e.preprocess_tiles(dev, goff, sparse=True)
    assert torch.equal(goff, g0)            # the dense kernel ran: every pixel written
    det = e.alloc_detections(B, MAX_MARKERS, True, pose=True)
    e.detect_pose_frames(goff, det, ML)
    _same(_host(det), want["sparse"], "misaligned sparse gray")
    # both off: k_preprocess_fused writes the gray bytes, no tile extrema, the detector reduces the unaligned gray itself
    det = e.alloc_detections(B, MAX_MARKERS, True, pose=True)
    goff.fill_(77)
    e.process_frames(off, det, ML, gray=goff)
    _same(_host(det), want["dense"], "misaligned source and gray")
    assert torch.equal(goff, g0)
    det = e.detect(goff, max_markers=MAX_MARKERS)
    assert torch.equal(det["ids"], e.detect(g0, max_markers=MAX_MARKERS)["ids"])
    e.close()


def test_context_reuse_across_frame_sizes(lut, camera, dictionary, ref_params):
    """One 4K context of 8 frames cycled through 1952x1100 (3 frames), 3840x2152 (2), 3840x2160 (5) and 1952x1100 (1), with
    set_camera between: every step equals a fresh context of exactly that size and batch (the ternary image of the detector is
    reset when the size changes, and every buffer is addressed with the strides of the current size)"""
    pytest.importorskip("cv2")
    import torch
    from tools import synth
    K, D = camera
    bl = dictionary.bytesList
    steps = [((1952, 1100), [synth.make_edge_frame(bl, 21, 1952, 1100), synth.make_dense_frame(bl, 22, 1952, 1100, n_markers=80),
                             synth.make_edge_frame(bl, 23, 1952, 1100)]),
             ((3840, 2152), [synth.make_dense_frame(bl, 24, 3840, 2152), synth.make_edge_frame(bl, 25, 3840, 2152)]),
             ((3840, 2160), [synth.make_dense_frame(bl, 26), synth.make_edge_frame(bl, 27, 3840, 2160), synth.make_frame(bl, 28),
                             synth.make_dense_frame(bl, 29), synth.make_frame(bl, 30, ids=(5, 6, 7, 8, 9), side_range=(30, 60))]),
             ((1952, 1100), [synth.make_dense_frame(bl, 31, 1952, 1100, n_markers=80)])]

    def outputs(e, frames):
        out = {m: _run(e, frames, m) for m in ("sparse", "dense", "tiles_sparse")}
        _, g = e.preprocess(frames)
        out["gray"] = g.cpu().numpy()
        return out

    fresh = []
    for (w, h), fr in steps:
        e = _engine(scaled_camera(K, w), D, lut, dictionary, ref_params, w, h, len(fr))
        fresh.append(outputs(e, torch.from_numpy(np.stack(fr)).cuda()))
        e.close()
    e = _engine(K, D, lut, dictionary, ref_params, W4K, H4K, 8)
    for k, ((w, h), fr) in enumerate(steps):
        e.set_camera(scaled_camera(K, w), D, w, h)
        got = outputs(e, torch.from_numpy(np.stack(fr)).cuda())
        assert np.array_equal(got["gray"], fresh[k]["gray"]), (k, w, h)
        for m in ("sparse", "dense", "tiles_sparse"):
            _same(got[m], fresh[k][m], f"step {k} ({w}x{h}, {len(fr)} frames) {m}")
        assert int(got["dense"]["n"].sum()) >= 8 * len(fr), (k, got["dense"]["n"])
    e.close()
