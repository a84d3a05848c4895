"""GPU: detectMarkers (APRILTAG mode, and the classic path where it shares the decode stage) past the shared-memory tiers of
its kernels, against the oracle (= cv2 4.13 on these frames, tests/test_oracle_scale.py):
  * k_fit_quads on boundary clusters of 4 000 - 50 000 points (sorted in global memory above 4 096);
  * k_decode above 512 candidates per frame (its arrays in global scratch), on a fresh context and after a classic detection;
  * candidates with equal perimeters: the order of the output follows the dependency's candidate order, run after run;
  * frames of very unequal work in one batch, the sparse evaluation on big markers, and the capacity limits.
"""
import copy

import numpy as np
import pytest
from conftest import has_cv2, cv2_params, classic_params
from test_oracle_scale import make_frames, perimeters, TIE_GRIDS

pytestmark = pytest.mark.gpu
MAXQ = 4096                   # APSE_MAX_QUADS: candidates per frame, and the output capacity used here
STAGE_FRAMES = ("big300", "big600", "big900", "big1500", "many600")
TIER_FRAMES = ("grid512", "grid513", "grid700_rot", "many600")
CLASSIC_WINS = (13, 13, 1)    # one threshold window: the grids stay under 4 096 classic candidates


@pytest.fixture(scope="module")
def frames(dictionary):
    return make_frames(dictionary.bytesList)


@pytest.fixture(scope="module")
def odet(frames, oracle, dictionary, ref_params):
    """oracle detectMarkers (APRILTAG mode) on every frame the point capacity admits"""
    return {k: oracle.detect_markers_apriltag(g, dictionary.raw, ref_params) for k, g in frames.items() if k != "capacity"}


def _engine(dictionary, params, batch=1, camera=None, lut=None):
    from apse_uav_b200.engine import Engine
    e = Engine(0, 3840, 2160, batch)
    bl = np.ascontiguousarray(dictionary.bytesList, np.uint8)
    e.set_dictionary(bl.reshape(bl.shape[0], -1), dictionary.markerSize, dictionary.maxCorrectionBits)
    e.set_params(params)
    if camera is not None:
        e.set_camera(camera[0], camera[1], 3840, 2160)
        e.set_lut(lut)
    return e


def _detect(e, grays):
    import torch
    g = np.stack(grays) if isinstance(grays, (list, tuple)) else grays[None]
    det = e.detect(torch.from_numpy(g).cuda(), max_markers=MAXQ)
    return {k: v.cpu().numpy() for k, v in det.items()}


def _assert_frame_equals(res, f, ref, name):
    oc, oi, orj = ref
    n, nr = int(res["n"][f]), int(res["n_rejected"][f])
    assert int(res["status"][f]) == 0, name
    assert n == len(oi) and nr == len(orj), (name, n, len(oi), nr, len(orj))
    assert np.array_equal(res["ids"][f, :n], oi), name
    assert np.array_equal(res["corners"][f, :n], oc), name
    assert np.array_equal(res["rejected"][f, :nr], orj), name


@pytest.mark.parametrize("name", STAGE_FRAMES)
def test_stages_on_big_clusters(frames, oracle, dictionary, ref_params, name):
    """threshold image, component labels, point / cluster / fitted counts and the bit-identical quad set, as
    test_gpu_detect.py::test_apriltag_stages_4k, on clusters far above what k_fit_quads sorts in shared memory"""
    import torch
    gray = frames[name]
    oq, st = oracle.at_quads(gray, ref_params, dumps=True)
    e = _engine(dictionary, ref_params)
    dbg = e.debug_apriltag(torch.from_numpy(gray).cuda(), max_quads=MAXQ)
    th = dbg["thresh"].cpu().numpy()
    assert np.array_equal(th, st["thresh"])
    lab = dbg["labels"].cpu().numpy().view(np.uint32)
    m = th != 127
    assert np.array_equal(lab[m], st["rep"][m])
    assert (dbg["points"], dbg["clusters"], dbg["fitted"], dbg["n_quads"]) == (st["points"], st["clusters"], st["fitted"], len(oq))
    gq = dbg["quads"].cpu().numpy().reshape(-1, 8)
    dist = np.abs(gq[:, None, :] - oq.reshape(-1, 8)[None, :, :]).max(-1)
    assert len(oq) >= 1 and (dist.min(1) == 0).all() and (dist.min(0) == 0).all()
    e.close()


@pytest.mark.parametrize("name", TIER_FRAMES)
def test_apriltag_beyond_512_candidates_fresh_engine(frames, odet, dictionary, ref_params, name):
    """512, 513, 700 and 595 candidates on an engine that never ran the classic path: status 0 and the oracle's ids, order,
    corners and rejected candidates (a context without the decode scratch used to report APSE_ERR_CAPACITY above 512)"""
    e = _engine(dictionary, ref_params)
    res = _detect(e, frames[name])
    _assert_frame_equals(res, 0, odet[name], name)
    e.close()
    if has_cv2() and name not in TIE_GRIDS:
        import cv2
        det = cv2.aruco.ArucoDetector(cv2.aruco.getPredefinedDictionary(cv2.aruco.DICT_4X4_50), cv2_params(ref_params))
        rc, ri, rr = det.detectMarkers(frames[name])
        n = int(res["n"][0])
        assert np.array_equal(res["ids"][0, :n], ri.ravel()) and np.array_equal(res["corners"][0, :n], np.array(rc).reshape(-1, 4, 2))
        assert int(res["n_rejected"][0]) == len(rr)


def test_detection_does_not_depend_on_call_history(frames, odet, dictionary, ref_params):
    """a classic detection first (it used to be what allocated the decode scratch), then the APRILTAG frames on the same
    engine: the same results as on a fresh engine, i.e. the oracle's"""
    from apse_uav_b200 import aruco
    e = _engine(dictionary, classic_params(aruco, 0, CLASSIC_WINS))
    res = _detect(e, frames["grid513"])
    assert int(res["status"][0]) == 0 and int(res["n"][0]) == 513
    e.set_params(ref_params)
    for name in TIER_FRAMES:
        _assert_frame_equals(_detect(e, frames[name]), 0, odet[name], name)
    e.close()


@pytest.mark.parametrize("mode", [3, 0])
def test_perimeter_ties_follow_the_candidate_order(frames, oracle, dictionary, ref_params, mode):
    """axis-aligned grids: the candidates' float32 perimeters tie (all of them on the APRILTAG path, in groups on the classic
    one), so the output order is decided by the candidate order (the oracle's: ascending cluster key on the APRILTAG path,
    window then contour order on the classic one).  Two runs give identical outputs."""
    from apse_uav_b200 import aruco
    p = ref_params if mode == 3 else classic_params(aruco, 0, CLASSIC_WINS)
    fn = oracle.detect_markers_apriltag if mode == 3 else oracle.detect_markers_classic
    e = _engine(dictionary, p, batch=len(TIE_GRIDS))
    grays = [frames[k] for k in TIE_GRIDS]
    first = _detect(e, grays)
    second = _detect(e, grays)
    for k in first:
        assert np.array_equal(first[k], second[k]), k
    for f, name in enumerate(TIE_GRIDS):
        ref = fn(frames[name], dictionary.raw, p)
        # APRILTAG: one perimeter for all; classic (integer contour corners on a noisy threshold): ~100 distinct values
        assert len(ref[1]) >= 512 and len(np.unique(perimeters(ref[0]))) <= (1 if mode == 3 else len(ref[1]) // 4), name
        _assert_frame_equals(first, f, ref, name)
    e.close()


def test_mixed_batch_equals_single_frames(frames, odet, dictionary, ref_params):
    """big-marker, many-marker and empty frames in one call: k_fit_quads shares its persistent work list between frames of
    a single 18 000-point cluster and of 600 small ones; the results equal one call per frame (and the oracle)"""
    rng = np.random.default_rng(4)
    empty = np.clip(np.rint(128 + rng.normal(0, 2, (2160, 3840))), 0, 255).astype(np.uint8)
    names = ["big1500", "many600", None, "big600"]
    grays = [frames[k] if k else empty for k in names]
    e = _engine(dictionary, ref_params, batch=4)
    batch = _detect(e, grays)
    for f, name in enumerate(names):
        single = _detect(e, grays[f])
        for k in ("n", "n_rejected", "status"):
            assert single[k][0] == batch[k][f], (name, k)
        n, nr = int(single["n"][0]), int(single["n_rejected"][0])
        assert np.array_equal(single["ids"][0, :n], batch["ids"][f, :n]) and np.array_equal(single["corners"][0, :n], batch["corners"][f, :n])
        assert np.array_equal(single["rejected"][0, :nr], batch["rejected"][f, :nr])
        if name:
            _assert_frame_equals(batch, f, odet[name], name)
        else:
            assert n == 0 and int(batch["status"][f]) == 0
    e.close()


def test_sparse_evaluation_on_big_markers(oracle, camera, lut, dictionary, ref_params):
    """process_frames without a gray output (sparse evaluation: the decode samples outside the evaluated tiles are computed by
    exact_gray_px) on markers of 300-900 px: detections and poses bit-identical to the dense call, and equal to the oracle
    chain (preprocess -> detectMarkers -> pose)"""
    import torch
    from tools import synth
    sides = (300, 600, 900)
    bgr = np.stack([synth.make_big_marker_frame(dictionary.bytesList, s) for s in sides])
    e = _engine(dictionary, ref_params, batch=len(sides), camera=camera, lut=lut)
    frames = torch.from_numpy(bgr).cuda()
    outs = []
    for gray in (None, torch.empty(frames.shape[:3], dtype=torch.uint8, device="cuda")):
        det = e.alloc_detections(len(sides), 64, True, pose=True)
        e.process_frames(frames, det, 0.55, gray=gray)
        torch.cuda.synchronize()
        outs.append({k: v.cpu().numpy() for k, v in det.items()})
    sparse, dense = outs
    for k in ("status", "n", "ids", "corners", "n_rejected", "rejected", "rvec", "tvec"):
        assert np.array_equal(sparse[k], dense[k]), k
    K, D = camera
    ox, oy = oracle.init_undistort_map(K, D, 3840, 2160)
    for f in range(len(sides)):
        _, g = oracle.preprocess(bgr[f], ox, oy, lut)
        oc, oi, orj = oracle.detect_markers_apriltag(g, dictionary.raw, ref_params)
        n = int(sparse["n"][f])
        assert n == len(oi) >= 1 and int(sparse["n_rejected"][f]) == len(orj), sides[f]
        assert np.array_equal(sparse["ids"][f, :n], oi) and np.array_equal(sparse["corners"][f, :n], oc), sides[f]
        orv, otv = oracle.estimate_pose_single_markers(oc, 0.55, K, D)
        assert np.abs(sparse["tvec"][f, :n] - otv[:, 0]).max() <= 1e-4 * np.abs(otv).max(), sides[f]
    e.close()


def test_capacity_is_reported_not_truncated(frames, oracle, dictionary, ref_params):
    """2 300 grid markers have more boundary points than a frame may have: status APSE_ERR_CAPACITY from detect, ApseError from
    aruco.detectMarkers.  A classic frame with 1 100 markers (3 335 candidates) returns all of them, as cv2 does."""
    from apse_uav_b200 import aruco, ApseError
    from tools import synth
    e = _engine(dictionary, ref_params)
    res = _detect(e, frames["capacity"])
    assert int(res["status"][0]) == -4
    e.close()
    with pytest.raises(ApseError):
        aruco.detectMarkers(frames["capacity"], dictionary, parameters=ref_params)
    p = classic_params(aruco, 0, CLASSIC_WINS)
    gray = synth.make_grid_frame(dictionary.bytesList, 1100, rotate=0.3, seed=1)
    assert len(oracle.classic_quads(gray, p)) < MAXQ
    oc, oi, orj = oracle.detect_markers_classic(gray, dictionary.raw, p)
    assert len(oi) > 1024
    c, ids, rej = aruco.detectMarkers(gray, dictionary, parameters=p)
    assert ids is not None and np.array_equal(ids.ravel(), oi) and len(rej) == len(orj)
    assert np.array_equal(np.array(c).reshape(-1, 4, 2), oc)
    if has_cv2():
        import cv2
        det = cv2.aruco.ArucoDetector(cv2.aruco.getPredefinedDictionary(cv2.aruco.DICT_4X4_50), cv2_params(p))
        rc, ri, rr = det.detectMarkers(gray)
        assert np.array_equal(ids.ravel(), ri.ravel()) and len(rej) == len(rr)
