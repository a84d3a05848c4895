"""GPU: the preprocess, projection and pose kernels on the lens models of tests/test_oracle_lens_models.py (LENSES), against the
oracle and cv2.

The test camera's map is smooth enough that the direct-gather path of k_preprocess_tma runs in 10 CTAs per 4K frame, and its
thin-prism terms are zero.  The lenses here send up to half the CTAs down the direct-gather path (pincushion5, wide_pin), change
the break pattern of the shared tap rows of the bounds pass, leave a quarter of the sparse tiles to the general sampler, and give
s1..s4 non-zero values (prism12).  path_coverage() asserts on the map the GPU built that each lens reaches the path it is meant
for.  Checked per lens:
  * the undistortion map equals the oracle's bit for bit (and cv2's up to a few float32 ulp that do not move a Q5 tap);
  * dense preprocess (gray only at 4K, corrected BGR, a run-time width, a width without TMA) equals oracle.preprocess;
  * the sparse evaluation: tile bounds contain the dense gray, every tile the threshold needs is evaluated exactly, and
    process_frames gives the same detections and poses with and without a gray output;
  * the dense detections equal the oracle chain's (their threshold reads the tile extrema the preprocess kernel emits), and
    their poses (k_pose_frames4) agree with the oracle and cv2;
  * the cv2.undistort drop-in is bit-exact, projectPoints and apse_project_points_multi agree with cv2 within 1e-8 px;
  * estimatePoseSingleMarkers (k_pose4) and pose_frames (k_pose_frames4) on markers of every size, tilt and frame position;
  * a tilted-sensor distortion vector (tauX / tauY) is refused by every entry point without writing an output, and a
    distortion vector of a length cv2 does not know is refused;
  * prism12: the device projections of the sequence post-pass (k_sequence_jobs) equal the Python mirror.
"""
import ctypes as C

import numpy as np
import pytest
from conftest import has_cv2
from test_oracle_lens_models import (H4K, LENS_NAMES, LENSES, MARKER_LENGTH, W4K, check_coverage, full_frame_points,
                                     path_coverage, pose_sample, q5, rel_err, well_posed)

pytestmark = pytest.mark.gpu


def _engine(K, D, lut, dictionary, params, w=W4K, h=H4K, batch=3):
    from apse_uav_b200.engine import Engine
    e = Engine(0, w, h, batch)
    e.set_camera(K, D, w, h)
    e.set_lut(lut)
    bl = np.ascontiguousarray(dictionary.bytesList, np.uint8)
    e.set_dictionary(bl.reshape(bl.shape[0], -1), dictionary.markerSize, dictionary.maxCorrectionBits)
    e.set_params(params)
    return e


@pytest.fixture(scope="module")
def frames(frames4k):
    """A sparse and a dense marker frame and full-range colour noise, 4K."""
    noise = np.random.default_rng(11).integers(0, 256, (H4K, W4K, 3), dtype=np.uint8)
    return np.stack([frames4k["sparse"], frames4k["dense"], noise])


def _oracle_chain(oracle, lut, name, frames):
    """oracle.preprocess of the three frames on the oracle map of the lens: (corrected BGR list, gray list)"""
    K, D = LENSES[name]
    ox, oy = oracle.init_undistort_map(K, D, W4K, H4K)
    return [oracle.preprocess(f, ox, oy, lut) for f in frames]


def _dil(a, f):
    p = np.pad(a, 1, mode="edge")
    out = a.copy()
    for dy in range(3):
        for dx in range(3):
            out = f(out, p[dy:dy + a.shape[0], dx:dx + a.shape[1]])
    return out


def _both(e, frames, max_markers=256):
    import torch
    outs = []
    for gray in (None, torch.empty(frames.shape[:3], dtype=torch.uint8, device="cuda")):
        det = e.alloc_detections(frames.shape[0], max_markers, True, pose=True)
        e.process_frames(frames, det, MARKER_LENGTH, gray=gray)     # gray=None: sparse evaluation; a gray output: dense kernel
        torch.cuda.synchronize()
        outs.append({k: v.cpu().numpy() for k, v in det.items()})
    return outs


def _check_poses(rv, tv, corners, K, D, oracle):
    """GPU poses of `corners` against the oracle and cv2: on the well-posed samples within 1e-6 of the oracle and 1e-4 of cv2,
    elsewhere finite; at least 90 % well posed."""
    from oracle import cv2_compat as Cv
    orv, otv = oracle.estimate_pose_single_markers(corners, MARKER_LENGTH, K, D)
    crv, ctv, _ = Cv.estimatePoseSingleMarkers(list(np.asarray(corners).reshape(-1, 1, 4, 2)), MARKER_LENGTH, K, D)
    ok = well_posed(orv, otv, crv, ctv)
    assert ok.mean() >= 0.9, ok.mean()
    assert np.isfinite(rv).all() and np.isfinite(tv).all()
    assert rel_err(rv, orv)[ok].max() < 1e-6 and rel_err(tv, otv)[ok].max() < 1e-6
    assert rel_err(rv, crv)[ok].max() < 1e-4 and rel_err(tv, ctv)[ok].max() < 1e-4
    return ok.mean()


# -------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", LENS_NAMES)
def test_lens_map_bit_exact_and_path_coverage(oracle, name):
    from apse_uav_b200.engine import Engine
    K, D = LENSES[name]
    e = Engine(0, W4K, H4K, 1)
    mx, my = e.init_undistort_map(K, D, W4K, H4K)
    mx, my = mx.cpu().numpy(), my.cpu().numpy()
    ox, oy = oracle.init_undistort_map(K, D, W4K, H4K)
    assert np.array_equal(mx, ox) and np.array_equal(my, oy)
    check_coverage(name, path_coverage(mx, my))
    if has_cv2():
        import cv2
        cx, cy = cv2.initUndistortRectifyMap(K, D, None, K, (W4K, H4K), 5)
        assert ((mx != cx) | (my != cy)).sum() <= 4
        assert np.array_equal(q5(mx), q5(cx)) and np.array_equal(q5(my), q5(cy))
    e.close()


@pytest.mark.parametrize("name", LENS_NAMES)
def test_lens_dense_preprocess_4k(oracle, lut, dictionary, ref_params, frames, name):
    """gray only (k_preprocess_tma<false, 48, 3840, true>) and gray + corrected BGR (<true, 64, 0>), map of set_camera"""
    import torch
    K, D = LENSES[name]
    e = _engine(K, D, lut, dictionary, ref_params)
    t = torch.from_numpy(frames).cuda()
    _, gray = e.preprocess(t)
    bgr, gray2 = e.preprocess(t, want_bgr=True)
    gray, gray2, bgr = gray.cpu().numpy(), gray2.cpu().numpy(), bgr.cpu().numpy()
    for i, (rb, rg) in enumerate(_oracle_chain(oracle, lut, name, frames)):
        assert np.array_equal(gray[i], rg), (i, int((gray[i] != rg).sum()))
        assert np.array_equal(gray2[i], rg), i
        assert np.array_equal(bgr[i], rb), i
    e.close()


@pytest.mark.parametrize("name", LENS_NAMES)
def test_lens_preprocess_other_geometries(oracle, lut, dictionary, ref_params, name):
    """1920x1080 (k_preprocess_tma with the run-time width) and 1000x564 (3 w bytes not a multiple of 16: k_preprocess_fused),
    K scaled with the frame, the same distortion."""
    import torch
    from tools import synth
    K, D = LENSES[name]
    for w, h in ((1920, 1080), (1000, 564)):
        Ks = K.copy()
        Ks[:2] *= w / W4K
        rng = np.random.default_rng(w)
        fr = np.stack([synth.make_frame(dictionary.bytesList, 5, w, h, ids=(1, 2, 3, 4, 7), side_range=(40, 80)),
                       rng.integers(0, 256, (h, w, 3), dtype=np.uint8)])
        e = _engine(Ks, D, lut, dictionary, ref_params, w, h, 2)
        t = torch.from_numpy(fr).cuda()
        _, gray = e.preprocess(t)
        bgr, gray2 = e.preprocess(t, want_bgr=True)
        ox, oy = oracle.init_undistort_map(Ks, D, w, h)
        for i in range(2):
            rb, rg = oracle.preprocess(fr[i], ox, oy, lut)
            assert np.array_equal(gray[i].cpu().numpy(), rg), (w, i)
            assert np.array_equal(gray2[i].cpu().numpy(), rg), (w, i)
            assert np.array_equal(bgr[i].cpu().numpy(), rb), (w, i)
        e.close()


@pytest.mark.parametrize("name", LENS_NAMES)
def test_lens_sparse_evaluation(lut, dictionary, ref_params, frames, name):
    import torch
    K, D = LENSES[name]
    mwbd = ref_params.aprilTagMinWhiteBlackDiff
    e = _engine(K, D, lut, dictionary, ref_params)
    ft = torch.from_numpy(frames).cuda()
    _, dense = e.preprocess(ft)
    gray = torch.full_like(dense, 77)
    e.preprocess_tiles(ft, gray, sparse=True)
    tb = torch.zeros((3, H4K // 4, W4K // 4), dtype=torch.int16, device="cuda")
    e._check(e.lib.apse_debug_tile_bounds(e.h, tb.data_ptr(), 3, e._stream()))
    flags = torch.zeros((3, H4K // 4, W4K // 4), dtype=torch.uint8, device="cuda")
    n = C.c_int(0)
    e._check(e.lib.apse_debug_sparse(e.h, None, flags.data_ptr(), 3, C.byref(n), e._stream()))
    torch.cuda.synchronize()
    tb = tb.cpu().numpy().view(np.uint16)
    lo, hi = (tb & 255).astype(int), (tb >> 8).astype(int)
    flags = flags.cpu().numpy().astype(bool)
    assert n.value == flags.sum()
    d, g = dense.cpu().numpy(), gray.cpu().numpy()
    for f in range(3):
        t = d[f].reshape(H4K // 4, 4, W4K // 4, 4)
        tmin, tmax = t.min((1, 3)).astype(int), t.max((1, 3)).astype(int)
        assert (lo[f] <= tmin).all(), f"frame {f}: lower bound above the exact minimum in {(lo[f] > tmin).sum()} tiles"
        assert (hi[f] >= tmax).all(), f"frame {f}: upper bound below the exact maximum in {(hi[f] < tmax).sum()} tiles"
        need = _dil((_dil(tmax, np.maximum) - _dil(tmin, np.minimum)) >= mwbd, np.logical_or)
        assert not (need & ~flags[f]).any(), f"frame {f}: a tile the detector reads was not evaluated"
        px = np.repeat(np.repeat(flags[f], 4, 0), 4, 1)
        assert np.array_equal(g[f][px], d[f][px]), f"frame {f}: gray of an evaluated tile differs from the dense kernel"
        assert (g[f][~px] == 77).all(), f"frame {f}: a tile outside the list was written"
    print(name, "evaluated tile fraction per frame:", flags.mean((1, 2)))
    sparse, dense_det = _both(e, ft[:2])     # the two marker frames
    assert (sparse["status"] == 0).all() and (dense_det["status"] == 0).all()
    assert dense_det["n"][1] >= 50, dense_det["n"]
    for k in ("n", "ids", "corners", "n_rejected", "rejected", "rvec", "tvec"):
        assert np.array_equal(sparse[k], dense_det[k]), k
    e.close()


@pytest.mark.parametrize("name", LENS_NAMES)
def test_lens_detection_and_frame_poses_vs_oracle(oracle, lut, dictionary, ref_params, frames, name):
    """dense 4K frame: ids and corners of process_frames (gray output, so the detector thresholds with the tile extrema the
    preprocess kernel emits) equal the oracle chain's; the poses of k_pose_frames4 agree with the oracle and cv2"""
    import torch
    K, D = LENSES[name]
    e = _engine(K, D, lut, dictionary, ref_params, batch=1)
    ft = torch.from_numpy(frames[1:2]).cuda()
    det = e.alloc_detections(1, 512, True, pose=True)
    e.process_frames(ft, det, MARKER_LENGTH, gray=torch.empty((1, H4K, W4K), dtype=torch.uint8, device="cuda"))
    torch.cuda.synchronize()
    det = {k: v.cpu().numpy() for k, v in det.items()}
    assert det["status"][0] == 0
    _, g = _oracle_chain(oracle, lut, name, frames[1:2])[0]
    oc, oi, _ = oracle.detect_markers_apriltag(g, dictionary.raw, ref_params)
    n = int(det["n"][0])
    assert n >= 50 and n == len(oi), (n, len(oi))
    assert np.array_equal(det["ids"][0, :n], oi) and np.abs(det["corners"][0, :n] - oc).max() <= 1e-3
    frac = _check_poses(det["rvec"][0, :n], det["tvec"][0, :n], det["corners"][0, :n], K, D, oracle)
    print(f"{name}: {n} markers, {frac:.3f} of their poses well posed")
    e.close()


@pytest.mark.parametrize("name", LENS_NAMES)
def test_lens_undistort_dropin_bit_exact(oracle, frames, name):
    import apse_uav_b200 as A
    K, D = LENSES[name]
    frame = frames[2]
    out = A.undistort(frame, K, D)
    assert np.array_equal(out, oracle.undistort(frame, K, D))
    assert np.array_equal(A.undistort(frame, K, D, None, K), out)
    Ks = K.copy()
    Ks[:2] *= 0.25
    newK = Ks.copy()
    newK[0, 0] *= 0.9; newK[1, 1] *= 0.95; newK[0, 2] += 7.3
    g = np.random.default_rng(4).integers(0, 256, (540, 960), dtype=np.uint8)
    got = A.undistort(g, Ks, D, None, newK)
    assert np.array_equal(got, oracle.undistort(g, Ks, D, newK))
    if has_cv2():
        import cv2
        assert np.array_equal(out, cv2.undistort(frame, K, D))
        assert np.array_equal(got, cv2.undistort(g, Ks, D, None, newK))


@pytest.mark.parametrize("name", LENS_NAMES)
def test_lens_project_points(oracle, name):
    """projectPoints (k_project_points) and apse_project_points_multi on points over the whole frame"""
    import apse_uav_b200 as A
    from apse_uav_b200.engine import default_engine
    K, D = LENSES[name]
    rng = np.random.default_rng(2)
    objs, rs, ts, refs = [], [], [], []
    for _ in range(6):
        obj, r, t = full_frame_points(oracle, K, rng)
        img, _ = A.projectPoints(obj, r, t, K, D)
        ref = oracle.project_points(obj, r, t, K, D)
        if has_cv2():
            import cv2
            ref = cv2.projectPoints(obj, r, t, K, D)[0].reshape(-1, 2)
        assert np.abs(img.reshape(-1, 2) - ref).max() < 1e-8
        objs.append(obj); rs.append(r); ts.append(t); refs.append(ref)
    idx = np.repeat(np.arange(6, dtype=np.int32), [len(o) for o in objs])
    multi = default_engine().project_points_multi(np.concatenate(objs), idx, np.array(rs), np.array(ts), K, D).cpu().numpy()
    assert np.abs(multi - np.concatenate(refs)).max() < 1e-8


@pytest.mark.parametrize("name", LENS_NAMES)
def test_lens_pose_sample(oracle, name):
    """estimatePoseSingleMarkers (k_pose4) and pose_frames (k_pose_frames4): markers 20 to 400 px wide, tilted up to 0.5 rad,
    anywhere in the frame"""
    import torch
    from apse_uav_b200 import aruco
    from apse_uav_b200.engine import default_engine
    K, D = LENSES[name]
    corners = pose_sample(oracle, K, D, np.random.default_rng(5))
    rv, tv, _ = aruco.estimatePoseSingleMarkers(list(corners), MARKER_LENGTH, K, D)
    frac = _check_poses(rv, tv, corners, K, D, oracle)
    B, M = 8, len(corners) // 8
    c = torch.from_numpy(np.ascontiguousarray(corners.reshape(B, M, 4, 2))).cuda()
    nm = torch.full((B,), M, dtype=torch.int32, device="cuda")
    frv, ftv = default_engine().pose_frames(c, nm, MARKER_LENGTH, K, D)
    _check_poses(frv.cpu().numpy().reshape(-1, 3), ftv.cpu().numpy().reshape(-1, 3), corners, K, D, oracle)
    print(f"{name}: {frac:.3f} of {len(corners)} pose samples well posed")


def test_tilted_sensor_is_refused_without_output(oracle, lut, dictionary, ref_params):
    """tauX / tauY (D[12], D[13]) are not implemented: every entry point raises APSE_ERR_UNSUPPORTED and leaves its outputs and
    the context's camera untouched."""
    import torch
    import apse_uav_b200 as A
    from apse_uav_b200 import aruco, sequence
    from apse_uav_b200._lib import ApseError, darr, SEQ_JOB_DTYPE, SEQ_RESULT_DTYPE
    K, D = LENSES["prism12"]
    w, h = 640, 480
    Ks = K.copy()
    Ks[:2] *= w / W4K
    e = _engine(Ks, D, lut, dictionary, ref_params, w, h, 1)
    frame = torch.from_numpy(np.random.default_rng(3).integers(0, 256, (1, h, w, 3), dtype=np.uint8)).cuda()
    _, before = e.preprocess(frame)
    st = e._stream()
    (_, kp) = darr(Ks)
    obj = torch.zeros((4, 3), dtype=torch.float64, device="cuda")
    obj[:, 2] = 5
    r3 = torch.zeros(3, dtype=torch.float64, device="cuda")
    idx = torch.zeros(4, dtype=torch.int32, device="cuda")
    corners = torch.from_numpy(pose_sample(oracle, Ks, D, np.random.default_rng(1), 4, w, h).reshape(1, 4, 4, 2)).cuda()
    nm = torch.full((1,), 4, dtype=torch.int32, device="cuda")
    for j in (12, 13):
        Dt = np.zeros(14)
        Dt[:12] = D
        Dt[j] = 0.01
        (_, dp) = darr(Dt)
        with pytest.raises(ApseError) as ei:
            e.set_camera(Ks, Dt, w, h)
        assert ei.value.code == -5
        _, after = e.preprocess(frame)
        assert torch.equal(after, before), "a refused set_camera changed the context's map"
        mx = torch.full((h, w), 7.0, dtype=torch.float32, device="cuda")
        my = mx.clone()
        assert e.lib.apse_init_undistort_map(e.h, kp, dp, w, h, mx.data_ptr(), my.data_ptr(), st) == -5
        img8 = frame[0].clone()
        dst = torch.full_like(img8, 77)
        assert e.lib.apse_undistort(e.h, img8.data_ptr(), w, h, 3, kp, dp, None, dst.data_ptr(), st) == -5
        img = torch.full((4, 2), 7.0, dtype=torch.float64, device="cuda")
        assert e.lib.apse_project_points(e.h, obj.data_ptr(), 4, r3.data_ptr(), r3.data_ptr(), kp, dp, img.data_ptr(), st) == -5
        assert e.lib.apse_project_points_multi(e.h, obj.data_ptr(), 4, idx.data_ptr(), r3.data_ptr(), r3.data_ptr(), kp, dp,
                                               img.data_ptr(), st) == -5
        rv = torch.full((1, 4, 3), 7.0, dtype=torch.float64, device="cuda")
        tv = rv.clone()
        assert e.lib.apse_pose(e.h, corners.data_ptr(), 4, None, MARKER_LENGTH, kp, dp, rv.data_ptr(), tv.data_ptr(), st) == -5
        assert e.lib.apse_pose_frames(e.h, corners.data_ptr(), nm.data_ptr(), 1, 4, None, MARKER_LENGTH, kp, dp, rv.data_ptr(),
                                      tv.data_ptr(), st) == -5
        torch.cuda.synchronize()
        assert (mx == 7).all() and (my == 7).all() and (dst == 77).all() and (img == 7).all() and (rv == 7).all() and (tv == 7).all()
        # the cv2-shaped drop-ins and the sequence camera
        for call in (lambda: A.initUndistortRectifyMap(Ks, Dt, None, Ks, (w, h), 5), lambda: A.undistort(frame[0].cpu().numpy(), Ks, Dt),
                     lambda: A.projectPoints(np.zeros((1, 3)) + [0, 0, 5], np.zeros(3), np.zeros(3), Ks, Dt),
                     lambda: aruco.estimatePoseSingleMarkers(list(corners[0].cpu().numpy().reshape(4, 1, 4, 2)), MARKER_LENGTH, Ks, Dt)):
            with pytest.raises(ApseError):
                call()
        jobs = np.zeros(2, SEQ_JOB_DTYPE)
        jobs["kind"] = 1
        jobs["tvec"] = [0, 0, 5]
        jobs["dim"] = [-0.5, 0.5, -0.3, 0.3]
        jobs["scale"] = 1.0
        res = np.zeros(2, SEQ_RESULT_DTYPE)
        res["dist_bbox"] = 7.0
        e.D = Dt
        with pytest.raises(ApseError):
            sequence.run_jobs(e, jobs, results=res)
        assert (res["dist_bbox"] == 7.0).all() and (res["valid"] == 0).all()
        e.D = D
    # a distortion vector of a length cv2 does not accept
    for n in (3, 6, 13, 15):
        Db = np.full(n, 0.01)
        for call in (lambda: e.set_camera(Ks, Db, w, h), lambda: A.initUndistortRectifyMap(Ks, Db, None, Ks, (w, h), 5),
                     lambda: A.undistort(frame[0].cpu().numpy(), Ks, Db),
                     lambda: A.projectPoints(np.zeros((1, 3)) + [0, 0, 5], np.zeros(3), np.zeros(3), Ks, Db),
                     lambda: aruco.estimatePoseSingleMarkers(list(corners[0].cpu().numpy().reshape(4, 1, 4, 2)), MARKER_LENGTH, Ks, Db)):
            with pytest.raises(ApseError):
                call()
    e.close()


def test_prism12_sequence_jobs_equal_python_mirror(oracle, lut, dictionary, ref_params):
    """k_sequence_jobs projects the vehicle outlines with its own copy of projectPoints: with the thin-prism terms set, the
    finished rows equal the per-frame Python mirror of the post-pass on the oracle's projection."""
    from apse_uav_b200 import sequence
    from test_sequence_native import eval_jobs_numpy, fabricate, python_rows
    K, D = LENSES["prism12"]
    n, ids, corners, rvec, tvec = fabricate(oracle, K, D, seed=4)
    project = lambda obj, r, t: oracle.project_points(obj, r, t, K, D)
    want, _ = python_rows(n, ids, corners, rvec, tvec, project)
    _, rows, jobs = sequence.scan(sequence.seq_config(start_frame=1), n, ids, corners, rvec, tvec)
    assert len(jobs) > 50 and (jobs["kind"] >= 1).all()
    e = _engine(K, D, lut, dictionary, ref_params, batch=1)
    res = sequence.run_jobs(e, jobs)
    ref = eval_jobs_numpy(jobs, project)
    assert (res["valid"] == 1).all()
    assert np.array_equal(res["dist_bbox"], ref["dist_bbox"]) and np.array_equal(res["dist_aruco"], ref["dist_aruco"])
    assert sequence.rows_to_dicts(sequence.finish(rows, res)) == want
    e.close()
