"""CPU: the frames that take detectMarkers (APRILTAG mode) past the shared-memory tiers of its kernels, checked on the oracle.

tests/test_gpu_scale.py runs the GPU on the same frames.  These tests make sure the frames really are what that file relies on
(non-vacuity: candidate counts on both sides of the 512-candidate tier of k_decode, boundary clusters above the 4 096 points
k_fit_quads sorts in shared memory, a frame above the per-frame point capacity), and that the oracle equals cv2 4.13 on them:
ids, order and float32 corners bit for bit where the candidates' perimeters are distinct, the same set of markers where they tie.
"""
import numpy as np
import pytest
from conftest import needs_cv2, cv2_params

MAX_POINTS = 1 << 20          # APSE_MAX_POINTS (csrc/common.cuh): boundary points per frame
SORT_SMEM = 4096              # APSE_SORT_SMEM: larger clusters are sorted in global memory by k_fit_quads
DEC_SMEMC = 512               # candidates k_decode keeps in shared memory

BIG_SIDES = (300, 600, 900, 1500)
GRIDS = {"grid512": (512, 0.0), "grid513": (513, 0.0), "grid520": (520, 0.0), "grid700_rot": (700, 0.3)}
TIE_GRIDS = ("grid512", "grid513", "grid520")


def make_frames(bytes_list):
    """name -> gray frame (3840x2160).  big<side>: one marker of that size; many600: 600 markers of 28-50 px; grid<n>: n markers
    of 30 px on a flat background (axis-aligned: equal perimeters); capacity: 2 300 grid markers, more boundary points than a
    frame may have."""
    from oracle import oracle as O
    from tools import synth
    frames = {f"big{s}": O.bgr2gray(synth.make_big_marker_frame(bytes_list, s)) for s in BIG_SIDES}
    frames["many600"] = O.bgr2gray(synth.make_frame(bytes_list, 77, ids=[i % 50 for i in range(600)], side_range=(28, 50), jitter=0.1,
                                                    margin=30, noise_sigma=3))
    for name, (n, rot) in GRIDS.items():
        frames[name] = synth.make_grid_frame(bytes_list, n, rotate=rot)
    frames["capacity"] = synth.make_grid_frame(bytes_list, 2300, pitch=56)
    return frames


def cluster_sizes(thresh, rep):
    """Points per boundary cluster, largest first: emit_points of oracle_apriltag.c restated in numpy (every pixel that is not 127,
    its 4 forward neighbours, a point where the two values sum to 255, keyed by the unordered pair of component representatives)."""
    h, w = thresh.shape
    v0 = thresh[1:h - 1, 1:w - 1].astype(np.int32)
    r0 = rep[1:h - 1, 1:w - 1].astype(np.uint64)
    keys = []
    for dx, dy in ((1, 0), (0, 1), (-1, 1), (1, 1)):
        v1 = thresh[1 + dy:h - 1 + dy, 1 + dx:w - 1 + dx].astype(np.int32)
        r1 = rep[1 + dy:h - 1 + dy, 1 + dx:w - 1 + dx].astype(np.uint64)
        m = (v0 != 127) & (v0 + v1 == 255)
        a, b = r0[m], r1[m]
        keys.append(np.where(a < b, (b << np.uint64(32)) + a, (a << np.uint64(32)) + b))
    _, counts = np.unique(np.concatenate(keys), return_counts=True)
    return np.sort(counts)[::-1]


def perimeters(corners):
    """float32 perimeters as the candidate filter computes them (sum of the four side lengths)."""
    c = np.asarray(corners, np.float32).reshape(-1, 4, 2)
    d = c - np.roll(c, -1, axis=1)
    p = np.zeros(len(c), np.float32)
    for k in range(4):
        p += np.sqrt(d[:, k, 0] * d[:, k, 0] + d[:, k, 1] * d[:, k, 1])
    return p


@pytest.fixture(scope="module")
def frames(dictionary):
    return make_frames(dictionary.bytesList)


@pytest.fixture(scope="module")
def stages(frames, oracle, ref_params):
    """name -> (oracle quads, oracle stage dumps, cluster sizes)"""
    out = {}
    for name, g in frames.items():
        q, st = oracle.at_quads(g, ref_params, dumps=True)
        out[name] = (q, st, cluster_sizes(st["thresh"], st["rep"]))
    return out


def test_cluster_helper_reproduces_the_oracle(stages):
    for name, (q, st, sizes) in stages.items():
        assert len(sizes) == st["clusters"], name
        assert sizes.sum() == st["points"], name


def test_frames_reach_the_tiers(stages):
    w, h = 3840, 2160
    fitted = {name: sizes[(sizes >= 100) & (sizes <= 3 * (2 * w + 2 * h))] for name, (_, _, sizes) in stages.items()}
    for name, (q, st, sizes) in stages.items():
        assert len(fitted[name]) == st["fitted"], name         # aprilTagMinClusterPixels = 100 and the size cap
    big = np.concatenate([fitted[f"big{s}"] for s in BIG_SIDES])
    assert ((big > SORT_SMEM) & (big <= 2 * SORT_SMEM)).any(), "no big-marker cluster in (4096, 8192]"
    assert (big > 4 * SORT_SMEM).any(), "no big-marker cluster above 16384"
    for s in BIG_SIDES:
        assert len(stages[f"big{s}"][0]) >= 1 and fitted[f"big{s}"].max() > SORT_SMEM, s
    assert len(stages["grid512"][0]) == DEC_SMEMC and len(stages["grid513"][0]) == DEC_SMEMC + 1
    assert 560 <= len(stages["grid700_rot"][0]) <= 900 and len(stages["many600"][0]) > DEC_SMEMC
    for name, (q, st, sizes) in stages.items():
        assert (st["points"] < MAX_POINTS) == (name != "capacity"), (name, st["points"])


@needs_cv2
def test_oracle_equals_cv2_on_scale_frames(frames, stages, oracle, dictionary, ref_params):
    import cv2
    det = cv2.aruco.ArucoDetector(cv2.aruco.getPredefinedDictionary(cv2.aruco.DICT_4X4_50), cv2_params(ref_params))
    for name, g in frames.items():
        if name == "capacity":
            continue
        oc, oi, orj = oracle.detect_markers_apriltag(g, dictionary.raw, ref_params)
        rc, ri, rr = det.detectMarkers(g)
        rc = np.array(rc, np.float32).reshape(-1, 4, 2)
        ri = ri.ravel() if ri is not None else np.zeros(0, np.int32)
        rr = np.array(rr, np.float32).reshape(-1, 4, 2)
        assert len(oi) >= 1 and len(orj) == len(rr), name
        per = perimeters(stages[name][0])
        if name in TIE_GRIDS:
            # every candidate has the same perimeter: cv2's sort is not stable here and returns the markers in another order
            # (DESIGN.md section 2); the set of markers and their corners are the same
            assert len(np.unique(per)) == 1 and len(oi) == len(per), name
            key = lambda c, i: np.lexsort((c[:, 0, 1], c[:, 0, 0], i))
            ko, kr = key(oc, oi), key(rc, ri)
            assert np.array_equal(oi[ko], ri[kr]) and np.array_equal(oc[ko], rc[kr]), name
        else:
            assert len(np.unique(per)) == len(per), name      # distinct perimeters: the order is fully determined
            assert np.array_equal(oi, ri) and np.array_equal(oc, rc), name
            assert np.array_equal(orj, rr), name
