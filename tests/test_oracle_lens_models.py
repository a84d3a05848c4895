"""CPU: the references (oracle/*.c and cv2) agree on lens models other than the test camera of tests/golden/cam_params.json.

The test camera has a strong 8-coefficient rational model whose thin-prism terms s1..s4 and tilt terms are zero, and its
undistortion map is so smooth that the preprocess kernels almost never leave their fast paths.  LENSES adds plain barrel and
pincushion lenses, a wide-angle pincushion, an off-centre principal point, a thin-prism model and the identity, with
distortion vectors of 4, 5, 12 and 14 entries.  tests/test_gpu_lens_models.py pins the kernels to the references on these
lenses; this file checks first that the references themselves hold there.

path_coverage() restates, from an undistortion map, which code paths of csrc/preprocess.cu that map sends the pixels down, so
that the lens tests can assert they reach the paths they are meant for.
"""
import json
import os

import numpy as np
import pytest
from conftest import GOLDEN, needs_cv2

W4K, H4K = 3840, 2160
MARKER_LENGTH = 0.55


def _lenses():
    cam = json.load(open(os.path.join(GOLDEN, "cam_params.json")))
    K = np.array(cam["mtx"], np.float64)
    wide = K.copy()
    wide[:2, :2] *= 0.6
    off = K.copy()
    off[0, 2], off[1, 2] = 700.0, 300.0
    return {
        "reference": (K, np.array(cam["dist"], np.float64).ravel()),
        "pincushion5": (K, np.array([0.45, 0.2, 0, 0, 0])),
        "wide_pin": (wide, np.array([0.25, 0.05, 0, 0, 0])),
        "barrel5": (K, np.array([-0.35, 0.12, 0, 0, 0])),
        "prism12": (K, np.array([-0.1, 0.02, 0.02, -0.015, 0, 0, 0, 0, 0.02, -0.004, 0.015, 0.003])),
        "offcentre": (off, np.array([-0.2, 0.05, 0, 0, 0])),
        "zero4": (K, np.zeros(4)),
    }


LENSES = _lenses()
LENS_NAMES = list(LENSES)


def q5(m):
    """Q5 source coordinate of cv2.remap / the kernels: rint(map * 32) in float32, saturated to int32 like __float2int_rn."""
    v = np.rint(np.asarray(m, np.float32) * np.float32(32)).astype(np.float64)
    return np.clip(v, -2.0 ** 31, 2.0 ** 31 - 1).astype(np.int64)


def path_coverage(mapx, mapy):
    """Which paths of csrc/preprocess.cu a 4K undistortion map takes (the map as the kernels read it: Q5 taps).

    * direct: k_preprocess_tma CTAs (64 x 24 output px) whose source box, with its left edge rounded down to 16 px for the bulk
      tensor copy (bx0 = xmin & ~15), exceeds the 85 x 32 px staging buffer -> the direct-gather path (MODE 0 and MODE 1);
      direct_inside: how many of those have every tap inside the frame (real pixels, not the zero fill);
    * brk: warps (32 columns x 4 rows) of the bounds pass where some pixel's successor one row down does not sit in the same
      source column one source row further, so the staged tap row is not shared (the `brk` mask);
    * edge_tiles: 4 x 4 tiles of k_sparse_exact with a pixel outside its interior test (general sampler instead of the gathered
      rows);
    * outside: output pixels whose source point lies outside the frame.
    """
    h, w = mapx.shape
    assert w % 64 == 0 and h % 24 == 0
    sx, sy = q5(mapx), q5(mapy)
    ix, iy = sx >> 5, sy >> 5
    cx, cy = np.clip(ix, -2, w + 1), np.clip(iy, -2, h + 1)     # taps wholly outside are clamped next to the frame
    blk = lambda a: a.reshape(h // 24, 24, w // 64, 64)
    xmin, xmax = blk(cx).min((1, 3)), blk(cx).max((1, 3)) + 1
    ymin, ymax = blk(cy).min((1, 3)), blk(cy).max((1, 3)) + 1
    bx0 = xmin & ~15
    direct = (xmax - bx0 + 1 > 85) | (ymax - ymin + 1 > 32)
    inside = (xmin >= 0) & (xmax <= w - 1) & (ymin >= 0) & (ymax <= h - 1)
    same = (cx[1:] == cx[:-1]) & (cy[1:] == cy[:-1] + 1)         # pixel (y + 1, x) against (y, x)
    brk = np.concatenate([~same, np.zeros((1, w), bool)]).reshape(h // 4, 4, w)[:, :3].any(1)   # pairs inside a 4-row group
    warp_brk = brk.reshape(h // 4, w // 32, 32).any(-1)
    interior = (ix >= 0) & (ix + 4 < w) & (iy >= 0) & (iy + 1 < h)
    edge_tiles = (~interior).reshape(h // 4, 4, w // 4, 4).any((1, 3))
    outside = ~((sx >= 0) & (sx <= 32 * (w - 1)) & (sy >= 0) & (sy <= 32 * (h - 1)))
    return dict(direct=float(direct.mean()), direct_inside=int((direct & inside).sum()), brk=float(warp_brk.mean()),
                edge_tiles=float(edge_tiles.mean()), outside=float(outside.mean()))


def check_coverage(name, cov):
    """The lenses meant for the direct-gather path reach it, on real pixels; the others keep the paths the tests rely on."""
    print(f"{name}: direct-gather CTAs {100 * cov['direct']:.2f} % ({cov['direct_inside']} inside the frame), warps with a break "
          f"{100 * cov['brk']:.1f} %, non-interior sparse tiles {100 * cov['edge_tiles']:.2f} %, source outside {100 * cov['outside']:.2f} %")
    if name in ("pincushion5", "wide_pin"):
        assert cov["direct"] >= 0.25, cov
    if name == "pincushion5":
        assert cov["direct_inside"] >= 1000, cov
    if name == "zero4":
        assert cov["direct"] == 0 and cov["brk"] == 0 and cov["outside"] == 0, cov
    if name in ("barrel5", "offcentre", "prism12"):
        assert cov["brk"] >= 0.5, cov


def full_frame_points(oracle, K, rng, n=400, zrange=(2.0, 60.0)):
    """(object points, rvec, tvec): points whose undistorted projections spread over (and a little beyond) the 4K frame."""
    u = rng.uniform(-0.05 * W4K, 1.05 * W4K, n)
    v = rng.uniform(-0.05 * H4K, 1.05 * H4K, n)
    z = rng.uniform(*zrange, n)
    P = np.stack([(u - K[0, 2]) / K[0, 0] * z, (v - K[1, 2]) / K[1, 1] * z, z], -1)
    r = rng.normal(0, 0.4, 3)
    t = rng.uniform([-2, -2, -1], [2, 2, 1])
    R = oracle.rodrigues(r)[0]
    return (P - t) @ R, r, t                                     # R obj + t = P


def pose_sample(oracle, K, D, rng, n=240, w=W4K, h=H4K):
    """Corners (n,1,4,2) float32 of markers of MARKER_LENGTH: tilt up to 0.5 rad, 20 to 400 px wide, anywhere in the frame
    (all four corners inside it), 0.1 px of noise."""
    hl = np.float32(MARKER_LENGTH) / np.float32(2)
    objm = np.array([[-hl, hl, 0], [hl, hl, 0], [hl, -hl, 0], [-hl, -hl, 0]], np.float64)
    out = []
    while len(out) < n:
        side = np.exp(rng.uniform(np.log(20), np.log(400)))
        z = MARKER_LENGTH * K[0, 0] / side
        c = oracle.undistort_points(rng.uniform([0, 0], [w, h]).reshape(1, 2), K, D)[0]
        t = np.array([c[0] * z, c[1] * z, z])
        axis = rng.normal(0, 1, 2)
        tilt = np.append(axis / np.linalg.norm(axis) * rng.uniform(0, 0.5), 0.0)
        R = oracle.rodrigues(tilt)[0] @ oracle.rodrigues(np.array([0, 0, rng.uniform(-np.pi, np.pi)]))[0]
        img = oracle.project_points(objm, oracle.rodrigues_inv(R), t, K, D) + rng.normal(0, 0.1, (4, 2))
        if np.all(np.isfinite(img)) and (img >= 0).all() and (img[:, 0] < w).all() and (img[:, 1] < h).all():
            out.append(img.astype(np.float32).reshape(1, 4, 2))
    return np.array(out)


def rel_err(a, b):
    a, b = np.asarray(a).reshape(-1, 3), np.asarray(b).reshape(-1, 3)
    return np.linalg.norm(a - b, axis=-1) / np.maximum(np.linalg.norm(b, axis=-1), 1e-300)


def well_posed(orv, otv, crv, ctv):
    """Samples where the oracle and cv2 reach the same pose (1e-7 relative): there the pose is a property of the input.  On the
    others (distant, small or strongly tilted markers) Levenberg-Marquardt stops at its iteration cap or in the other planar
    minimum, and neither result is the reference."""
    return (rel_err(orv, crv) < 1e-7) & (rel_err(otv, ctv) < 1e-7)


# -------------------------------------------------------------------------------------------------------------------------
def test_dist14_pads_the_accepted_lengths_and_refuses_others():
    from apse_uav_b200._lib import ApseError, dist14
    d = np.arange(1, 15, dtype=np.float64) / 100
    for n in (4, 5, 8, 12, 14):
        k = dist14(d[:n])
        assert k.shape == (14,) and np.array_equal(k[:n], d[:n]) and not k[n:].any()
        assert np.array_equal(dist14(d[:n].reshape(-1, 1)), k)          # the (n,1) column cv2 returns
    assert not dist14(None).any()
    for n in (0, 1, 3, 6, 7, 9, 13, 15):
        with pytest.raises(ApseError):
            dist14(d[:n] if n <= 14 else np.zeros(n))


@needs_cv2
@pytest.mark.parametrize("name", LENS_NAMES)
def test_lens_map_vs_cv2(oracle, name):
    import cv2
    K, D = LENSES[name]
    mx, my = cv2.initUndistortRectifyMap(K, D, None, K, (W4K, H4K), 5)
    ox, oy = oracle.init_undistort_map(K, D, W4K, H4K)
    bad = (ox != mx) | (oy != my)
    assert bad.sum() <= 4, bad.sum()
    assert np.array_equal(q5(ox), q5(mx)) and np.array_equal(q5(oy), q5(my))
    check_coverage(name, path_coverage(ox, oy))


@needs_cv2
@pytest.mark.parametrize("name", LENS_NAMES)
def test_lens_preprocess_vs_cv2(oracle, lut, name):
    """oracle.preprocess on the oracle map == cv2.remap + the colour chain of aruco_detect.py:250-259 on cv2's map, on
    full-range colour noise (every tap of every path sees distinct pixels)."""
    import cv2
    from oracle import cv2_compat as C
    K, D = LENSES[name]
    frame = np.random.default_rng(7).integers(0, 256, (H4K, W4K, 3), dtype=np.uint8)
    mx, my = cv2.initUndistortRectifyMap(K, D, None, K, (W4K, H4K), 5)
    ox, oy = oracle.init_undistort_map(K, D, W4K, H4K)
    bgr, gray = oracle.preprocess(frame, ox, oy, lut)
    ref = C.preprocess_frame(frame, mx, my, lut.reshape(1, 256))
    assert np.array_equal(bgr, ref)
    assert np.array_equal(gray, cv2.cvtColor(ref, cv2.COLOR_BGR2GRAY))


@needs_cv2
@pytest.mark.parametrize("name", LENS_NAMES)
def test_lens_project_undistort_vs_cv2(oracle, name):
    import cv2
    K, D = LENSES[name]
    rng = np.random.default_rng(1)
    for _ in range(6):
        obj, r, t = full_frame_points(oracle, K, rng)
        a, jac = cv2.projectPoints(obj, r, t, K, D)
        b, dr, dt = oracle.project_points(obj, r, t, K, D, jacobian=True)
        assert np.abs(a.reshape(-1, 2) - b).max() < 1e-9
        assert np.abs(jac[:, :3] - dr).max() < 1e-6 * np.abs(jac[:, :3]).max()
        assert np.abs(jac[:, 3:6] - dt).max() < 1e-6 * np.abs(jac[:, 3:6]).max()
    pts = rng.uniform([0, 0], [W4K, H4K], (400, 2))
    a = cv2.undistortPoints(pts.reshape(-1, 1, 2), K, D).reshape(-1, 2)
    assert np.abs(a - oracle.undistort_points(pts, K, D)).max() < 1e-13


@needs_cv2
@pytest.mark.parametrize("name", LENS_NAMES)
def test_lens_pose_sample_is_mostly_well_posed(oracle, name):
    from oracle import cv2_compat as C
    K, D = LENSES[name]
    corners = pose_sample(oracle, K, D, np.random.default_rng(5))
    crv, ctv, _ = C.estimatePoseSingleMarkers(list(corners), MARKER_LENGTH, K, D)
    orv, otv = oracle.estimate_pose_single_markers(corners, MARKER_LENGTH, K, D)
    ok = well_posed(orv, otv, crv, ctv)
    print(f"{name}: {ok.mean():.3f} of {len(ok)} pose samples well posed")
    assert ok.mean() >= 0.9
    assert np.isfinite(orv).all() and np.isfinite(otv).all()
