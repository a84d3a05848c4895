"""Seeded synthetic 4K UAV frames with ArUco markers (test / bench input data, not product code).

The reference's datasets are Google-Drive links (reference README.md:50-56) and unavailable offline, so
every parity fixture and benchmark in this repository runs on frames produced here.  Recipe = SURVEY.md
section 8(d): smooth random background, `DICT_4X4_50` markers rendered at 48 px + 8 px quiet zone, warped by
a random rotation + corner-jitter homography with bilinear blur, pasted, optional occluders and Gaussian
noise.  Frames play the role of RAW camera frames (pre-undistortion) so the preprocess stage is exercised.

Marker bitmaps are rendered from the dictionary byte list directly (no cv2.aruco call), so the generator
only needs cv2 for resize/warpPerspective.
"""
from __future__ import annotations

import numpy as np
import cv2

# ---------------------------------------------------------------------------------------------------------
# marker bitmaps


def marker_bits(bytes_list: np.ndarray, marker_id: int, marker_size: int = 4) -> np.ndarray:
    """Inner bit matrix (marker_size x marker_size, 1 = white) of a dictionary marker, rotation 0."""
    row = np.asarray(bytes_list)[marker_id].reshape(-1)  # (nbytes*4,) rotation-major
    nbytes = (marker_size * marker_size + 7) // 8
    b = np.unpackbits(row[:nbytes].astype(np.uint8))
    # Dictionary::getByteListFromBits packs MSB-first, the last byte holds the remaining bits right-aligned
    nbits = marker_size * marker_size
    if nbits % 8:
        full = (nbits // 8) * 8
        tail = b[full:full + 8][8 - (nbits - full):]
        b = np.concatenate([b[:full], tail])
    return b[:nbits].reshape(marker_size, marker_size)


def render_marker(bytes_list: np.ndarray, marker_id: int, side_px: int = 48, marker_size: int = 4,
                  border_bits: int = 1, quiet_px: int = 8) -> np.ndarray:
    """Canonical marker image (uint8) with a white quiet zone; equals generateImageMarker for side_px
    divisible by (marker_size + 2*border_bits)."""
    n = marker_size + 2 * border_bits
    cells = np.zeros((n, n), np.uint8)
    cells[border_bits:border_bits + marker_size, border_bits:border_bits + marker_size] = \
        marker_bits(bytes_list, marker_id, marker_size) * 255
    img = cv2.resize(cells, (side_px, side_px), interpolation=cv2.INTER_NEAREST)
    out = np.full((side_px + 2 * quiet_px, side_px + 2 * quiet_px), 255, np.uint8)
    out[quiet_px:quiet_px + side_px, quiet_px:quiet_px + side_px] = img
    return out


# ---------------------------------------------------------------------------------------------------------
# frames


def background(rng: np.random.Generator, width: int, height: int) -> np.ndarray:
    small = rng.integers(60, 200, size=(max(2, height // 16), max(2, width // 16), 3), dtype=np.uint8)
    return cv2.resize(small, (width, height), interpolation=cv2.INTER_CUBIC)


def _paste_marker(frame: np.ndarray, tile: np.ndarray, quad: np.ndarray, quiet_frac: float) -> None:
    """Warp `tile` (marker + quiet zone) so that the MARKER corners land on `quad` (4x2, clockwise from
    top-left), bilinear, and paste it (with its quiet zone) into frame (all 3 channels)."""
    s = tile.shape[0]
    q = quiet_frac * s
    src = np.float32([[q, q], [s - q, q], [s - q, s - q], [q, s - q]])
    H = cv2.getPerspectiveTransform(src, quad.astype(np.float32))
    # bounding box of the warped full tile
    full = cv2.perspectiveTransform(np.float32([[[0, 0], [s, 0], [s, s], [0, s]]]), H)[0]
    x0, y0 = np.floor(full.min(0)).astype(int) - 2
    x1, y1 = np.ceil(full.max(0)).astype(int) + 2
    h, w = frame.shape[:2]
    x0, y0, x1, y1 = max(x0, 0), max(y0, 0), min(x1, w), min(y1, h)
    if x1 <= x0 or y1 <= y0:
        return
    T = np.array([[1, 0, -x0], [0, 1, -y0], [0, 0, 1]], np.float64) @ H
    size = (int(x1 - x0), int(y1 - y0))
    warped = cv2.warpPerspective(tile, T, size, flags=cv2.INTER_LINEAR, borderValue=0)
    mask = cv2.warpPerspective(np.full_like(tile, 255), T, size, flags=cv2.INTER_LINEAR, borderValue=0)
    a = (mask.astype(np.float32) / 255.0)[..., None]
    roi = frame[y0:y1, x0:x1].astype(np.float32)
    roi = roi * (1 - a) + warped[..., None].astype(np.float32) * a
    frame[y0:y1, x0:x1] = np.clip(np.rint(roi), 0, 255).astype(np.uint8)


# LED strip of the host vehicle, metres in the marker frame (x right, y up; aruco_detect.py:340-341), marker side 0.55 m
LED_AXIS = np.float32([[-0.419, -0.42], [-0.414, -0.305], [-0.409, -0.19], [-0.404, -0.07], [-0.399, 0.065], [-0.393, 0.19],
                       [-0.388, 0.315], [-0.382, 0.435]])


def _draw_leds(frame: np.ndarray, quad: np.ndarray, pattern: int, marker_length: float = 0.55, radius: int = 7) -> None:
    """Bright disc for every set bit of `pattern` (bit 7 = first LED) at the LED's place in the marker plane."""
    unit = np.float32([[-0.5, 0.5], [0.5, 0.5], [0.5, -0.5], [-0.5, -0.5]]) * marker_length   # corner order of solvePnP
    H = cv2.getPerspectiveTransform(unit, quad.astype(np.float32))
    px = cv2.perspectiveTransform(LED_AXIS.reshape(1, -1, 2), H)[0]
    for j in range(8):
        on = (pattern >> (7 - j)) & 1
        cv2.circle(frame, (int(round(px[j][0])), int(round(px[j][1]))), radius, (255, 255, 255) if on else (25, 25, 25), -1)


def _random_quad(rng, cx, cy, side, jitter):
    ang = rng.uniform(0, 2 * np.pi)
    c, s = np.cos(ang), np.sin(ang)
    base = np.float32([[-1, -1], [1, -1], [1, 1], [-1, 1]]) * (side / 2)
    rot = base @ np.float32([[c, s], [-s, c]])
    rot += rng.uniform(-jitter * side, jitter * side, size=(4, 2)).astype(np.float32)
    return rot + np.float32([cx, cy])


def make_frame(bytes_list, seed: int, width: int = 3840, height: int = 2160, ids=(1, 2, 3, 4),
               side_range=(50, 90), jitter: float = 0.06, noise_sigma: float = 3.0,
               occlude_frac: float = 0.0, centers=None, angles=None, margin: int = 90,
               return_truth: bool = False, leds=None):
    """One synthetic BGR frame (uint8 HxWx3).  `centers` (list of (x,y)) pins marker positions (sequence
    drift); otherwise positions are rejection-sampled without overlap."""
    rng = np.random.default_rng(seed)
    frame = background(rng, width, height)
    placed, truth = [], []
    for k, mid in enumerate(ids):
        side = float(rng.uniform(*side_range))
        if centers is not None:
            cx, cy = centers[k]
        else:
            for _ in range(200):
                cx = float(rng.uniform(margin, width - margin))
                cy = float(rng.uniform(margin, height - margin))
                if all((cx - px) ** 2 + (cy - py) ** 2 > (1.1 * (side + ps)) ** 2 for px, py, ps in placed):
                    break
            else:
                continue
        placed.append((cx, cy, side))
        quad = _random_quad(rng, cx, cy, side, jitter)
        if angles is not None:  # fixed orientation for sequences (keeps yaw stable between frames)
            c, s = np.cos(angles[k]), np.sin(angles[k])
            base = np.float32([[-1, -1], [1, -1], [1, 1], [-1, 1]]) * (side / 2)
            quad = base @ np.float32([[c, s], [-s, c]]) + np.float32([cx, cy]) + \
                rng.uniform(-jitter * side, jitter * side, size=(4, 2)).astype(np.float32)
        tile = render_marker(bytes_list, int(mid))
        _paste_marker(frame, tile, quad, quiet_frac=8.0 / tile.shape[0])
        if leds is not None and int(mid) == 4:
            _draw_leds(frame, quad, leds)
        if occlude_frac > 0 and rng.uniform() < occlude_frac:
            ow, oh = rng.uniform(0.15, 0.45, size=2) * side
            ox = cx + rng.uniform(-0.5, 0.5) * side
            oy = cy + rng.uniform(-0.5, 0.5) * side
            col = rng.integers(40, 220, size=3).tolist()
            cv2.rectangle(frame, (int(ox), int(oy)), (int(ox + ow), int(oy + oh)), col, -1)
        truth.append((int(mid), quad))
    if noise_sigma > 0:
        noise = rng.normal(0.0, noise_sigma, size=frame.shape).astype(np.float32)
        frame = np.clip(np.rint(frame.astype(np.float32) + noise), 0, 255).astype(np.uint8)
    return (frame, truth) if return_truth else frame


def make_dense_frame(bytes_list, seed: int, width: int = 3840, height: int = 2160, n_markers: int = 200,
                     noise_sigma: float = 4.0, n_ids: int = 50):
    """Config-5 stress frame: ~200 markers, ids 0..49 cycled, side 28-90 px, jitter 0.2, 15 % occluded."""
    ids = [i % n_ids for i in range(n_markers)]
    return make_frame(bytes_list, seed, width, height, ids=ids, side_range=(28, 90), jitter=0.2,
                      noise_sigma=noise_sigma, occlude_frac=0.15, margin=70)


def make_nested_frame(bytes_list, seed: int, width: int = 1920, height: int = 1080, levels: int = 3, noise_sigma: float = 2.0):
    """Markers inside markers: a big marker, a medium one inside one of its white cells, (levels = 3) a tiny one inside a white
    cell of the medium one, and a free-standing marker.  Exercises the candidate tree of detectMarkers (a quad that encloses an
    already decoded marker).  Returns (frame, ids placed outermost first)."""
    rng = np.random.default_rng(seed)
    frame = background(rng, width, height)

    def square(cx, cy, s, ang):
        c, s_ = np.cos(ang), np.sin(ang)
        base = np.float32([[-1, -1], [1, -1], [1, 1], [-1, 1]]) * (s / 2)
        return base @ np.float32([[c, s_], [-s_, c]]) + np.float32([cx, cy])

    def paste(mid, quad):
        tile = render_marker(bytes_list, int(mid))
        _paste_marker(frame, tile, np.float32(quad), quiet_frac=8.0 / tile.shape[0])

    def white_cell(mid, k, cx, cy, side, ang):
        ys, xs = np.nonzero(marker_bits(bytes_list, int(mid)))
        k %= len(ys)
        u, v = (xs[k] + 1.5) / 6 - 0.5, (ys[k] + 1.5) / 6 - 0.5
        c, s_ = np.cos(ang), np.sin(ang)
        off = np.float32([u * side, v * side]) @ np.float32([[c, s_], [-s_, c]])
        return cx + off[0], cy + off[1]

    sc = min(width / 1920.0, height / 1080.0)
    a1, a2 = rng.uniform(-0.5, 0.5, 2)
    ids = [int(v) for v in rng.choice(len(bytes_list), 4, replace=False)]
    bx, by, bs = 0.36 * width, 0.5 * height, 900 * sc
    paste(ids[0], square(bx, by, bs, a1))
    mx, my = white_cell(ids[0], int(rng.integers(0, 16)), bx, by, bs, a1)
    paste(ids[1], square(mx, my, 100 * sc, a2))
    if levels >= 3:
        tx, ty = white_cell(ids[1], int(rng.integers(0, 16)), mx, my, 100 * sc, a2)
        paste(ids[2], square(tx, ty, 11 * sc, rng.uniform(-0.5, 0.5)))
    paste(ids[3], square(0.83 * width, 0.28 * height, 150 * sc, 0.3))
    if noise_sigma > 0:
        frame = np.clip(np.rint(frame.astype(np.float32) + rng.normal(0, noise_sigma, frame.shape)), 0, 255).astype(np.uint8)
    return frame, ids


def make_edge_frame(bytes_list, seed: int, width: int, height: int, n_band: int = 6, noise_sigma: float = 3.0):
    """BGR frame whose markers sit where the preprocess kernels have partial work: k_preprocess_tma covers the frame with CTAs of
    64 x 24 output px, so a width or height that is not a multiple of those leaves a last CTA column or row with idle threads.
    On the textured background, n_band rotated markers (side 34-52 px) straddle the left edge of the last CTA column
    (x0 = width - width % 64, or width - 64) and n_band the top edge of the last CTA row (y0 likewise with 24), and three
    markers are cut by the right and bottom frame edges (part of each in the last 8 px).  Positions are in the raw frame; the
    undistortion moves them by a few pixels.  Frames narrower than 640 px get full-range colour noise over a colour gradient
    instead (no marker fits)."""
    rng = np.random.default_rng(seed)
    if width < 640:
        ramp = np.stack(np.broadcast_arrays((np.arange(width) * 255 // max(1, width - 1))[None, :],
                                            (np.arange(height) * 255 // max(1, height - 1))[:, None],
                                            ((np.arange(width)[None, :] + np.arange(height)[:, None]) * 4) % 256), -1)
        noise = rng.integers(-60, 61, (height, width, 3))
        return np.clip(ramp + noise, 0, 255).astype(np.uint8)
    frame = background(rng, width, height)
    x0 = width - (width % 64 or 64)
    y0 = height - (height % 24 or 24)
    ids = rng.choice(len(bytes_list), 2 * n_band + 3, replace=False)

    def paste(mid, cx, cy, side):
        tile = render_marker(bytes_list, int(mid))
        _paste_marker(frame, tile, _random_quad(rng, cx, cy, side, 0.04), quiet_frac=8.0 / tile.shape[0])

    for k in range(n_band):
        side = float(rng.uniform(34, 52))
        reach = side * 0.75 + 4                                   # half diagonal of the marker and its quiet zone
        t = 0.12 + 0.6 * (k + rng.uniform(0.2, 0.8)) / n_band     # along the band, clear of the corner where the bands meet
        paste(ids[2 * k], min(x0 + rng.uniform(-6, 14), width - reach), t * height, side)
        paste(ids[2 * k + 1], t * width, min(y0 + rng.uniform(-6, 14), height - reach), side)
    for j, (cx, cy) in enumerate(((width - 12, 0.8 * height), (0.85 * width, height - 12), (width - 10, height - 10))):
        paste(ids[2 * n_band + j], cx, cy, float(rng.uniform(34, 52)))
    if noise_sigma > 0:
        frame = np.clip(np.rint(frame + rng.normal(0, noise_sigma, frame.shape)), 0, 255).astype(np.uint8)
    return frame


def make_sequence(bytes_list, base_seed: int, n_frames: int, width: int = 3840, height: int = 2160,
                  noise_sigma: float = 3.0, leds=None, events=None):
    """Sparse sequence (ids 1,2,3 = vehicles, 4 = host) with slow drift so that the track gating of
    aruco_detect.py:613 passes.  Frame k uses seed base_seed + k.  Yields frames.
    events (optional): {frame index: {"hide": [ids not drawn in that frame], "jump": {id: (dx, dy)}}} -- a jump is a
    persistent teleport from that frame on (further than DIFF_MAX of aruco_detect.py:524), a hidden marker simply is not
    rendered; together they drive the gating / relabel branches of aruco_detect.py:613,637,669."""
    rng = np.random.default_rng(base_seed)
    start = np.array([[0.30, 0.35], [0.55, 0.30], [0.70, 0.60], [0.45, 0.65]]) * [width, height]
    start += rng.uniform(-0.04, 0.04, size=start.shape) * [width, height]
    vel = rng.uniform(-1.5, 1.5, size=start.shape)  # px / frame
    ang = rng.uniform(0, 2 * np.pi, size=4)
    all_ids = (1, 2, 3, 4)
    offset = np.zeros_like(start)
    for k in range(n_frames):
        ev = (events or {}).get(k, {})
        for mid, (dx, dy) in ev.get("jump", {}).items():
            offset[all_ids.index(int(mid))] += (dx, dy)
        centers = start + vel * k + offset
        keep = [i for i, mid in enumerate(all_ids) if mid not in ev.get("hide", ())]
        yield make_frame(bytes_list, base_seed + k, width, height, ids=tuple(all_ids[i] for i in keep), side_range=(64, 66),
                         jitter=0.01, noise_sigma=noise_sigma, centers=[centers[i].tolist() for i in keep],
                         angles=[float(ang[i]) for i in keep], leds=None if leds is None else leds[k % len(leds)])


def make_inverted_frame(bytes_list, seed: int, width: int = 1920, height: int = 1080, n_markers: int = 6, noise_sigma: float = 3.0):
    """Every other marker as a WHITE marker on a black quiet zone (detectInvertedMarker of cv2's DetectorParameters): random ids,
    side 40-100 px, rotation + corner jitter, Gaussian noise.  Returns the frame."""
    rng = np.random.default_rng(seed)
    frame = background(rng, width, height)
    placed = []
    for k in range(n_markers):
        side = float(rng.uniform(40, 100))
        for _ in range(200):
            cx, cy = float(rng.uniform(90, width - 90)), float(rng.uniform(90, height - 90))
            if all((cx - px) ** 2 + (cy - py) ** 2 > (1.1 * (side + ps)) ** 2 for px, py, ps in placed):
                break
        else:
            continue
        placed.append((cx, cy, side))
        quad = _random_quad(rng, cx, cy, side, 0.06)
        tile = render_marker(bytes_list, int(rng.integers(0, 50)))
        if k % 2 == 0:
            tile = 255 - tile
        _paste_marker(frame, tile, quad, quiet_frac=8.0 / tile.shape[0])
    noise = rng.normal(0.0, noise_sigma, size=frame.shape).astype(np.float32)
    return np.clip(np.rint(frame.astype(np.float32) + noise), 0, 255).astype(np.uint8)


def make_grid_frame(bytes_list, n: int, pitch: int = 64, side: int = 30, rotate: float = 0.0, seed: int = 0,
                    width: int = 3840, height: int = 2160, noise_sigma: float = 2.0):
    """Gray frame (uint8 HxW) with n markers on a grid (row by row, `pitch` px apart, ids 0..49 cycled) over a flat background of
    128: many candidates per frame.  Every tile is rendered at its on-frame size (side px, quiet zone side // 6).  rotate = 0:
    tiles pasted axis-aligned, every marker has the same perimeter; rotate > 0: each marker turned by a random angle of
    rotate / 4 to rotate radians either way and shrunk by up to 15 % (distinct perimeters).  Raises if the grid holds fewer
    than n markers."""
    rng = np.random.default_rng(seed)
    frame = np.full((height, width, 1), 128, np.uint8)
    quiet = max(2, side // 6)
    k = 0
    for cy in range(pitch // 2 + 8, height - pitch // 2, pitch):
        for cx in range(pitch // 2 + 8, width - pitch // 2, pitch):
            if k >= n:
                break
            tile = render_marker(bytes_list, k % 50, side_px=side, quiet_px=quiet)
            if rotate > 0:
                # not near 0 (a marker turned by a few hundredths of a radian still fits to an axis-aligned quad), and a size
                # that varies too (markers turned by +a and -a have the same perimeter)
                a = rng.uniform(0.25, 1.0) * rotate * rng.choice((-1.0, 1.0))
                c, s = np.cos(a), np.sin(a)
                half = rng.uniform(0.85, 1.0) * side / 2
                quad = np.float32([[-1, -1], [1, -1], [1, 1], [-1, 1]]) * half @ np.float32([[c, s], [-s, c]]) + np.float32([cx, cy])
                _paste_marker(frame, tile, quad, quiet_frac=quiet / tile.shape[0])
            else:
                y0, x0 = cy - tile.shape[0] // 2, cx - tile.shape[1] // 2
                frame[y0:y0 + tile.shape[0], x0:x0 + tile.shape[1], 0] = tile
            k += 1
    if k < n:
        raise ValueError(f"a {width}x{height} grid of pitch {pitch} holds {k} markers, not {n}")
    frame = frame[..., 0]
    if noise_sigma > 0:
        frame = np.clip(np.rint(frame + rng.normal(0, noise_sigma, frame.shape)), 0, 255).astype(np.uint8)
    return frame


def make_big_marker_frame(bytes_list, side: int, seed: int = 1, marker_id: int = 7, width: int = 3840, height: int = 2160,
                          jitter: float = 0.03, noise_sigma: float = 3.0):
    """BGR frame with ONE marker of about `side` px (rotated, corner jitter) in the middle of the textured background: boundary
    clusters of thousands of points.  The tile is rendered sharp at its on-frame size (side // 6 * 6 px, quiet zone side // 12):
    a small tile upscaled by the warp would have ramped edges, which neither cv2 nor the oracle detects at these sizes."""
    rng = np.random.default_rng(seed)
    frame = background(rng, width, height)
    quiet = side // 12
    tile = render_marker(bytes_list, marker_id, side_px=side // 6 * 6, quiet_px=quiet)
    quad = _random_quad(rng, width / 2, height / 2, side, jitter)
    _paste_marker(frame, tile, quad, quiet_frac=quiet / tile.shape[0])
    if noise_sigma > 0:
        frame = np.clip(np.rint(frame + rng.normal(0, noise_sigma, frame.shape)), 0, 255).astype(np.uint8)
    return frame
