"""Synthetic random-dot stereo pairs (the workload BASELINE.json's configs are quoted on).

The matching convention is the reference's: a left pixel at column c corresponds to the right
pixel at column c - disparity (device_functions.cuh:68), so right[:, r, c] = left[:, r, c + g[r, c]].
Deterministic per (seed, frame index); numpy only (no GPU, no oracle).
"""
import numpy as np


def ground_truth(H, W, D, rng):
    """Piecewise-constant disparity in [D/16, 3D/4] with one horizontally slanted ramp."""
    g = np.full((H, W), max(1, D // 8), np.int32)
    lo, hi = max(1, D // 16), max(2, (3 * D) // 4)
    for _ in range(6):
        h = int(rng.integers(max(2, H // 8), max(3, H // 2)))
        w = int(rng.integers(max(2, W // 8), max(3, W // 2)))
        r0 = int(rng.integers(0, max(1, H - h)))
        c0 = int(rng.integers(0, max(1, W - w)))
        g[r0:r0 + h, c0:c0 + w] = int(rng.integers(lo, hi + 1))
    # slanted region: 1 px of disparity per 16 columns -> odd disparities, sub-pixel coverage
    h, w = max(2, H // 4), max(2, W // 3)
    r0 = int(rng.integers(0, max(1, H - h)))
    c0 = int(rng.integers(0, max(1, W - w)))
    ramp = lo + (np.arange(w, dtype=np.int32) // 16) % max(1, hi - lo)
    g[r0:r0 + h, c0:c0 + w] = ramp[None, :]
    return g


def make_pair(H, W, D, seed=1234, frame=0):
    """Returns (left u8 [3,H,W], right u8 [3,H,W], gt int32 [H,W])."""
    rng = np.random.default_rng(seed + frame)
    left = rng.integers(0, 256, (3, H, W), dtype=np.uint8)
    g = ground_truth(H, W, D, rng)
    cols = np.arange(W, dtype=np.int64)[None, :] + g
    valid = cols < W
    src = np.where(valid, cols, 0)
    right = np.take_along_axis(left, np.broadcast_to(src[None], (3, H, W)), axis=2)
    fresh = rng.integers(0, 256, (3, H, W), dtype=np.uint8)
    right = np.where(valid[None], right, fresh)
    noise = rng.integers(-2, 3, (3, H, W), dtype=np.int16)
    right = np.clip(right.astype(np.int16) + noise, 0, 255).astype(np.uint8)
    return left, right, g


def make_layered_pair(H, W, D, seed=1234):
    """A physically consistent scene for occlusion studies: fronto-parallel rectangles defined in the LEFT view over a
    background at the smallest disparity, a larger disparity being nearer and drawn on top.  The right view is the
    left one forward-warped (left column c -> right column c - d) with a z-buffer: where several left pixels land on
    one right pixel the nearest wins.  Right pixels no left pixel reaches get fresh noise, and every right pixel gets
    +-2 of noise.  Returns (left u8 [3,H,W], right u8 [3,H,W], gt_left float32 [H,W], visible bool [H,W]); visible is
    False for left pixels that are occluded in the right view or land outside it."""
    rng = np.random.default_rng(seed)
    left = rng.integers(0, 256, (3, H, W), dtype=np.uint8)
    lo, hi = max(1, D // 16), max(2, (3 * D) // 4)
    gt = np.full((H, W), lo, np.int64)
    layers = []
    for _ in range(8):
        h = int(rng.integers(max(2, H // 8), max(3, H // 2)))
        w = int(rng.integers(max(2, W // 10), max(3, W // 3)))
        r0 = int(rng.integers(0, max(1, H - h)))
        c0 = int(rng.integers(0, max(1, W - w)))
        layers.append((int(rng.integers(lo + 1, hi + 1)), r0, h, c0, w))
    for d, r0, h, c0, w in sorted(layers):   # far to near
        gt[r0:r0 + h, c0:c0 + w] = d
    rows = np.broadcast_to(np.arange(H)[:, None], (H, W))
    target = np.arange(W)[None, :] - gt
    inside = target >= 0
    zbuf = np.full((H, W), -1, np.int64)
    np.maximum.at(zbuf, (rows[inside], target[inside]), gt[inside])
    visible = inside & (zbuf[rows, np.where(inside, target, 0)] == gt)
    right = rng.integers(0, 256, (3, H, W), dtype=np.uint8)
    right[:, rows[visible], target[visible]] = left[:, rows[visible], np.nonzero(visible)[1]]
    noise = rng.integers(-2, 3, (3, H, W), dtype=np.int16)
    right = np.clip(right.astype(np.int16) + noise, 0, 255).astype(np.uint8)
    return left, right, gt.astype(np.float32), visible


def _bilinear(img, x, y):
    """float32 [C,H,W] image sampled at float coordinates x, y ([H',W']); zero outside."""
    C, H, W = img.shape
    x0, y0 = np.floor(x).astype(np.int64), np.floor(y).astype(np.int64)
    ax, ay = (x - x0).astype(np.float32), (y - y0).astype(np.float32)
    out = np.zeros((C,) + x.shape, np.float32)
    for dy, dx, w in ((0, 0, (1 - ay) * (1 - ax)), (0, 1, (1 - ay) * ax), (1, 0, ay * (1 - ax)), (1, 1, ay * ax)):
        yy, xx = y0 + dy, x0 + dx
        inside = (yy >= 0) & (yy < H) & (xx >= 0) & (xx < W)
        out += np.where(inside, img[:, np.clip(yy, 0, H - 1), np.clip(xx, 0, W - 1)], 0) * w
    return out


def _rotation(pitch, roll):
    cp, sp, cr, sr = np.cos(pitch), np.sin(pitch), np.cos(roll), np.sin(roll)
    about_x = np.array([[1, 0, 0], [0, cp, -sp], [0, sp, cp]])
    about_z = np.array([[cr, -sr, 0], [sr, cr, 0], [0, 0, 1]])
    return about_z @ about_x


def make_unrectified_pair(H, W, D, seed=1234, degrees=1.0):
    """A make_pair scene as a stereo rig whose cameras are slightly rotated about their optical centres: the left camera
    by +degrees of pitch and +degrees/2 of roll, the right one by the opposite.  Focal length W pixels, principal point
    at the image centre.  A rotation about the optical centre maps the rectified image by the homography
    Hm = Kc R Kc^-1 (rectified pixel -> raw pixel), so the raw views are the rectified ones resampled (bilinear, zero
    outside) at Hm^-1, and the rectification maps are Hm itself -- what cv2.initUndistortRectifyMap gives for such a rig
    without lens distortion.  Returns (left_raw u8 [3,H,W], right_raw u8 [3,H,W],
    ((left map_x, left map_y), (right map_x, right map_y)) float32 [H,W] each, gt int32 [H,W] in rectified left
    coordinates)."""
    left, right, gt = make_pair(H, W, D, seed)
    raws = []
    for img, (Hm, pix) in zip((left, right), _rotated_rig(H, W, degrees)):
        q = np.einsum("ij,jhw->ihw", np.linalg.inv(Hm), pix)
        raw = _bilinear(img.astype(np.float32), q[0] / q[2], q[1] / q[2])
        raws.append(np.clip(np.rint(raw), 0, 255).astype(np.uint8))
    return raws[0], raws[1], rotated_rig_maps(H, W, degrees), gt


def _rotated_rig(H, W, degrees):
    """(homography rectified -> raw pixel, homogeneous pixel grid [3,H,W]) of the left and the right camera."""
    f = float(W)
    Kc = np.array([[f, 0, (W - 1) / 2], [0, f, (H - 1) / 2], [0, 0, 1]])
    a = np.deg2rad(degrees)
    cols, rows = np.meshgrid(np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64))
    pix = np.stack([cols, rows, np.ones_like(cols)])
    return [(Kc @ _rotation(s * a, s * a / 2) @ np.linalg.inv(Kc), pix) for s in (1.0, -1.0)]


def rotated_rig_maps(H, W, degrees=1.0):
    """The rectification maps of make_unrectified_pair's rig without rendering its views:
    ((left map_x, left map_y), (right map_x, right map_y)), float32 [H,W] each."""
    out = []
    for Hm, pix in _rotated_rig(H, W, degrees):
        p = np.einsum("ij,jhw->ihw", Hm, pix)
        out.append(((p[0] / p[2]).astype(np.float32), (p[1] / p[2]).astype(np.float32)))
    return out[0], out[1]


def make_batch(n, H, W, D, seed=1234, first_frame=0):
    ls, rs = [], []
    for f in range(n):
        l, r, _ = make_pair(H, W, D, seed, first_frame + f)
        ls.append(l)
        rs.append(r)
    return np.stack(ls), np.stack(rs)


def natural_pair_path():
    import os
    return os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "data", "_ref", "natural_pair.npz")


def load_natural_pair():
    """The one natural stereo pair the reference ships (src/python/data/im0.png, im1.png, calib.txt: 1920x1080,
    vmin=75, vmax=262), as extracted by oracle/make_natural.py into the git-ignored data/_ref/.  Returns
    (left u8 [3,H,W], right u8 [3,H,W], vmin, vmax) or None when the file is not there."""
    import os
    p = natural_pair_path()
    if not os.path.exists(p):
        return None
    z = np.load(p)
    return z["left"], z["right"], int(z["vmin"]), int(z["vmax"])
