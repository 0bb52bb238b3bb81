"""Rectification remap (DESIGN.md §14) on the CPU: a numpy reference of the rule, held bit for bit against cv2.remap
(INTER_LINEAR, BORDER_CONSTANT 0, CV_32FC1 maps) where OpenCV imports, and the quality it buys through the CPU oracle on
a rig with rotated cameras (synthetic.make_unrectified_pair)."""
import numpy as np
import pytest

from oracle import oracle as O
from stereo_depth_b200.synthetic import make_pair, make_unrectified_pair


def reference_remap(src, map_x, map_y):
    """The rule of DESIGN.md §14 for every [H,W] plane of a [..., H, W] uint8 or float32 array; the output has the
    maps' shape in its last two axes."""
    src = np.asarray(src)
    H, W = src.shape[-2:]

    def taps(v):
        v32 = v.astype(np.float32) * np.float32(32)
        nan = np.isnan(v32)
        i = np.clip(np.rint(np.where(nan, 0, v32).astype(np.float64)), -2.0 ** 31, 2.0 ** 31 - 1).astype(np.int64)
        return i >> 5, i & 31, nan

    x0, fx, nan_x = taps(map_x)
    y0, fy, nan_y = taps(map_y)
    one, ax, ay = np.float32(1), fx.astype(np.float32) / np.float32(32), fy.astype(np.float32) / np.float32(32)
    c = [(one - ay) * (one - ax), (one - ay) * ax, ay * (one - ax), ay * ax]
    vals = []
    for ty, tx in ((y0, x0), (y0, x0 + 1), (y0 + 1, x0), (y0 + 1, x0 + 1)):
        inside = (tx >= 0) & (tx < W) & (ty >= 0) & (ty < H) & ~nan_x & ~nan_y
        vals.append(np.where(inside, src[..., np.where(inside, ty, 0), np.where(inside, tx, 0)], 0))
    if src.dtype == np.uint8:
        w = [np.rint(ci.astype(np.float64) * 32768).astype(np.int64) for ci in c]
        largest = np.argmax(np.stack(c), axis=0)            # first on ties
        diff = 32768 - sum(w)
        w = [w[k] + np.where(largest == k, diff, 0) for k in range(4)]
        acc = sum(w[k] * vals[k].astype(np.int64) for k in range(4))
        return np.clip((acc + (1 << 14)) >> 15, 0, 255).astype(np.uint8)
    assert src.dtype == np.float32
    v = [x.astype(np.float32) for x in vals]
    return ((c[0] * v[0] + c[1] * v[1]) + c[2] * v[2]) + c[3] * v[3]


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and bool((a.view(np.uint8) == b.view(np.uint8)).all())


# ---- maps that reach every clause of the rule (shared with the GPU tests) ----------------------------------------------

def fraction_maps(H, W, x0=5, y0=7):
    """[32,32] maps whose entry (j, i) is (x0 + i/32, y0 + j/32): all 1024 fraction pairs."""
    i = np.arange(32, dtype=np.float32) / np.float32(32)
    return np.broadcast_to(np.float32(x0) + i[None, :], (32, 32)).copy(), \
        np.broadcast_to(np.float32(y0) + i[:, None], (32, 32)).copy()


SPECIAL = np.float32([np.nan, np.inf, -np.inf, 1e30, -1e30, 40000, -40000, 32767.5, -32768.5, 0.0, -0.0, -0.5, -1.0,
                      -1.01, -1 / 64, 1 / 64, 3 / 64])


def special_maps(H, W):
    """[H,W] maps mixing pathological values, taps that straddle every border, exact half-way ties (x*32 ending in .5)
    and random coordinates reaching past every edge."""
    rng = np.random.default_rng(H * 7919 + W)
    mx = rng.uniform(-3, W + 2, (H, W)).astype(np.float32)
    my = rng.uniform(-3, H + 2, (H, W)).astype(np.float32)
    edges_x = np.float32([-1, -0.5, -1 / 32, 0, W - 1, W - 1 + 1 / 32, W - 0.5, W - 1 / 64, W, W + 0.5])
    edges_y = np.float32([-1, -0.5, -1 / 32, 0, H - 1, H - 1 + 1 / 32, H - 0.5, H - 1 / 64, H, H + 0.5])
    k = rng.random((H, W))
    mx = np.where(k < 0.15, rng.choice(edges_x, (H, W)), mx)
    my = np.where((k > 0.1) & (k < 0.25), rng.choice(edges_y, (H, W)), my)
    ties = (np.floor(rng.uniform(-2, W + 1, (H, W)) * 32) + 0.5) / 32
    mx = np.where((k > 0.25) & (k < 0.35), ties, mx).astype(np.float32)
    tiesy = (np.floor(rng.uniform(-2, H + 1, (H, W)) * 32) + 0.5) / 32
    my = np.where((k > 0.3) & (k < 0.4), tiesy, my).astype(np.float32)
    s = rng.random((H, W))
    mx = np.where(s < 0.05, rng.choice(SPECIAL, (H, W)), mx).astype(np.float32)
    my = np.where((s > 0.03) & (s < 0.08), rng.choice(SPECIAL, (H, W)), my).astype(np.float32)
    return mx, my


def stereo_rectify_maps(H, W):
    """Maps of a realistic rig: cv2.stereoRectify of two cameras with lens distortion and a small relative rotation,
    then cv2.initUndistortRectifyMap(..., m1type=cv2.CV_32FC1)."""
    import cv2
    f = 0.9 * W
    K1 = np.array([[f, 0, W / 2 + 3.5], [0, f * 1.01, H / 2 - 2.25], [0, 0, 1]])
    K2 = np.array([[f * 0.99, 0, W / 2 - 4.0], [0, f, H / 2 + 1.5], [0, 0, 1]])
    d1 = np.array([-0.12, 0.05, 0.001, -0.0005, 0.0])
    d2 = np.array([-0.10, 0.03, -0.0008, 0.0004, 0.0])
    R, _ = cv2.Rodrigues(np.array([0.01, -0.02, 0.005]))
    T = np.array([-0.12, 0.002, 0.001])
    R1, R2, P1, P2, _, _, _ = cv2.stereoRectify(K1, d1, K2, d2, (W, H), R, T, alpha=0)
    lm = cv2.initUndistortRectifyMap(K1, d1, R1, P1, (W, H), cv2.CV_32FC1)
    rm = cv2.initUndistortRectifyMap(K2, d2, R2, P2, (W, H), cv2.CV_32FC1)
    return lm, rm


def cv2_remap(src, mx, my):
    """cv2.remap of every [H,W] plane of a [..., H, W] array."""
    import cv2
    flat = src.reshape((-1,) + src.shape[-2:])
    out = [cv2.remap(p, mx, my, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0) for p in flat]
    return np.stack(out).reshape(src.shape[:-2] + mx.shape)


def images(shape, dtype, seed):
    rng = np.random.default_rng(seed)
    if dtype == np.uint8:
        return rng.integers(0, 256, shape, dtype=np.uint8)
    return (rng.standard_normal(shape) * 100).astype(np.float32)   # non-integer values: the order of the sum matters


# ---- the reference alone --------------------------------------------------------------------------------------------

@pytest.mark.parametrize("dtype", [np.uint8, np.float32])
def test_identity_and_integer_shift(dtype):
    img = images((3, 20, 30), dtype, 1)
    cols, rows = np.meshgrid(np.arange(30, dtype=np.float32), np.arange(20, dtype=np.float32))
    assert same_bits(reference_remap(img, cols, rows), img)
    shifted = reference_remap(img, cols + 2, rows - 1)
    want = np.zeros_like(img)
    want[:, 1:, :28] = img[:, :19, 2:]
    assert same_bits(shifted, want)


def test_nan_and_far_coordinates_read_zero_and_weights_sum_to_one():
    img = np.full((1, 8, 8), 255, np.uint8)
    mx = np.float32([[np.nan, 3, np.inf, -np.inf, 1e30, 40000, 3.5, 7.5]])
    my = np.float32([[3, np.nan, 3, 3, 3, 3, 3.5, 3]])
    got = reference_remap(img, mx, my)[0, 0]
    assert list(got[:6]) == [0] * 6
    assert got[6] == 255                         # four inside taps: the weights sum to one
    assert got[7] == 128                         # (255 * 16384 + 16384) >> 15: right tap outside keeps its weight
    f = reference_remap(img.astype(np.float32), mx, my)[0, 0]
    assert list(f[:6]) == [0.0] * 6 and f[6] == 255.0 and f[7] == 127.5


# ---- bit for bit against OpenCV ----------------------------------------------------------------------------------------

@pytest.fixture
def cv2():
    return pytest.importorskip("cv2")


@pytest.mark.parametrize("dtype", [np.uint8, np.float32])
def test_every_fraction_pair(cv2, dtype):
    for seed in range(4):
        img = images((3, 40, 50), dtype, seed)
        if seed == 0 and dtype == np.uint8:
            img[:] = 255                                       # largest sums
        mx, my = fraction_maps(40, 50, x0=5 + seed, y0=7 + seed)
        assert same_bits(reference_remap(img, mx, my), cv2_remap(img, mx, my)), seed


@pytest.mark.parametrize("dtype", [np.uint8, np.float32])
@pytest.mark.parametrize("H,W", [(1, 1), (1, 17), (9, 1), (31, 45), (64, 64)])
def test_pathological_maps(cv2, dtype, H, W):
    img = images((2, H, W), dtype, H + W)
    mx, my = special_maps(H, W)
    assert same_bits(reference_remap(img, mx, my), cv2_remap(img, mx, my))


def test_special_values_on_both_axes(cv2):
    img = images((3, 33, 35), np.uint8, 3)
    a, b = np.meshgrid(SPECIAL, SPECIAL)
    for mx, my in ((a, b), (b, a), (a + 0, np.full_like(a, 4.25)), (np.full_like(a, 4.25), a + 0)):
        mx, my = np.ascontiguousarray(mx, np.float32), np.ascontiguousarray(my, np.float32)
        assert same_bits(reference_remap(img, mx, my), cv2_remap(img, mx, my))
        f = img.astype(np.float32) + np.float32(0.375)
        assert same_bits(reference_remap(f, mx, my), cv2_remap(f, mx, my))


@pytest.mark.parametrize("dtype", [np.uint8, np.float32])
def test_realistic_stereo_rectify_maps(cv2, dtype):
    H, W = 120, 200
    lm, rm = stereo_rectify_maps(H, W)
    for (mx, my), seed in ((lm, 1), (rm, 2)):
        assert mx.dtype == np.float32 and mx.shape == (H, W)
        img = images((3, H, W), dtype, seed)
        assert same_bits(reference_remap(img, mx, my), cv2_remap(img, mx, my))


def test_unrectified_pair_maps_are_what_opencv_computes(cv2):
    """make_unrectified_pair's maps equal cv2.initUndistortRectifyMap for its rig (no distortion) to float rounding."""
    H, W = 60, 80
    _, _, (lm, rm), _ = make_unrectified_pair(H, W, 16, degrees=1.0)
    Kc = np.array([[W, 0, (W - 1) / 2], [0, W, (H - 1) / 2], [0, 0, 1]], np.float64)
    a = np.deg2rad(1.0)
    from stereo_depth_b200.synthetic import _rotation
    for (mx, my), sign in ((lm, 1.0), (rm, -1.0)):
        R = _rotation(sign * a, sign * a / 2)
        # initUndistortRectifyMap's R maps raw camera rays to rectified ones: the inverse of the view's rotation
        ox, oy = cv2.initUndistortRectifyMap(Kc, None, R.T, Kc, (W, H), cv2.CV_32FC1)
        assert np.abs(ox - mx).max() < 1e-3 and np.abs(oy - my).max() < 1e-3


# ---- what rectification buys, through the CPU oracle ------------------------------------------------------------------

def within_one(out, gt):
    """Fraction of the central 80 % (rows and columns) of pixels with |out - gt| <= 1."""
    H, W = gt.shape
    m = np.zeros((H, W), bool)
    m[H // 10:H - H // 10, W // 10:W - W // 10] = True
    return float((np.abs(out - gt)[m] <= 1).mean())


def test_rectified_raw_pair_is_nearly_as_good_as_a_rectified_rig():
    H, W, D = 160, 256, 48
    kw = dict(height=H, width=W, downscale_factor=2, min_disparity=0, max_disparity=D - 1)
    cfg = O.make_config(**kw)
    lraw, rraw, (lm, rm), gt = make_unrectified_pair(H, W, D, seed=5)
    l, r, gt2 = make_pair(H, W, D, seed=5)
    assert (gt == gt2).all()
    direct = within_one(O.run(cfg, l, r)["out"], gt)
    rectified = within_one(O.run(cfg, reference_remap(lraw, *lm), reference_remap(rraw, *rm))["out"], gt)
    raw = within_one(O.run(cfg, lraw, rraw)["out"], gt)
    # measured: 0.803 rectified rig, 0.817 raw pair rectified, 0.075 raw pair as is
    assert direct > 0.75
    assert rectified >= direct - 0.03, (rectified, direct)
    assert raw < 0.3, raw
