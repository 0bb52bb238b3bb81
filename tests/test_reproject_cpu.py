"""Reprojection to 3-D (DESIGN.md §15) on the CPU: a numpy reference of cv2.reprojectImageTo3D's rule, held bit for bit
against OpenCV where it imports -- random and crafted Q matrices, special disparity values, handleMissingValues, the Q
of cv2.stereoRectify, a float32 Q, degenerate sizes -- and the one deliberate deviation: the minimum of a map with NaN
is the minimum over its non-NaN values."""
import numpy as np
import pytest

FLT_EPS = float(np.finfo(np.float32).eps)


def reference_reproject(disp, Q, handle_missing=False):
    """The rule of DESIGN.md §15: disp float32 [H,W] -> float32 [H,W,3].  The minimum starts at FLT_MAX, as in OpenCV,
    so a disparity of exactly FLT_MAX gets Z = 10000 with handle_missing off too."""
    disp = np.asarray(disp, np.float32)
    H, W = disp.shape
    q = np.asarray(Q, np.float64)
    X = np.broadcast_to(np.arange(W, dtype=np.float64)[None], (H, W))
    Y = np.broadcast_to(np.arange(H, dtype=np.float64)[:, None], (H, W))
    D = disp.astype(np.float64)
    with np.errstate(all="ignore"):
        h = [((((0.0 + q[k, 0] * X) + q[k, 1] * Y) + q[k, 2] * D) + q[k, 3]) for k in range(4)]
        ia = 1.0 / h[3]
        out = np.stack([(h[k].astype(np.float32).astype(np.float64) * ia).astype(np.float32) for k in range(3)], -1)
        m = float(np.finfo(np.float32).max)
        if handle_missing and not np.isnan(disp).all():
            m = float(np.nanmin(disp))
        out[..., 2][np.abs(D - m) <= FLT_EPS] = np.float32(10000.0)
    return out


def reference_reproject_batch(disp, Q, handle_missing=False):
    """[N,H,W] -> [N,H,W,3], each frame with its own minimum."""
    return np.stack([reference_reproject(d, Q, handle_missing) for d in disp])


def cv2_reproject(disp, Q, handle_missing=False):
    import cv2
    return cv2.reprojectImageTo3D(np.ascontiguousarray(disp, np.float32), np.asarray(Q), handleMissingValues=handle_missing)


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and bool((a.view(np.uint8) == b.view(np.uint8)).all())


# ---- inputs that reach every clause of the rule (shared with the GPU tests) --------------------------------------------

DENORMALS = np.array([1, 0x7fffff, 0x400000, 0x80000001, 0x807fffff], np.uint32).view(np.float32)
SPECIAL = np.concatenate([np.float32([0.0, -0.0, np.inf, -np.inf, 3e38, -3e38, 3.4028235e38, 1.0, -1.0, 0.5, 127.75,
                                      1e-30, -1e-30]), DENORMALS])


def near_minimum(m):
    """Float32 values within FLT_EPSILON of m and just outside it, on both sides (the handleMissingValues boundary)."""
    m = np.float32(m)
    out = [m]
    for sign in (1.0, -1.0):
        edge = np.float32(float(m) + sign * FLT_EPS)           # nearest float32 to the boundary
        for v in (edge, np.nextafter(edge, np.float32(sign * np.inf)), np.nextafter(edge, np.float32(-sign * np.inf))):
            if v > m or sign < 0:
                out.append(np.float32(v))
    return np.float32(out)


def special_map(H, W, seed, nan=False, minimum=0.25):
    """A disparity map of random values in [minimum, 200) with special values, values at and around the minimum's
    FLT_EPSILON boundary, and (nan=True) NaNs scattered over it."""
    rng = np.random.default_rng(seed)
    d = (rng.random((H, W)) * 200 + minimum).astype(np.float32)
    flat = d.ravel()
    k = rng.random(flat.size) < 0.05
    flat[k] = rng.choice(SPECIAL, int(k.sum()))
    vals = near_minimum(minimum)
    k = rng.random(flat.size) < 0.05
    flat[k] = rng.choice(vals, int(k.sum()))
    if nan:
        flat[rng.random(flat.size) < 0.03] = np.nan
    return d


def random_q(rng, scale):
    """A dense random Q at `scale`, with some entries set to +-0 and some rows shaped like stereoRectify's."""
    q = (rng.standard_normal((4, 4)) * scale).astype(np.float64)
    k = rng.random((4, 4)) < 0.2
    q[k] = rng.choice([0.0, -0.0], int(k.sum()))
    return q


def crafted_qs():
    """Q matrices built to give signed zeros, overflow of float32(h_k) (1e300 entries) and h_3 = 0."""
    return [
        np.array([[-1, -1, -1, -0.0], [-1, -1, -1, -0.0], [0, 0, -1, -0.0], [0, 0, 0, 1.0]]),     # -0 sums -> +0
        np.array([[-0.0, -0.0, -0.0, -0.0], [-0.0, -0.0, -0.0, -0.0], [-0.0, -0.0, -0.0, -0.0], [0, 0, 0, 1.0]]),
        np.array([[1e300, 1, 1, 0], [0, 1e300, 0, 0], [0, 0, 1e10, 1], [0, 0, 1e-300, 1]]),       # overflow to +-inf
        np.array([[-1e300, 1, 1, 0], [0, 1, -1e300, 0], [0, 0, 1, 1e300], [0, 0, -1e300, 1]]),
        np.array([[1, 0, 0, -5], [0, 1, 0, -3], [0, 0, 0, 100], [0, 0, 0, 0]]),                   # h_3 = 0: inf / NaN
        np.array([[1, 0, 0, -5], [0, 1, 0, -3], [0, 0, 0, 100], [0, 0, 1, 0]]),                   # h_3 = d (d = +-0)
        np.array([[1e-8, 0, 0, 0], [0, 1e-8, 0, 0], [0, 0, 1e-8, 0], [0, 0, 1e30, 1]]),            # denormal outputs
    ]


def stereo_rectify_q(H, W, zero_disparity):
    """Q of cv2.stereoRectify for a rig with lens distortion and a small relative rotation; without
    CALIB_ZERO_DISPARITY the rectified principal points differ, so Q[3][3] != 0."""
    import cv2
    f = 1.1 * W
    K1 = np.array([[f, 0, W / 2 - 7.3], [0, f * 1.001, H / 2 + 4.1], [0, 0, 1]])
    K2 = np.array([[f * 0.998, 0, W / 2 + 5.2], [0, f, H / 2 - 3.3], [0, 0, 1]])
    d1, d2 = np.array([-0.12, 0.05, 0.001, -0.0007, 0.0]), np.array([-0.1, 0.04, -0.0005, 0.0009, 0.0])
    R, _ = cv2.Rodrigues(np.array([0.01, -0.02, 0.005]))
    T = np.array([-0.12, 0.002, 0.001])
    flags = cv2.CALIB_ZERO_DISPARITY if zero_disparity else 0
    Q = cv2.stereoRectify(K1, d1, K2, d2, (W, H), R, T, flags=flags, alpha=0)[4]
    return Q


# ---- the rule against OpenCV --------------------------------------------------------------------------------------------

@pytest.fixture
def cv2():
    return pytest.importorskip("cv2")


@pytest.mark.parametrize("scale", [1e-3, 0.1, 1.0, 13.0, 700.0])
@pytest.mark.parametrize("handle_missing", [False, True])
def test_random_q_over_scales(cv2, scale, handle_missing):
    rng = np.random.default_rng(int(scale * 1000) + handle_missing)
    for i in range(6):
        Q = random_q(rng, scale)
        if i == 5:                       # one huge entry per row
            Q[np.arange(4), rng.integers(0, 4, 4)] = rng.choice([1e300, -1e300], 4)
        d = special_map(37, 53, seed=i, minimum=float(rng.choice([0.25, 1.0, -3.5, 1e-8])))
        assert same_bits(reference_reproject(d, Q, handle_missing), cv2_reproject(d, Q, handle_missing)), (scale, i)


@pytest.mark.parametrize("handle_missing", [False, True])
def test_crafted_q_signed_zeros_overflow_and_zero_w(cv2, handle_missing):
    d = np.concatenate([SPECIAL, near_minimum(0.0), near_minimum(2.0)]).reshape(1, -1)
    d = np.concatenate([d, d[:, ::-1], -d], 0)
    for Q in crafted_qs():
        got = reference_reproject(d, Q, handle_missing)
        assert same_bits(got, cv2_reproject(d, Q, handle_missing)), Q
    # the leading `0 +`: all-zero terms sum to +0, never -0
    got = reference_reproject(np.float32([[0.0, -0.0, 5.0]]), crafted_qs()[1])
    assert (got == 0).all() and not np.signbit(got).any()


def test_denormal_outputs_are_kept(cv2):
    d = np.float32([[1e-30, 3e-39, 1.0, 0.5]])
    Q = crafted_qs()[-1]
    got = reference_reproject(d, Q)
    tiny = (np.abs(got) < np.finfo(np.float32).tiny) & (got != 0)
    assert tiny.any()
    assert same_bits(got, cv2_reproject(d, Q))


@pytest.mark.parametrize("minimum", [0.0, -0.0, 1.0, 1e-8, 63.0, -2.0, 3e38])
def test_missing_values_boundary(cv2, minimum):
    vals = near_minimum(minimum)
    d = np.concatenate([vals, np.float32([minimum + 10, 3e38])]).reshape(1, -1)
    Q = np.array([[1, 0, 0, -10.5], [0, 1, 0, -7.25], [0, 0, 0, 500.0], [0, 0, 0.1, 0]])
    got = reference_reproject(d, Q, True)
    assert same_bits(got, cv2_reproject(d, Q, True))
    inside = np.abs(d.astype(np.float64) - float(d.min())) <= FLT_EPS
    assert inside.sum() >= (2 if abs(minimum) <= 1 else 1)     # (above 1 no other float32 lies that close)
    assert (got[..., 2][inside] == 10000).all()


@pytest.mark.parametrize("zero_disparity", [True, False])
@pytest.mark.parametrize("handle_missing", [False, True])
def test_stereo_rectify_q_at_1080p(cv2, zero_disparity, handle_missing):
    H, W = 1080, 1920
    Q = stereo_rectify_q(H, W, zero_disparity)
    assert (Q[3, 3] == 0) == zero_disparity
    d = special_map(H, W, seed=5)
    assert same_bits(reference_reproject(d, Q, handle_missing), cv2_reproject(d, Q, handle_missing))


def test_float32_q(cv2):
    Q = stereo_rectify_q(480, 640, False).astype(np.float32)
    d = special_map(48, 64, seed=6)
    for hm in (False, True):
        assert same_bits(reference_reproject(d, Q, hm), cv2_reproject(d, Q, hm))


@pytest.mark.parametrize("H,W", [(1, 1), (1, 9), (1, 1920), (7, 1), (1080, 1), (5, 3), (9, 6), (33, 17), (2, 4097)])
def test_sizes(cv2, H, W):
    rng = np.random.default_rng(H * 10000 + W)
    Q = random_q(rng, 3.0)
    d = special_map(H, W, seed=H + W)
    for hm in (False, True):
        assert same_bits(reference_reproject(d, Q, hm), cv2_reproject(d, Q, hm)), (H, W, hm)


def test_naive_formulations_differ():
    """The two natural shortcuts -- float32 arithmetic, or one float64 division without the float32 rounding of h_k --
    are each wrong in the last bit on most pixels: the rule's roundings are all needed."""
    rng = np.random.default_rng(9)
    H, W = 64, 64
    Q = stereo_rectify_q(H, W, False) if _has_cv2() else random_q(rng, 10.0)
    d = (rng.random((H, W)) * 100 + 1).astype(np.float32)
    want = reference_reproject(d, Q)
    X = np.arange(W, dtype=np.float64)[None].repeat(H, 0)
    Y = np.arange(H, dtype=np.float64)[:, None].repeat(W, 1)
    h = [Q[k, 0] * X + Q[k, 1] * Y + Q[k, 2] * d + Q[k, 3] for k in range(4)]
    direct = np.stack([(h[k] / h[3]).astype(np.float32) for k in range(3)], -1)
    q32, X32, Y32 = Q.astype(np.float32), X.astype(np.float32), Y.astype(np.float32)
    h32 = [q32[k, 0] * X32 + q32[k, 1] * Y32 + q32[k, 2] * d + q32[k, 3] for k in range(4)]
    single = np.stack([h32[k] / h32[3] for k in range(3)], -1)
    for other in (direct, single):
        assert (want.view(np.uint32) != other.view(np.uint32)).mean() > 0.1


def _has_cv2():
    try:
        import cv2  # noqa: F401
        return True
    except ImportError:
        return False


# ---- the deliberate deviation: NaN in the map ---------------------------------------------------------------------------

def test_nan_maps_take_the_minimum_over_non_nan_values(cv2):
    Q = np.array([[1, 0, 0, -10.5], [0, 1, 0, -7.25], [0, 0, 0, 500.0], [0, 0, 0.1, 0]])
    for seed in range(4):
        rng = np.random.default_rng(seed)
        d = (rng.random((31, 45)) * 100 + 1).astype(np.float32)
        d.ravel()[rng.integers(0, d.size, 60)] = rng.choice(near_minimum(1.0), 60)
        d.ravel()[rng.integers(0, d.size, 40)] = np.nan
        d[0, 0] = np.nan                                      # where OpenCV's minMaxLoc would return NaN
        m = float(np.nanmin(d))
        got = reference_reproject(d, Q, True)
        finite = ~np.isnan(d)
        with np.errstate(invalid="ignore"):
            hit = np.abs(d.astype(np.float64) - m) <= FLT_EPS
        assert hit.sum() >= 1 and (got[..., 2][hit] == 10000).all()
        assert same_bits(got[~hit], reference_reproject(d, Q)[~hit])      # every other pixel is untouched
        # with handleMissingValues off no minimum is involved: OpenCV agrees on NaN maps too
        assert same_bits(reference_reproject(d, Q), cv2_reproject(d, Q))
        # on the same map without its NaNs, OpenCV agrees with handleMissingValues on
        clean = np.where(finite, d, np.float32(50.0))
        assert same_bits(reference_reproject(clean, Q, True), cv2_reproject(clean, Q, True))
    all_nan = np.full((3, 5), np.nan, np.float32)
    assert same_bits(reference_reproject(all_nan, Q, True), reference_reproject(all_nan, Q, False))


def test_flt_max_disparity_is_marked_without_handle_missing(cv2):
    """OpenCV's minimum starts at FLT_MAX: a disparity of exactly FLT_MAX gets Z = 10000 even with handleMissingValues
    off, and with it on only when it is the frame's minimum."""
    fmax = np.finfo(np.float32).max
    d = np.float32([[fmax, np.nextafter(fmax, np.float32(0)), 3e38, np.inf, 1.0]])
    Q = np.array([[1, 0, 0, -10.5], [0, 1, 0, -7.25], [0, 0, 0, 500.0], [0, 0, 0.1, 0]])
    for hm, want in ((False, [True, False, False, False, False]), (True, [False, False, False, False, True])):
        got = reference_reproject(d, Q, hm)
        assert same_bits(got, cv2_reproject(d, Q, hm))
        assert list(got[0, :, 2] == 10000) == want


# ---- Q and the pipeline's configuration, without a GPU ----------------------------------------------------------------

def test_reprojection_matrix_conversion_and_errors():
    import torch
    from stereo_depth_b200 import consumers, pipeline
    q = np.arange(16, dtype=np.float32).reshape(4, 4) / 7
    for given in (q, torch.from_numpy(q), torch.from_numpy(q).half(), q.tolist(), np.eye(4, dtype=np.int64),
                  np.eye(4, dtype=np.uint8), torch.eye(4, dtype=torch.int32), [[1, 0, 0, -5]] * 4):
        got = consumers.reprojection_matrix(given)
        assert got.dtype == np.float64 and got.flags.c_contiguous and got.shape == (4, 4)
    assert same_bits(consumers.reprojection_matrix(q), q.astype(np.float64))
    assert same_bits(consumers.reprojection_matrix(crafted_qs()[4]), crafted_qs()[4].astype(np.float64))
    for bad in (np.eye(3), np.eye(4)[:, :3], np.eye(4, dtype=bool), np.eye(4, dtype=np.complex128), np.zeros(16)):
        with pytest.raises(RuntimeError, match="4x4"):
            consumers.reprojection_matrix(bad)
    with pytest.raises(RuntimeError, match="4x4"):       # checked when the pipeline is built
        pipeline.DepthEstimationPipeline(pipeline.DepthEstimationPipelineConfig(reprojection_matrix=np.eye(3)))


def test_integer_q(cv2):
    """OpenCV converts an integer Q to float64 like a float one; so does the rule."""
    d = special_map(9, 13, seed=4)
    for Q in (crafted_qs()[4], crafted_qs()[5], np.eye(4, dtype=np.int32), np.eye(4, dtype=np.uint8)):
        assert Q.dtype.kind in "iu"
        for hm in (False, True):
            assert same_bits(reference_reproject(d, Q, hm), cv2_reproject(d, Q, hm))
