"""Rectification on the GPU (-m gpu): the remap kernel is bit-exact against the numpy rule and cv2.remap on every width,
dtype and pathological map; a handle with rectification on gives, bit for bit, what the same handle gives with it off on
reference-rectified frames -- output and intermediates, on every entry point and mode; maps are owned by the handle;
switching, launch counts, errors, guard bands and memory are covered; a 1080p rig with rotated cameras is matched
nearly as well as a rectified one."""
import ctypes

import numpy as np
import pytest

from parity_util import mismatch
from stereo_depth_b200.synthetic import make_pair, make_unrectified_pair
from test_gpu_parity import SEEDED, cfg_kw
from test_lr_check_cpu import reference_check
from test_lr_check_gpu import _matcher
from test_lr_fill_cpu import reference_background_fill
from test_rectify_cpu import (cv2_remap, fraction_maps, images, reference_remap, same_bits, special_maps,
                              within_one)

pytestmark = pytest.mark.gpu


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _maps(H, W, seed=0):
    """Maps that rotate each view by about one degree about the image centre and shift it by a fraction of a pixel, with
    a few pathological entries (NaN, inf, far outside)."""
    rng = np.random.default_rng(seed)
    out = []
    for sign in (1.0, -1.0):
        cols, rows = np.meshgrid(np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64))
        a = sign * 0.02
        mx = (cols - W / 2) * np.cos(a) - (rows - H / 2) * np.sin(a) + W / 2 + sign * 0.3
        my = (cols - W / 2) * np.sin(a) + (rows - H / 2) * np.cos(a) + H / 2 + sign * 1.7
        mx, my = mx.astype(np.float32), my.astype(np.float32)
        k = rng.random((H, W)) < 0.002
        mx[k] = rng.choice(np.float32([np.nan, np.inf, -1e30, 40000, -0.5]), int(k.sum()))
        out.append((mx, my))
    return out


def _raw(H, W, D, dtype, seed):
    l, r, _ = make_pair(H, W, D, seed=seed)
    if dtype == "u8":
        return l, r
    rng = np.random.default_rng(seed)
    f = lambda a: (a.astype(np.float32) * np.float32(0.98) + rng.random(a.shape).astype(np.float32) * 0.3)  # noqa: E731
    return f(l), f(r)


STAGES = ("gray_l", "gray_r", "refined")


def _stages(sm):
    return {s: sm.stage(s).cpu().numpy() for s in STAGES}


def _equivalence(sm, raw_l, raw_r, maps, batch=False, host=False):
    """Output and intermediates with rectification on (raw frames) == off (reference-rectified frames), same handle."""
    import torch
    (lmx, lmy), (rmx, rmy) = maps
    rect_l, rect_r = reference_remap(raw_l, lmx, lmy), reference_remap(raw_r, rmx, rmy)

    def run(a, b):
        if host:
            return sm.compute_disparity_host(torch.from_numpy(np.ascontiguousarray(a)),
                                             torch.from_numpy(np.ascontiguousarray(b))).numpy().copy()
        if batch:
            return sm.compute_disparity_batch(_cuda(a), _cuda(b)).cpu().numpy()
        return sm.compute_disparity_map(_cuda(a), _cuda(b)).cpu().numpy().copy()

    sm.set_rectification(None, None)
    assert not sm.rectification
    want, want_st = run(rect_l, rect_r), _stages(sm)
    sm.set_rectification((lmx, lmy), (rmx, rmy))
    assert sm.rectification
    got, got_st = run(raw_l, raw_r), _stages(sm)
    assert mismatch(got, want) == 0, "output"
    for s in STAGES:
        assert mismatch(got_st[s], want_st[s]) == 0, s
    return got


# ---- the kernel through consumers.rectify / sd_rectify ---------------------------------------------------------------

@pytest.mark.parametrize("W", [1, 2, 3, 5, 17, 64, 255, 1000, 2049, 4097])
@pytest.mark.parametrize("dtype", [np.uint8, np.float32])
def test_rectify_every_width(W, dtype):
    from stereo_depth_b200 import consumers
    try:
        import cv2  # noqa: F401
        have_cv2 = True
    except ImportError:
        have_cv2 = False
    for H, planes in ((1, 1), (7, 3), (33, 7), (3, 2)):
        mx, my = special_maps(H, W)
        img = images((planes, H, W), dtype, W * 31 + H)
        want = reference_remap(img, mx, my)
        got = consumers.rectify(_cuda(img), _cuda(mx), _cuda(my)).cpu().numpy()
        assert same_bits(got, want), (H, W, planes)
        if have_cv2:
            assert same_bits(got, cv2_remap(img, mx, my)), (H, W, planes)


@pytest.mark.parametrize("dtype", [np.uint8, np.float32])
def test_rectify_every_fraction_and_special_value(dtype):
    from stereo_depth_b200 import consumers
    from test_rectify_cpu import SPECIAL
    H, W = 64, 96
    fx, fy = fraction_maps(H, W, x0=40, y0=20)
    mx, my = np.tile(fx, (2, 3)) + np.float32(0), np.tile(fy, (2, 3)) + np.float32(0)
    a, b = np.meshgrid(SPECIAL, SPECIAL)
    mx[:a.shape[0], :a.shape[1]], my[:a.shape[0], :a.shape[1]] = a, b
    mx[-a.shape[0]:, -a.shape[1]:], my[-a.shape[0]:, -a.shape[1]:] = b, a
    for seed in range(3):
        img = images((5, H, W), dtype, seed)
        got = consumers.rectify(_cuda(img), _cuda(mx), _cuda(my)).cpu().numpy()
        assert same_bits(got, reference_remap(img, mx, my)), seed


def test_rectify_unaligned_buffers_out_and_errors():
    """Maps and output off their 16-byte alignment take the scalar path; `out`, 4-D input; argument errors."""
    import torch
    from stereo_depth_b200 import _native as N
    from stereo_depth_b200 import consumers
    H, W = 30, 44
    mx, my = special_maps(H, W)
    img = images((2, 3, H, W), np.uint8, 5)
    big_x, big_y = _cuda(np.concatenate([[0], mx.ravel()]).astype(np.float32)), _cuda(
        np.concatenate([[0], my.ravel()]).astype(np.float32))
    ux, uy = big_x[1:].view(H, W), big_y[1:].view(H, W)
    store = torch.zeros(img.size + 1, dtype=torch.uint8, device="cuda")
    out = store[1:].view(img.shape)
    got = consumers.rectify(_cuda(img), ux, uy, out=out)
    assert got.data_ptr() == out.data_ptr()
    assert same_bits(out.cpu().numpy(), reference_remap(img, mx, my))
    t = _cuda(img)
    with pytest.raises(RuntimeError, match="in place"):
        consumers.rectify(t, _cuda(mx), _cuda(my), out=t)
    with pytest.raises(RuntimeError, match="CV_32FC1"):
        consumers.rectify(t, _cuda(mx).double(), _cuda(my))
    with pytest.raises(RuntimeError):
        consumers.rectify(t.long(), _cuda(mx), _cuda(my))
    lib, p, q = N.lib(), t.data_ptr(), out.data_ptr()
    x, y = _cuda(mx), _cuda(my)
    assert lib.sd_rectify(x.data_ptr(), y.data_ptr(), p, p, N.SD_U8, 6, H, W, None) == N.SD_ERR_BAD_ARG
    assert lib.sd_rectify(None, y.data_ptr(), p, q, N.SD_U8, 6, H, W, None) == N.SD_ERR_BAD_ARG
    assert lib.sd_rectify(x.data_ptr(), y.data_ptr(), p, q, 7, 6, H, W, None) == N.SD_ERR_BAD_ARG
    assert lib.sd_rectify(x.data_ptr(), y.data_ptr(), p, q, N.SD_U8, 0, H, W, None) == N.SD_ERR_BAD_ARG
    assert lib.sd_rectify(x.data_ptr(), y.data_ptr(), p, q, N.SD_U8, 1, 32768, 1, None) == N.SD_ERR_BAD_ARG
    assert lib.sd_rectify(x.data_ptr(), y.data_ptr(), p, q, N.SD_U8, 6, H, W, None) == N.SD_OK


# ---- the handle: rectification on == off on reference-rectified frames --------------------------------------------------

@pytest.mark.parametrize("shape", SEEDED)
@pytest.mark.parametrize("variant", ["generic", "fast", "ws"])
def test_handle_equals_reference_rectified_input(shape, variant):
    H, W, K, mn, mx = shape
    kw = cfg_kw(H, W, K, mn, mx)
    if variant == "ws" and mx // K - mn // K + 1 > 150:
        pytest.skip("warp-specialised variant needs L <= ~150")
    maps = _maps(H, W, seed=H)
    screens = (True, False) if variant == "fast" else (None,)
    for dtype in ("u8", "f32"):
        raw_l, raw_r = _raw(H, W, mx + 1, dtype, seed=200 + H)
        for screen in screens:
            sm = _matcher(kw, 2, variant)
            if screen is not None and screen != sm.screen_active:
                try:
                    sm.set_screen(screen)
                except RuntimeError:     # no level screen for this configuration
                    continue
            _equivalence(sm, raw_l, raw_r, maps)


@pytest.mark.parametrize("dtype", ["u8", "f32"])
def test_batches_single_frames_host_path_and_compat(dtype):
    from stereo_depth_b200 import cuda_depth
    H, W, D = 120, 256, 48
    maps = _maps(H, W, seed=3)
    ls, rs = zip(*[_raw(H, W, D, dtype, seed=60 + f) for f in range(7)])
    L, R = np.stack(ls), np.stack(rs)
    for mn in (0, 16):                   # min_disparity 16: reference-compat mode
        kw = cfg_kw(H, W, 2, mn, mn + D - 1)
        sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=3)
        _equivalence(sm, L, R, maps, batch=True)              # 7 frames on a 3-frame handle: 3 + 2 + 2
        _equivalence(sm, L[:1], R[:1], maps, batch=True)      # one frame per call
        _equivalence(sm, L[4], R[4], maps)
        _equivalence(sm, L, R, maps, host=True)


@pytest.mark.parametrize("fill", [False, True])
def test_left_right_check_rectifies_each_frame_once(fill):
    from stereo_depth_b200 import cuda_depth
    H, W, D = 96, 160, 32
    kw = cfg_kw(H, W, 2, 0, D - 1)
    maps = _maps(H, W, seed=4)
    ls, rs = zip(*[_raw(H, W, D, "u8", seed=80 + f) for f in range(5)])
    L, R = np.stack(ls), np.stack(rs)
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=4)
    sm.set_left_right_check(0.5, -3.0, background_fill=fill)
    got = _equivalence(sm, L, R, maps, batch=True)
    right = sm.stage("right").cpu().numpy()
    sm.set_left_right_check(None)
    (lmx, lmy), (rmx, rmy) = maps
    plain = sm.compute_disparity_batch(_cuda(L), _cuda(R)).cpu().numpy()   # rectified, unchecked
    rule = reference_background_fill if fill else reference_check
    assert mismatch(got[-1], rule(plain[-1], right, 0.5, -3.0)) == 0
    sm.set_left_right_check(0.5, -3.0, background_fill=fill)
    _equivalence(sm, L, R, maps, host=True)


# ---- maps -----------------------------------------------------------------------------------------------------------

def test_maps_are_copied_switched_and_replaced():
    import torch
    from stereo_depth_b200 import cuda_depth
    H, W, D = 96, 192, 32
    kw = cfg_kw(H, W, 2, 0, D - 1)
    l, r = (_cuda(a) for a in _raw(H, W, D, "u8", seed=9))
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=2)
    never = sm.compute_disparity_map(l, r).cpu().numpy().copy()
    counts_off = [sm.launches_per_call(k) for k in range(1, 8)]
    m1 = _maps(H, W, seed=1)
    m2 = [m1[1], m1[0]]                   # the views' rotations swapped
    dev = [tuple(_cuda(m) for m in pair) for pair in m1]
    sm.set_rectification(*dev)
    with_m1 = sm.compute_disparity_map(l, r).cpu().numpy().copy()
    for pair in dev:                      # the caller's maps change after the call: the handle has its own copy
        for t in pair:
            t.fill_(3.0)
    assert mismatch(sm.compute_disparity_map(l, r).cpu().numpy(), with_m1) == 0
    counts_on = [sm.launches_per_call(k) for k in range(1, 8)]
    assert counts_on == [c + -(-k // 2) for k, c in zip(range(1, 8), counts_off)]   # + 1 per chunk of 2 frames
    sm.set_rectification(None, None)
    want2 = sm.compute_disparity_map(_cuda(reference_remap(l.cpu().numpy(), *m2[0])),
                                     _cuda(reference_remap(r.cpu().numpy(), *m2[1]))).cpu().numpy().copy()
    sm.set_rectification(*m2)            # numpy maps this time; new maps take effect
    got2 = sm.compute_disparity_map(l, r).cpu().numpy().copy()
    assert mismatch(got2, want2) == 0 and mismatch(got2, with_m1) != 0
    sm.set_rectification(None, None)     # off: the unrectified outputs and launch counts
    assert not sm.rectification
    assert [sm.launches_per_call(k) for k in range(1, 8)] == counts_off
    assert mismatch(sm.compute_disparity_map(l, r).cpu().numpy(), never) == 0
    # the pipeline config
    from stereo_depth_b200 import pipeline
    pc = pipeline.DepthEstimationPipelineConfig(image_shape=(H, W), min_disparity=0, max_disparity=D - 1,
                                                rectification_maps=tuple(m2))
    res = pipeline.DepthEstimationPipeline(pc).process(l.cpu(), r.cpu())
    assert mismatch(res.disparity_map.cpu().numpy(), got2) == 0
    torch.cuda.synchronize()


def test_errors_and_row_band_refusals():
    import torch
    from stereo_depth_b200 import _native as N
    from stereo_depth_b200 import cuda_depth
    H, W = 64, 128
    kw = cfg_kw(H, W, 2, 0, 31)
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=2)
    maps = _maps(H, W)
    with pytest.raises(RuntimeError, match="m1type=cv2.CV_32FC1"):
        sm.set_rectification((maps[0][0].astype(np.float64), maps[0][1]), maps[1])
    with pytest.raises(RuntimeError, match="m1type=cv2.CV_32FC1"):
        sm.set_rectification((np.zeros((H, W, 2), np.int16), np.zeros((H, W), np.uint16)), maps[1])
    with pytest.raises(RuntimeError, match="m1type=cv2.CV_32FC1"):
        sm.set_rectification((maps[0][0][:, :-1], maps[0][1]), maps[1])
    with pytest.raises(RuntimeError, match="pair"):
        sm.set_rectification(maps[0], None)
    assert not sm.rectification
    lib, h = N.lib(), sm._handle._h
    x = _cuda(maps[0][0])
    assert lib.sd_set_rectification(None, x.data_ptr(), x.data_ptr(), x.data_ptr(), x.data_ptr(), None) == N.SD_ERR_BAD_ARG
    assert lib.sd_set_rectification(h, x.data_ptr(), None, x.data_ptr(), x.data_ptr(), None) == N.SD_ERR_BAD_ARG
    assert lib.sd_set_rectification(h, None, None, None, None, None) == N.SD_OK
    # row-band modes, in either order
    g = torch.zeros((H, W), dtype=torch.float32, device="cuda")
    sm.set_rectification(*maps)
    assert lib.sd_set_band(h, 0, 2 * H, g.data_ptr()) == N.SD_ERR_UNSUPPORTED
    img = torch.zeros((1, 3, H, W), dtype=torch.uint8, device="cuda")
    out = torch.zeros((1, H, W), dtype=torch.float32, device="cuda")
    assert lib.sd_compute_range(h, img.data_ptr(), img.data_ptr(), N.SD_U8, 1, out.data_ptr(), None, 0, 3) == \
        N.SD_ERR_UNSUPPORTED
    rows = (ctypes.c_int32 * 2)(0, H)
    buf = ctypes.create_string_buffer(64)
    assert lib.sd_band_p2p_init(h, 1, 0, rows, 0, N.SD_U8, buf) == N.SD_ERR_UNSUPPORTED
    sm.set_rectification(None, None)
    assert lib.sd_set_band(h, 0, 2 * H, g.data_ptr()) == N.SD_OK
    x = _cuda(maps[0][0])
    assert lib.sd_set_rectification(h, x.data_ptr(), x.data_ptr(), x.data_ptr(), x.data_ptr(), None) == \
        N.SD_ERR_UNSUPPORTED
    assert lib.sd_set_band(h, 0, 0, None) == N.SD_OK
    assert lib.sd_set_rectification(h, x.data_ptr(), x.data_ptr(), x.data_ptr(), x.data_ptr(), None) == N.SD_OK


# ---- guard bands, memory, quality -----------------------------------------------------------------------------------

@pytest.mark.parametrize("shape,dtype", [
    ((75, 133, 2, 0, 30), "u8"),     # ragged: H * W % 4 != 0 -> scalar map loads and stores
    ((75, 133, 2, 0, 30), "f32"),
    ((24, 44, 2, 0, 17), "u8"),
    ((136, 264, 2, 0, 63), "f32"),
    ((64, 256, 2, 0, 63), "u8"),
])
def test_guard_bands_with_rectification(shape, dtype, monkeypatch):
    import torch
    from stereo_depth_b200 import cuda_depth
    monkeypatch.setenv("SD_DEBUG_GUARDS", "1")
    H, W, K, mn, mx = shape
    kw = cfg_kw(H, W, K, mn, mx)
    l, r = _raw(H, W, mx + 1, dtype, seed=900 + H)
    maps = _maps(H, W, seed=H)
    for fpl in (2, 5):
        sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=fpl)
        sm.set_rectification(*maps)
        L, R = _cuda(np.stack([l] * 3)), _cuda(np.stack([r] * 3))
        sm.compute_disparity_batch(L, R)
        sm.compute_disparity_host(L.cpu(), R.cpu())
        sm.set_left_right_check(1.0, background_fill=True)
        sm.compute_disparity_batch(L, R)
        torch.cuda.synchronize()
        assert sm._handle.check_guards() == 0, (shape, dtype, fpl)


def test_closed_handle_with_rectification_returns_its_device_memory():
    import gc
    import torch
    from stereo_depth_b200 import cuda_depth
    H, W = 1080, 1920
    maps = [tuple(_cuda(m) for m in pair) for pair in _maps(H, W)]
    gen = torch.Generator().manual_seed(11)
    left = torch.randint(0, 256, (2, 3, H, W), dtype=torch.uint8, generator=gen)

    def cycle():
        sm = cuda_depth.StereoMatching()
        sm.set_rectification(*maps)
        sm.compute_disparity_batch(left.cuda(), left.cuda())
        sm.compute_disparity_host(left.float(), left.float())
        sm.set_rectification(None, None)
        sm.set_rectification(*maps)
        sm.compute_disparity_map(left[0].cuda(), left[1].cuda())
        sm._handle.close()

    def free():
        gc.collect()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        return torch.cuda.mem_get_info()[0]

    cycle()
    base = free()
    for _ in range(3):
        cycle()
    drift = base - free()
    assert abs(drift) <= 1 << 20, drift


def test_rotated_rig_at_1080p():
    from oracle import oracle as O
    from stereo_depth_b200 import cuda_depth
    H, W, D = 1080, 1920, 128
    lraw, rraw, maps, gt = make_unrectified_pair(H, W, D, seed=3)
    l, r, _ = make_pair(H, W, D, seed=3)
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**cfg_kw(H, W, 2, 0, D - 1)))
    direct = sm.compute_disparity_map(_cuda(l), _cuda(r)).cpu().numpy().copy()
    raw = sm.compute_disparity_map(_cuda(lraw), _cuda(rraw)).cpu().numpy().copy()
    sm.set_rectification(*maps)
    rect = sm.compute_disparity_map(_cuda(lraw), _cuda(rraw)).cpu().numpy().copy()
    q = {k: within_one(v, gt) for k, v in (("direct", direct), ("rectified", rect), ("raw", raw))}
    print("1080p rotated rig:", {k: round(v, 4) for k, v in q.items()})
    assert q["rectified"] >= q["direct"] - 0.03 and q["raw"] < 0.5 * q["rectified"], q
    (lmx, lmy), (rmx, rmy) = maps
    cfg = O.make_config(**cfg_kw(H, W, 2, 0, D - 1))
    assert mismatch(rect, O.run(cfg, reference_remap(lraw, lmx, lmy), reference_remap(rraw, rmx, rmy))["out"]) == 0
