"""Reprojection to 3-D on the GPU (-m gpu): sd_reproject / consumers.reproject_image_to_3d are bit-exact against the
numpy rule of tests/test_reproject_cpu.py, and against cv2.reprojectImageTo3D where OpenCV imports (NaN-free maps), on
every width, batch size, special value, crafted Q and alignment, with handleMissingValues on and off; errors; and the
pipeline's points on a rectified 1080p rig."""
import numpy as np
import pytest

from test_rectify_cpu import within_one
from test_reproject_cpu import (DENORMALS, SPECIAL, crafted_qs, near_minimum, random_q, reference_reproject,
                                reference_reproject_batch, same_bits, special_map)

pytestmark = pytest.mark.gpu


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _cv2():
    try:
        import cv2
        return cv2
    except ImportError:
        return None


def _check(d, Q, hm, got):
    """got == the numpy rule, frame by frame; == OpenCV too when it imports and the frame has no NaN."""
    d = d.reshape((-1,) + d.shape[-2:])
    got = got.reshape(d.shape + (3,))
    assert same_bits(got, reference_reproject_batch(d, Q, hm))
    cv2 = _cv2()
    if cv2 is not None:
        for f in range(d.shape[0]):
            if not np.isnan(d[f]).any():
                assert same_bits(got[f], cv2.reprojectImageTo3D(d[f], np.asarray(Q), handleMissingValues=hm)), f


def _rig_q(H, W, baseline):
    f = float(W)
    return np.array([[1, 0, 0, -(W - 1) / 2], [0, 1, 0, -(H - 1) / 2], [0, 0, 0, f], [0, 0, 1 / baseline, 0]])


@pytest.mark.parametrize("W", [1, 2, 3, 4, 5, 6, 7, 8, 9, 1920])
def test_every_width_and_batch_size(W):
    from stereo_depth_b200 import consumers
    rng = np.random.default_rng(W)
    H = 7 if W == 1920 else 3
    sizes = (1, 2, 29) if W == 1920 else range(1, 30)
    Qs = [random_q(rng, 5.0), _rig_q(H, W, 0.12), random_q(rng, 1e-3)]
    for n in sizes:
        d = np.stack([special_map(H, W, seed=100 * W + 7 * n + f, minimum=float(rng.choice([0.25, 1.0, -3.5])))
                      for f in range(n)])
        Q = Qs[n % len(Qs)]
        for hm in (False, True):
            got = consumers.reproject_image_to_3d(_cuda(d), Q, handle_missing_values=hm).cpu().numpy()
            assert got.shape == (n, H, W, 3)
            _check(d, Q, hm, got)
    one = consumers.reproject_image_to_3d(_cuda(d[0]), Q).cpu().numpy()        # [H,W] in, [H,W,3] out
    assert one.shape == (H, W, 3) and same_bits(one, reference_reproject(d[0], Q))


@pytest.mark.parametrize("hm", [False, True])
def test_special_values_crafted_q_and_denormal_outputs(hm):
    from stereo_depth_b200 import consumers
    row = np.concatenate([SPECIAL, near_minimum(0.0), near_minimum(2.0), np.float32([np.finfo(np.float32).max])])
    d = np.stack([row, row[::-1], -row, np.roll(row, 5)])[None].repeat(3, 0)
    d[1] = np.abs(d[1])
    for i, Q in enumerate(crafted_qs()):
        got = consumers.reproject_image_to_3d(_cuda(d), Q, handle_missing_values=hm).cpu().numpy()
        _check(d, Q, hm, got)
        if i == len(crafted_qs()) - 1:          # denormal output bits survive (no flush to zero)
            tiny = (np.abs(got) < np.finfo(np.float32).tiny) & (got != 0)
            assert tiny.any()
    d = np.float32([[1e-30, 3e-39, 1.0, 0.5], list(DENORMALS[:4])])
    got = consumers.reproject_image_to_3d(_cuda(d), crafted_qs()[-1], handle_missing_values=hm).cpu().numpy()
    _check(d, crafted_qs()[-1], hm, got)


def test_nan_frames_take_the_minimum_over_non_nan_values():
    from stereo_depth_b200 import consumers
    H, W = 33, 70
    Q = _rig_q(H, W, 0.5)
    frames = [np.full((H, W), np.nan, np.float32)]                       # all NaN: no minimum
    for seed in range(4):                                                # partly NaN, NaN at index 0
        d = special_map(H, W, seed=seed, nan=True, minimum=1.0)
        d[0, 0] = np.nan
        frames.append(d)
    frames.append(special_map(H, W, seed=9, minimum=2.0))               # clean
    frames.append(np.where(np.arange(W) % 2 == 0, np.nan, np.float32(3.0)).astype(np.float32)[None].repeat(H, 0))
    d = np.stack(frames)
    for hm in (False, True):
        got = consumers.reproject_image_to_3d(_cuda(d), Q, handle_missing_values=hm).cpu().numpy()
        _check(d, Q, hm, got)
    assert not (got[0, ..., 2] == 10000).any() and (got[-1, :, 1::2, 2] == 10000).all()


def test_large_batch_and_ragged_1080p():
    """29 frames at 1080p (the vector path), and 1080 x 1917 (W % 4 != 0: the scalar path)."""
    from stereo_depth_b200 import consumers
    rng = np.random.default_rng(3)
    for H, W, n in ((1080, 1920, 29), (1080, 1917, 3)):
        d = (rng.random((n, H, W)) * 127 + 1).astype(np.float32)
        d[:, ::97, ::89] = -1.0
        Q = _rig_q(H, W, 0.1)
        Q[3, 3] = 0.37                      # differing principal points
        for hm in (False, True):
            got = consumers.reproject_image_to_3d(_cuda(d), Q, handle_missing_values=hm).cpu().numpy()
            assert same_bits(got, reference_reproject_batch(d, Q, hm)), (H, W, hm)


def test_unaligned_buffers_and_out():
    import torch
    from stereo_depth_b200 import consumers
    H, W, n = 11, 40, 5
    d = np.stack([special_map(H, W, seed=f) for f in range(n)])
    Q = random_q(np.random.default_rng(1), 2.0)
    dstore = torch.zeros(d.size + 1, dtype=torch.float32, device="cuda")
    dstore[1:] = _cuda(d.ravel())
    ostore = torch.zeros(3 * d.size + 1, dtype=torch.float32, device="cuda")
    for dv, ov in ((dstore[1:], ostore[1:]), (dstore[1:], ostore[:-1]), (_cuda(d).view(-1), ostore[1:])):
        out = ov.view(n, H, W, 3)
        for hm in (False, True):
            got = consumers.reproject_image_to_3d(dv.view(n, H, W), Q, handle_missing_values=hm, out=out)
            assert got.data_ptr() == out.data_ptr()
            _check(d, Q, hm, out.cpu().numpy())


def test_errors_and_empty_batches():
    import torch
    from stereo_depth_b200 import _native as N
    from stereo_depth_b200 import consumers
    import ctypes
    H, W = 8, 12
    t = torch.ones((2, H, W), dtype=torch.float32, device="cuda")
    Q = np.eye(4)
    with pytest.raises(RuntimeError, match="4x4"):
        consumers.reproject_image_to_3d(t, np.eye(3))
    with pytest.raises(RuntimeError, match="4x4"):
        consumers.reproject_image_to_3d(t, np.eye(4, dtype=bool))
    with pytest.raises(RuntimeError, match="float32 CUDA"):
        consumers.reproject_image_to_3d(t.double(), Q)
    with pytest.raises(RuntimeError, match="float32 CUDA"):
        consumers.reproject_image_to_3d(t.cpu(), Q)
    with pytest.raises(RuntimeError, match="float32 CUDA"):
        consumers.reproject_image_to_3d(t[None], Q)
    with pytest.raises(TypeError):
        consumers.reproject_image_to_3d(t.cpu().numpy(), Q)
    with pytest.raises(RuntimeError, match="shape"):
        consumers.reproject_image_to_3d(t, Q, out=torch.empty((2, H, W, 4), device="cuda"))
    big = torch.zeros(3 * t.numel(), dtype=torch.float32, device="cuda")
    with pytest.raises(RuntimeError, match="overlap"):
        consumers.reproject_image_to_3d(big[:t.numel()].view(2, H, W), Q, out=big.view(2, H, W, 3))
    empty = torch.empty((0, H, W), dtype=torch.float32, device="cuda")
    assert consumers.reproject_image_to_3d(empty, Q).shape == (0, H, W, 3)
    assert consumers.reproject_image_to_3d(torch.empty((5, 0), device="cuda"), Q).shape == (5, 0, 3)
    lib = N.lib()
    q = (ctypes.c_double * 16)(*np.eye(4).ravel())
    out = torch.empty((2, H, W, 3), dtype=torch.float32, device="cuda")
    d, x = t.data_ptr(), out.data_ptr()
    assert lib.sd_reproject(None, 2, H, W, q, 0, x, None) == N.SD_ERR_BAD_ARG
    assert lib.sd_reproject(d, 2, H, W, None, 0, x, None) == N.SD_ERR_BAD_ARG
    assert lib.sd_reproject(d, 2, H, W, q, 1, None, None) == N.SD_ERR_BAD_ARG
    for n, h, w in ((0, H, W), (2, 0, W), (2, H, -1), (-1, H, W), (1 << 30, 1 << 30, 1 << 30)):
        assert lib.sd_reproject(d, n, h, w, q, 0, x, None) == N.SD_ERR_BAD_ARG, (n, h, w)
    assert lib.sd_reproject(d, 2, H, W, q, 0, d, None) == N.SD_ERR_BAD_ARG          # xyz == disparity
    assert lib.sd_reproject(d + 4, 2, H, W, q, 0, d, None) == N.SD_ERR_BAD_ARG      # overlapping
    assert lib.sd_reproject(d, 2, H, W, q, 1, x, None) == N.SD_OK
    torch.cuda.synchronize()
    assert (out[..., 2] == 10000).all()     # every pixel holds the minimum


def test_pipeline_points_on_a_rectified_1080p_rig():
    import torch
    from stereo_depth_b200 import consumers, pipeline
    from stereo_depth_b200.synthetic import make_unrectified_pair
    H, W, D, B = 1080, 1920, 128, 0.25
    lraw, rraw, maps, gt = make_unrectified_pair(H, W, D, seed=3)
    Q = _rig_q(H, W, B)
    f = float(W)

    class Hook:
        def __init__(self):
            self.points = []

        def on_pipeline_start(self):
            pass

        def process(self, context):
            self.points.append(context.points)

        def on_pipeline_end(self):
            pass

    base = dict(image_shape=(H, W), min_disparity=0, max_disparity=D - 1, rectification_maps=maps)
    frames = [(torch.from_numpy(lraw), torch.from_numpy(rraw))]
    with_q = pipeline.DepthEstimationPipeline(pipeline.DepthEstimationPipelineConfig(**base, reprojection_matrix=Q))
    res = with_q.process(*frames[0])
    disp = res.disparity_map
    assert res.points.shape == (H, W, 3) and res.points.dtype == torch.float32
    assert same_bits(res.points.cpu().numpy(), consumers.reproject_image_to_3d(disp, Q).cpu().numpy())
    dn = disp.cpu().numpy()
    assert same_bits(res.points.cpu().numpy(), reference_reproject(dn, Q))
    assert within_one(dn, gt) > 0.8
    m = np.zeros((H, W), bool)
    m[H // 10:H - H // 10, W // 10:W - W // 10] = True
    m &= (np.abs(dn - gt) <= 1) & (gt > 1)
    Z = res.points[..., 2].cpu().numpy()[m].astype(np.float64)
    g = gt[m].astype(np.float64)
    assert m.sum() > 0.4 * H * W
    assert ((Z >= f * B / (g + 1) * (1 - 1e-6)) & (Z <= f * B / (g - 1) * (1 + 1e-6))).all()
    hook = Hook()
    pipeline.run_depth_estimation_pipeline(frames, with_q, hooks=[hook])
    assert len(hook.points) == 1 and same_bits(hook.points[0].cpu().numpy(), res.points.cpu().numpy())
    # unset: no points, the same disparity map bit for bit
    without = pipeline.DepthEstimationPipeline(pipeline.DepthEstimationPipelineConfig(**base))
    res0 = without.process(*frames[0])
    assert res0.points is None and same_bits(res0.disparity_map.cpu().numpy(), dn)
    hook0 = Hook()
    pipeline.run_depth_estimation_pipeline(frames, without, hooks=[hook0])
    assert hook0.points == [None]
