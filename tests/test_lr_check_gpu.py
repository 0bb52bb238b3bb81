"""Left-right consistency check on the GPU (-m gpu): the right view's map is bit-exact against the oracle run on the
mirrored pair, the checked left map is exactly the numpy reference of the check applied to the unchecked output, every
entry point honours the switch, and switching it off restores the old path bit for bit."""
import ctypes as C
import math

import numpy as np
import pytest

from oracle import oracle as O
from parity_util import mismatch
from stereo_depth_b200.synthetic import make_pair
from test_gpu_parity import SEEDED, cfg_kw
from test_lr_check_cpu import left_ground_truth, oracle_right_map, reference_check

pytestmark = pytest.mark.gpu


def _mode(kw, compat=None):
    if compat is None:
        compat = kw["min_disparity"] // kw["downscale_factor"] != 0
    return O.MODE_COMPAT if compat else O.MODE_SAFE


def _matcher(kw, frames_per_launch=0, variant="auto", compat=None, screen=None, split=None):
    from stereo_depth_b200 import cuda_depth
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=frames_per_launch)
    sm.set_variant(variant)
    if compat is not None:
        sm.set_compat(compat)
    if screen is not None:
        sm.set_screen(screen)
    if split is not None:
        sm.set_level_split(split)
    return sm


def _tensors(l, r, dtype):
    import torch
    lt, rt = torch.from_numpy(l).cuda(), torch.from_numpy(r).cuda()
    if dtype == "f32":
        lt, rt = lt.float(), rt.float()
    return lt.contiguous(), rt.contiguous()


def _check_case(sm, kw, l, r, dtype, mode, tol=1.0, inval=-1.0):
    """Unchecked, then checked output of one frame on the same handle; both maps against the oracle."""
    lt, rt = _tensors(l, r, dtype)
    sm.set_left_right_check(None)
    plain = sm.compute_disparity_map(lt, rt).cpu().numpy().copy()
    sm.set_left_right_check(tol, inval)
    checked = sm.compute_disparity_map(lt, rt).cpu().numpy().copy()
    right = sm.stage("right").cpu().numpy()
    cfg = O.make_config(**kw)
    ref_right = oracle_right_map(cfg, l, r, mode)
    ref_left = O.run(cfg, l, r, mode=mode)["out"]
    assert mismatch(plain, ref_left) == 0
    assert mismatch(right, ref_right) == 0, "right map"
    want = reference_check(plain, right, tol, inval)
    assert mismatch(checked, want) == 0, "checked left map"
    keep = checked != np.float32(inval)
    assert mismatch(checked[keep], plain[keep]) == 0
    sm.set_left_right_check(None)
    return checked


@pytest.mark.parametrize("shape", SEEDED)
@pytest.mark.parametrize("variant", ["generic", "fast", "ws"])
def test_right_map_and_check_bit_exact(shape, variant):
    H, W, K, mn, mx = shape
    kw = cfg_kw(H, W, K, mn, mx)
    if variant == "ws" and mx // K - mn // K + 1 > 150:
        pytest.skip("warp-specialised variant needs L <= ~150")
    l, r, _ = make_pair(H, W, mx + 1, seed=100 + H)
    # specialised kernel: with and without the level screen, with and without the level split
    combos = [(s, p) for s in (True, False) for p in (True, False)] if variant == "fast" else [(None, None)]
    for dtype in ("u8", "f32"):
        for screen, split in combos:
            sm = _matcher(kw, 2, variant, split=split)
            if screen is not None and screen != sm.screen_active:
                try:
                    sm.set_screen(screen)
                except RuntimeError:     # no level screen for this configuration
                    continue
            _check_case(sm, kw, l, r, dtype, _mode(kw))


@pytest.mark.parametrize("shape", [sh for sh in SEEDED if sh[3] // sh[2] != 0] + [(150, 560, 2, 75, 262)])
@pytest.mark.parametrize("compat", [True, False])
@pytest.mark.parametrize("screen", [True, False])
def test_min_disparity_compat_on_and_off(shape, compat, screen):
    H, W, K, mn, mx = shape
    kw = cfg_kw(H, W, K, mn, mx)
    l, r, _ = make_pair(H, W, mx + 1, seed=300 + H)
    sm = _matcher(kw, 4, "fast", compat=compat)
    try:
        sm.set_screen(screen)
    except RuntimeError:
        pytest.skip("no level screen for this configuration")
    for dtype in ("u8", "f32"):
        _check_case(sm, kw, l, r, dtype, _mode(kw, compat))


def test_entry_points_batches_host_backend_pipeline():
    import torch
    from stereo_depth_b200 import backend, consumers, cuda_depth, pipeline
    H, W, K, D = 120, 256, 2, 48
    kw = cfg_kw(H, W, K, 0, D - 1)
    cfg = O.make_config(**kw)
    n = 7
    ls, rs = zip(*[make_pair(H, W, D, seed=40, frame=f)[:2] for f in range(n)])
    L, R = np.stack(ls), np.stack(rs)
    want = np.stack([reference_check(O.run(cfg, L[f], R[f])["out"], oracle_right_map(cfg, L[f], R[f]), 0.5, -3.0)
                     for f in range(n)])
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=4)
    assert sm.left_right_check is None
    sm.set_left_right_check(0.5, -3.0)
    assert sm.left_right_check == 0.5
    # single frame (aliasing output buffer, like the reference)
    out = sm.compute_disparity_map(torch.from_numpy(L[3]).cuda(), torch.from_numpy(R[3]).cuda())
    assert out.data_ptr() == sm._out.data_ptr()
    assert mismatch(out.cpu().numpy(), want[3]) == 0
    # 7 frames on a 4-frame handle: chunks of 2 pairs -> 2+2+2+1
    got = sm.compute_disparity_batch(torch.from_numpy(L).cuda(), torch.from_numpy(R).cuda()).cpu().numpy()
    assert mismatch(got, want) == 0
    # the last chunk held frame 6 alone: its right map
    assert mismatch(sm.stage("right", 0).cpu().numpy(), oracle_right_map(cfg, L[6], R[6])) == 0
    # host path from pinned memory
    host = sm.compute_disparity_host(torch.from_numpy(L).pin_memory(), torch.from_numpy(R).pin_memory())
    assert mismatch(host.numpy(), want) == 0
    # the backend through .native, on CPU and CUDA batches
    be = backend.CudaStereoMatchingBackend(cuda_depth.StereoMatchingConfiguration(**kw))
    be.native.set_left_right_check(0.5, -3.0)
    assert mismatch(be.process_batch(torch.from_numpy(L), torch.from_numpy(R)).numpy(), want) == 0
    assert mismatch(be.process_batch(torch.from_numpy(L).cuda(), torch.from_numpy(R).cuda()).cpu().numpy(), want) == 0
    assert mismatch(be.process(torch.from_numpy(L[1]), torch.from_numpy(R[1])).cpu().numpy(), want[1]) == 0
    # the pipeline: left_right_check with the config's invalid_disparity; point_cloud drops exactly the invalid pixels
    pc = pipeline.DepthEstimationPipelineConfig(image_shape=(H, W), min_disparity=0, max_disparity=D - 1,
                                                left_right_check=1.0)
    pipe = pipeline.DepthEstimationPipeline(pc)
    res = pipe.process(torch.from_numpy(L[2]), torch.from_numpy(R[2]))
    want2 = reference_check(O.run(cfg, L[2], R[2])["out"], oracle_right_map(cfg, L[2], R[2]), 1.0, -1.0)
    d = res.disparity_map.cpu().numpy()
    assert mismatch(d, want2) == 0
    assert (d == -1.0).sum() > 0
    pts = consumers.point_cloud(res.disparity_map, 1.0, 1.0, invalid_disparity=pc.invalid_disparity)
    assert pts.shape[0] == int((d != -1.0).sum())
    off = pipeline.DepthEstimationPipeline(pipeline.DepthEstimationPipelineConfig(image_shape=(H, W), min_disparity=0,
                                                                                  max_disparity=D - 1))
    assert mismatch(off.process(torch.from_numpy(L[2]), torch.from_numpy(R[2])).disparity_map.cpu().numpy(),
                    O.run(cfg, L[2], R[2])["out"]) == 0


def test_switching_off_restores_the_old_path():
    import torch
    from stereo_depth_b200 import cuda_depth
    H, W, K, D = 200, 384, 2, 64
    kw = cfg_kw(H, W, K, 0, D - 1)
    n = 5
    ls, rs = zip(*[make_pair(H, W, D, seed=50, frame=f)[:2] for f in range(n)])
    L, R = torch.from_numpy(np.stack(ls)).cuda(), torch.from_numpy(np.stack(rs)).cuda()
    never = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=4)
    base = never.compute_disparity_batch(L, R).cpu().numpy()
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=4)
    counts_off = [sm.launches_per_call(k) for k in range(1, 10)]
    sm.set_left_right_check(1.0)
    counts_on = [sm.launches_per_call(k) for k in range(1, 10)]
    checked = sm.compute_disparity_batch(L, R).cpu().numpy()
    sm.set_left_right_check(None)
    assert sm.left_right_check is None
    assert [sm.launches_per_call(k) for k in range(1, 10)] == counts_off
    again = sm.compute_disparity_batch(L, R).cpu().numpy()
    assert mismatch(again, base) == 0
    assert mismatch(checked, base) > 0
    # documented count: chunks of frames_per_launch/2 = 2 pairs (equal sizes), each counted as the unchecked launches of
    # twice its frames (one chunk of <= 4 frames) + the second fill launch
    for k in range(1, 10):
        nch = -(-k // 2)
        sizes = [k // nch + (1 if c < k % nch else 0) for c in range(nch)]
        assert counts_on[k - 1] == sum(counts_off[2 * s - 1] + 1 for s in sizes), (k, sizes)
    # a single-frame call is ONE two-frame launch per stage (+ the second fill), not two one-frame calls
    sm.set_left_right_check(1.0)
    one_on = sm.launches_per_call(1)
    sm.set_left_right_check(None)
    assert one_on == sm.launches_per_call(2) + 1


def test_errors():
    import torch
    from stereo_depth_b200 import _native as N
    from stereo_depth_b200 import cuda_depth
    kw = cfg_kw(64, 128, 2, 0, 31)
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=2)
    h = sm._handle._h
    lib = N.lib()
    for bad in (-1.0, math.nan, math.inf, -math.inf):
        with pytest.raises(ValueError):
            sm.set_left_right_check(bad)
        assert lib.sd_set_lr_check(h, 1, bad, -1.0) == N.SD_ERR_BAD_ARG
    assert sm.left_right_check is None
    # the right map exists only with the check on
    with pytest.raises(RuntimeError):
        sm.stage("right")
    dst = torch.empty((64, 128), device="cuda")
    assert lib.sd_get_stage(h, 7, 0, dst.data_ptr(), None) == N.SD_ERR_UNSUPPORTED
    sm.set_left_right_check(1.0)
    assert lib.sd_get_stage(h, 7, 1, dst.data_ptr(), None) == N.SD_ERR_SHAPE      # 1 pair per chunk
    p = C.c_void_p()
    assert lib.sd_stage_pointer(h, 7, 0, C.byref(p)) == N.SD_ERR_UNSUPPORTED
    # row-band modes, both orders
    gray = torch.zeros((128, 128), device="cuda")
    assert lib.sd_set_band(h, 0, 128, gray.data_ptr()) == N.SD_ERR_UNSUPPORTED
    assert lib.sd_compute_range(h, dst.data_ptr(), dst.data_ptr(), N.SD_U8, 1, dst.data_ptr(), None, 0, 3) == \
        N.SD_ERR_UNSUPPORTED
    rows = (C.c_int32 * 2)(0, 64)
    buf = C.create_string_buffer(64)
    assert lib.sd_band_p2p_init(h, 1, 0, rows, 0, N.SD_U8, buf) == N.SD_ERR_UNSUPPORTED
    sm.set_left_right_check(None)
    assert lib.sd_set_band(h, 0, 128, gray.data_ptr()) == N.SD_OK
    assert lib.sd_set_lr_check(h, 1, 1.0, -1.0) == N.SD_ERR_UNSUPPORTED
    assert lib.sd_set_band(h, 0, 0, None) == N.SD_OK
    assert lib.sd_set_lr_check(h, 1, 1.0, -1.0) == N.SD_OK
    assert lib.sd_set_lr_check(h, 0, 0.0, 0.0) == N.SD_OK
    # frames_per_launch = 1
    one = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=1)
    with pytest.raises(RuntimeError, match="frames_per_launch >= 2"):
        one.set_left_right_check(1.0)
    assert lib.sd_set_lr_check(one._handle._h, 1, 1.0, -1.0) == N.SD_ERR_SHAPE


@pytest.mark.parametrize("shape,dtype", [
    ((75, 133, 2, 0, 30), "u8"),     # ragged: W % 16 != 0, H odd -> generic ingest
    ((75, 133, 2, 0, 30), "f32"),
    ((24, 44, 2, 0, 17), "u8"),      # smaller than a tile
    ((136, 264, 2, 0, 63), "f32"),   # tile overhang, W % 16 == 8 -> f32 fast path, u8 generic
    ((136, 264, 2, 0, 63), "u8"),
    ((90, 120, 3, 0, 29), "f32"),
    ((64, 256, 2, 0, 63), "u8"),     # u8 fast path
])
def test_guard_bands_with_the_check(shape, dtype, monkeypatch):
    import torch
    from stereo_depth_b200 import cuda_depth
    monkeypatch.setenv("SD_DEBUG_GUARDS", "1")
    H, W, K, mn, mx = shape
    kw = cfg_kw(H, W, K, mn, mx)
    l, r, _ = make_pair(H, W, mx + 1, seed=900 + H)
    lt, rt = _tensors(l, r, dtype)
    for fpl in (2, 5):
        sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=fpl)
        sm.set_left_right_check(1.0)
        sm.compute_disparity_batch(torch.stack([lt] * 3), torch.stack([rt] * 3))
        sm.compute_disparity_host(torch.stack([lt] * 3).cpu(), torch.stack([rt] * 3).cpu())
        sm.stage("right", 0)
        torch.cuda.synchronize()
        assert sm._handle.check_guards() == 0, (shape, dtype, fpl)


def test_quality_at_1080p():
    import torch
    from stereo_depth_b200 import cuda_depth
    H, W, K, D = 1080, 1920, 2, 128
    l, r, g = make_pair(H, W, D, seed=70, frame=0)
    kw = cfg_kw(H, W, K, 0, D - 1)
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw))
    lt, rt = torch.from_numpy(l).cuda(), torch.from_numpy(r).cuda()
    plain = sm.compute_disparity_map(lt, rt).cpu().numpy().copy()
    sm.set_left_right_check(1.0)
    checked = sm.compute_disparity_map(lt, rt).cpu().numpy().copy()
    right = sm.stage("right").cpu().numpy()
    assert mismatch(checked, reference_check(plain, right, 1.0)) == 0
    cfg = O.make_config(**kw)
    assert mismatch(right, oracle_right_map(cfg, l, r)) == 0
    gt = left_ground_truth(g)
    occluded = np.isnan(gt)
    invalid = checked == -1.0
    good = ~occluded & (np.abs(plain - np.nan_to_num(gt)) <= 1.0)
    print(f"1080p: occluded {occluded.mean():.4f}, invalid {invalid.mean():.4f}, "
          f"invalid among occluded {invalid[occluded].mean():.4f}, among good {invalid[good].mean():.4f}")
    assert invalid[occluded].mean() >= 0.65
    assert invalid[good].mean() <= 0.02


@pytest.mark.parametrize("rng_", [(75, 262, True), (0, 127, False)])
def test_natural_pair(rng_):
    import torch
    from stereo_depth_b200 import cuda_depth
    from stereo_depth_b200.synthetic import load_natural_pair
    nat = load_natural_pair()
    if nat is None:
        pytest.skip("natural pair not extracted (data/_ref)")
    l, r, _, _ = nat
    mn, mx, compat = rng_
    H, W = l.shape[1:]
    kw = cfg_kw(H, W, 2, mn, mx)
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw))
    sm.set_left_right_check(1.0)
    checked = sm.compute_disparity_map(torch.from_numpy(l).cuda(), torch.from_numpy(r).cuda()).cpu().numpy()
    right = sm.stage("right").cpu().numpy()
    assert mismatch(right, oracle_right_map(O.make_config(**kw), l, r, _mode(kw))) == 0
    print(f"natural pair {mn}..{mx}: invalid fraction {(checked == -1.0).mean():.4f}")
