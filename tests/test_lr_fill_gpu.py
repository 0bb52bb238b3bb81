"""Background fill of the left-right check on the GPU (-m gpu): the filled map is bit-exact against the numpy rule
applied to the unchecked GPU output and the GPU right map, and to the oracle's maps; the stateless entry point matches
the rule on crafted rows; every entry point honours the switch; switching back restores the check-only and unchecked
paths bit for bit."""
import numpy as np
import pytest

from oracle import oracle as O
from parity_util import mismatch
from stereo_depth_b200.synthetic import make_layered_pair, make_pair
from test_gpu_parity import SEEDED, cfg_kw
from test_lr_check_cpu import oracle_right_map, reference_check
from test_lr_check_gpu import _matcher, _mode, _tensors
from test_lr_fill_cpu import craft, fill_quality, keep_mask, reference_background_fill, same_bits

pytestmark = pytest.mark.gpu


def _fill_case(sm, kw, l, r, dtype, mode, tol=1.0, inval=-1.0):
    """Unchecked, then checked + filled output of one frame on the same handle; against the rule on the GPU's own maps
    and on the oracle's."""
    lt, rt = _tensors(l, r, dtype)
    sm.set_left_right_check(None)
    plain = sm.compute_disparity_map(lt, rt).cpu().numpy().copy()
    sm.set_left_right_check(tol, inval, background_fill=True)
    assert sm.background_fill
    filled = sm.compute_disparity_map(lt, rt).cpu().numpy().copy()
    right = sm.stage("right").cpu().numpy()
    assert mismatch(filled, reference_background_fill(plain, right, tol, inval)) == 0
    cfg = O.make_config(**kw)
    ref = reference_background_fill(O.run(cfg, l, r, mode=mode)["out"], oracle_right_map(cfg, l, r, mode), tol, inval)
    assert mismatch(filled, ref) == 0, "against the oracle's maps"
    sm.set_left_right_check(None)
    assert not sm.background_fill
    return filled


@pytest.mark.parametrize("shape", SEEDED)
@pytest.mark.parametrize("variant", ["generic", "fast", "ws"])
def test_filled_map_bit_exact(shape, variant):
    H, W, K, mn, mx = shape
    kw = cfg_kw(H, W, K, mn, mx)
    if variant == "ws" and mx // K - mn // K + 1 > 150:
        pytest.skip("warp-specialised variant needs L <= ~150")
    l, r, _ = make_pair(H, W, mx + 1, seed=100 + H)
    combos = [(s, p) for s in (True, False) for p in (True, False)] if variant == "fast" else [(None, None)]
    for dtype in ("u8", "f32"):
        for screen, split in combos:
            sm = _matcher(kw, 2, variant, split=split)
            if screen is not None and screen != sm.screen_active:
                try:
                    sm.set_screen(screen)
                except RuntimeError:     # no level screen for this configuration
                    continue
            _fill_case(sm, kw, l, r, dtype, _mode(kw))


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
        _fill_case(sm, kw, l, r, dtype, _mode(kw, compat), tol=0.5, inval=-3.0)


# ---- the stateless entry point on crafted maps ---------------------------------------------------------------------

def _gpu_fill(dl, dr, tol, inval, in_place):
    import torch
    from stereo_depth_b200 import consumers
    lt, rt = torch.from_numpy(np.ascontiguousarray(dl)).cuda(), torch.from_numpy(np.ascontiguousarray(dr)).cuda()
    if in_place:
        got = consumers.left_right_fill(lt, rt, tol, inval, out=lt)
        assert got.data_ptr() == lt.data_ptr()
    else:
        got = consumers.left_right_fill(lt, rt, tol, inval)
        assert mismatch(lt.cpu().numpy(), dl) == 0        # the input is left alone
    return got.cpu().numpy()


def _crafted_cases():
    """(values, keep, invalid) for every clause of the rule; values in (-0.5, 0.5) so that craft() applies."""
    cases = []
    k = np.array([True, False, False, True])
    cases.append((np.float32([[0.3, 0.0, 0.0, 0.1], [0.1, 0.4, 0.4, 0.3]]), np.stack([k, k]), -1.0))   # min both ways
    cases.append((np.float32([[-0.0, 0.2, 0.0], [0.0, 0.2, -0.0], [0.25, 0.0, 0.25]]),
                  np.array([[True, False, True]] * 3), -1.0))                                         # ties, +-0
    cases.append((np.float32([[0.4, 0.4, 0.2, 0.1, 0.4, 0.4]]),
                  np.array([[False, False, True, True, False, False]]), -1.0))                        # border runs
    cases.append((np.float32([[0.4, 0.4, 0.4, -0.3, 0.4]]), np.array([[False, False, False, True, False]]), -1.0))
    v = np.full((6, 3), 0.4, np.float32)
    kk = np.zeros((6, 3), bool)
    v[1], kk[1] = [0.1, 0.4, 0.2], [True, False, True]
    v[4], kk[4] = [0.3, 0.4, 0.4], [True, False, False]
    cases.append((v, kk, -1.0))                                                                       # empty rows
    cases.append((v, kk, np.nan))                                                                     # NaN invalid
    cases.append((np.full((3, 5), 0.2, np.float32), np.zeros((3, 5), bool), -1.0))                    # all rejected
    cases.append((np.full((3, 5), 0.2, np.float32), np.zeros((3, 5), bool), np.nan))
    cases.append((np.float32([[0.3, 0.0, 0.4, 0.2], [0.3, 0.0, 0.0, 0.4]]),
                  np.array([[True, True, False, True], [True, False, True, True]]), 0.0))             # kept == invalid
    cases.append((np.float32([[0.125], [0.2], [-0.0]]), np.array([[False], [True], [False]]), -1.0))  # W = 1
    return cases


@pytest.mark.parametrize("in_place", [False, True])
def test_crafted_rows(in_place):
    for i, (values, keep, inval) in enumerate(_crafted_cases()):
        dl, dr = craft(values, keep)
        want = reference_background_fill(dl, dr, 0.0, inval)
        got = _gpu_fill(dl, dr, 0.0, inval, in_place)
        assert same_bits(got, want), (i, got, want)


@pytest.mark.parametrize("W", [1, 7, 2047, 2048, 2049, 5000, 8192])
@pytest.mark.parametrize("in_place", [False, True])
def test_random_maps_every_width(W, in_place):
    """Rows of every density, from one kept pixel to all kept, over row widths of one to four 2048-column tiles
    (runs that cross tiles stay pending until their right bound is found)."""
    rng = np.random.default_rng(W)
    n, H = 3, 24
    dl = (rng.random((n, H, W)) * min(16, W)).astype(np.float32)
    dl[rng.random(dl.shape) < 0.02] = np.nan
    dl[:, :, ::13] = 2.5                                   # rint ties
    c = np.arange(W)
    yr = np.clip(c - np.rint(np.nan_to_num(dl)).astype(np.int64), 0, W - 1)
    dr = np.full((n, H, W), 1e6, np.float32)               # nothing kept unless set below
    density = rng.choice([0.0, 0.0005, 0.01, 0.3, 0.9, 1.0], size=(n, H))
    want_keep = (rng.random((n, H, W)) < density[..., None])
    f_idx, r_idx, c_idx = np.nonzero(want_keep)
    dr[f_idx, r_idx, yr[f_idx, r_idx, c_idx]] = dl[f_idx, r_idx, c_idx] + rng.integers(-1, 2, c_idx.size)
    dr[rng.random(dr.shape) < 0.01] = -0.0
    for tol, inval in ((1.0, -1.0), (0.5, np.nan), (2.0, 0.0)):
        keep = keep_mask(dl, dr, tol)
        assert (keep.any() or W == 1) and not keep.all()
        want = reference_background_fill(dl, dr, tol, inval)
        got = _gpu_fill(dl, dr, tol, inval, in_place)
        assert same_bits(got, want), (tol, inval, int((got.view(np.uint32) != want.view(np.uint32)).sum()))


def test_two_dimensional_maps_and_argument_errors():
    import torch
    from stereo_depth_b200 import _native as N
    from stereo_depth_b200 import consumers
    rng = np.random.default_rng(9)
    dl = (rng.random((40, 300)) * 8).astype(np.float32)
    dr = (rng.random((40, 300)) * 8).astype(np.float32)
    assert same_bits(_gpu_fill(dl, dr, 1.0, -1.0, False), reference_background_fill(dl, dr, 1.0, -1.0))
    lt, rt = torch.from_numpy(dl).cuda(), torch.from_numpy(dr).cuda()
    with pytest.raises(ValueError):
        consumers.left_right_fill(lt, rt, -1.0)
    with pytest.raises(RuntimeError):
        consumers.left_right_fill(lt, rt, 1.0, out=rt)
    with pytest.raises(RuntimeError):
        consumers.left_right_fill(lt, rt[:, :299].contiguous(), 1.0)
    lib = N.lib()
    p = lt.data_ptr()
    assert lib.sd_lr_fill(None, p, 1, 40, 300, 1.0, -1.0, p, None) == N.SD_ERR_BAD_ARG
    assert lib.sd_lr_fill(p, rt.data_ptr(), 0, 40, 300, 1.0, -1.0, p, None) == N.SD_ERR_BAD_ARG
    assert lib.sd_lr_fill(p, rt.data_ptr(), 1, 40, 0, 1.0, -1.0, p, None) == N.SD_ERR_BAD_ARG
    assert lib.sd_lr_fill(p, rt.data_ptr(), 1, 40, 300, float("inf"), -1.0, p, None) == N.SD_ERR_BAD_ARG
    assert lib.sd_lr_fill(p, rt.data_ptr(), 1, 40, 300, 1.0, -1.0, rt.data_ptr(), None) == N.SD_ERR_BAD_ARG


# ---- entry points and switching ---------------------------------------------------------------------------------------

def test_entry_points_batches_host_backend_pipeline():
    import torch
    from stereo_depth_b200 import backend, consumers, cuda_depth, pipeline
    H, W, K, D = 120, 256, 2, 48
    kw = cfg_kw(H, W, K, 0, D - 1)
    cfg = O.make_config(**kw)
    n = 7
    ls, rs = zip(*[make_pair(H, W, D, seed=40, frame=f)[:2] for f in range(n)])
    L, R = np.stack(ls), np.stack(rs)
    want = np.stack([reference_background_fill(O.run(cfg, L[f], R[f])["out"], oracle_right_map(cfg, L[f], R[f]), 0.5,
                                               -3.0) for f in range(n)])
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=4)
    assert not sm.background_fill
    sm.set_left_right_check(0.5, -3.0, background_fill=True)
    assert sm.background_fill and sm.left_right_check == 0.5
    # single frame (aliasing output buffer, like the reference)
    out = sm.compute_disparity_map(torch.from_numpy(L[3]).cuda(), torch.from_numpy(R[3]).cuda())
    assert out.data_ptr() == sm._out.data_ptr()
    assert mismatch(out.cpu().numpy(), want[3]) == 0
    # 7 frames on a 4-frame handle: chunks of 2 pairs -> 2+2+2+1
    got = sm.compute_disparity_batch(torch.from_numpy(L).cuda(), torch.from_numpy(R).cuda()).cpu().numpy()
    assert mismatch(got, want) == 0
    # host path from pinned memory
    host = sm.compute_disparity_host(torch.from_numpy(L).pin_memory(), torch.from_numpy(R).pin_memory())
    assert mismatch(host.numpy(), want) == 0
    # the backend through .native, on CPU and CUDA batches
    be = backend.CudaStereoMatchingBackend(cuda_depth.StereoMatchingConfiguration(**kw))
    be.native.set_left_right_check(0.5, -3.0, background_fill=True)
    assert mismatch(be.process_batch(torch.from_numpy(L), torch.from_numpy(R)).numpy(), want) == 0
    assert mismatch(be.process_batch(torch.from_numpy(L).cuda(), torch.from_numpy(R).cuda()).cpu().numpy(), want) == 0
    assert mismatch(be.process(torch.from_numpy(L[1]), torch.from_numpy(R[1])).cpu().numpy(), want[1]) == 0
    # the pipeline: a dense map, so the point cloud has every pixel
    pc = pipeline.DepthEstimationPipelineConfig(image_shape=(H, W), min_disparity=0, max_disparity=D - 1,
                                                left_right_check=1.0, left_right_background_fill=True)
    res = pipeline.DepthEstimationPipeline(pc).process(torch.from_numpy(L[2]), torch.from_numpy(R[2]))
    want2 = reference_background_fill(O.run(cfg, L[2], R[2])["out"], oracle_right_map(cfg, L[2], R[2]), 1.0, -1.0)
    d = res.disparity_map.cpu().numpy()
    assert mismatch(d, want2) == 0
    assert (d == -1.0).sum() == 0
    pts = consumers.point_cloud(res.disparity_map, 1.0, 1.0, invalid_disparity=pc.invalid_disparity)
    assert pts.shape[0] == H * W


def test_switching_restores_check_only_and_unchecked_paths():
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
    counts_check = [sm.launches_per_call(k) for k in range(1, 10)]
    check_only = sm.compute_disparity_batch(L, R).cpu().numpy()
    sm.set_left_right_check(1.0, background_fill=True)
    counts_fill = [sm.launches_per_call(k) for k in range(1, 10)]
    filled = sm.compute_disparity_batch(L, R).cpu().numpy()
    assert (check_only == -1.0).sum() > 0 and (filled == -1.0).sum() == 0
    # check + fill -> check only: exactly the check-only output
    sm.set_left_right_check(1.0)
    assert not sm.background_fill
    assert [sm.launches_per_call(k) for k in range(1, 10)] == counts_check
    assert mismatch(sm.compute_disparity_batch(L, R).cpu().numpy(), check_only) == 0
    # a new tolerance keeps the fill on (C ABI: sd_set_lr_check with the check on keeps the fill setting)
    sm.set_left_right_check(1.0, background_fill=True)
    sm._handle.set_lr_check(True, 1.0, -1.0)
    assert mismatch(sm.compute_disparity_batch(L, R).cpu().numpy(), filled) == 0
    # check off: the never-checked output and launch counts
    sm.set_left_right_check(None)
    assert not sm.background_fill
    assert [sm.launches_per_call(k) for k in range(1, 10)] == counts_off
    assert mismatch(sm.compute_disparity_batch(L, R).cpu().numpy(), base) == 0
    # documented count: the check's launches + the row and column passes per chunk of frames_per_launch/2 pairs
    for k in range(1, 10):
        nch = -(-k // 2)
        assert counts_fill[k - 1] == counts_check[k - 1] + 2 * nch, k
    # the fill without the check is refused; the check off switches the fill off
    with pytest.raises(RuntimeError, match="left-right check"):
        sm._handle.set_lr_fill(True)
    sm.set_left_right_check(1.0)
    assert [sm.launches_per_call(k) for k in range(1, 10)] == counts_check


def test_errors():
    from stereo_depth_b200 import _native as N
    from stereo_depth_b200 import cuda_depth, pipeline
    kw = cfg_kw(64, 128, 2, 0, 31)
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=2)
    lib = N.lib()
    h = sm._handle._h
    assert lib.sd_set_lr_fill(h, 1) == N.SD_ERR_UNSUPPORTED
    assert lib.sd_set_lr_fill(h, 0) == N.SD_ERR_UNSUPPORTED
    assert lib.sd_set_lr_fill(None, 1) == N.SD_ERR_BAD_ARG
    with pytest.raises(ValueError):
        sm.set_left_right_check(-1.0, background_fill=True)
    assert not sm.background_fill and sm.left_right_check is None
    assert lib.sd_set_lr_check(h, 1, 1.0, -1.0) == N.SD_OK
    assert lib.sd_set_lr_fill(h, 1) == N.SD_OK
    assert lib.sd_set_lr_check(h, 0, 0.0, 0.0) == N.SD_OK
    assert lib.sd_set_lr_fill(h, 1) == N.SD_ERR_UNSUPPORTED
    with pytest.raises(RuntimeError, match="left_right_background_fill needs left_right_check"):
        pipeline.DepthEstimationPipeline(pipeline.DepthEstimationPipelineConfig(image_shape=(64, 128), min_disparity=0,
                                                                                max_disparity=31,
                                                                                left_right_background_fill=True))


@pytest.mark.parametrize("shape,dtype", [
    ((75, 133, 2, 0, 30), "u8"),     # ragged: W % 16 != 0, H odd -> generic ingest
    ((75, 133, 2, 0, 30), "f32"),
    ((24, 44, 2, 0, 17), "u8"),      # smaller than a tile
    ((136, 264, 2, 0, 63), "f32"),   # tile overhang, W % 16 == 8 -> f32 fast path, u8 generic
    ((136, 264, 2, 0, 63), "u8"),
    ((90, 120, 3, 0, 29), "f32"),
    ((64, 256, 2, 0, 63), "u8"),     # u8 fast path
])
def test_guard_bands_with_the_fill(shape, dtype, monkeypatch):
    import torch
    from stereo_depth_b200 import cuda_depth
    monkeypatch.setenv("SD_DEBUG_GUARDS", "1")
    H, W, K, mn, mx = shape
    kw = cfg_kw(H, W, K, mn, mx)
    l, r, _ = make_pair(H, W, mx + 1, seed=900 + H)
    lt, rt = _tensors(l, r, dtype)
    for fpl in (2, 5):
        sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=fpl)
        sm.set_left_right_check(1.0, background_fill=True)
        sm.compute_disparity_batch(torch.stack([lt] * 3), torch.stack([rt] * 3))
        sm.compute_disparity_host(torch.stack([lt] * 3).cpu(), torch.stack([rt] * 3).cpu())
        sm.stage("right", 0)
        torch.cuda.synchronize()
        assert sm._handle.check_guards() == 0, (shape, dtype, fpl)


def test_layered_scene_at_1080p():
    import torch
    from stereo_depth_b200 import cuda_depth
    H, W, K, D = 1080, 1920, 2, 128
    l, r, gt, visible = make_layered_pair(H, W, D, seed=3)
    kw = cfg_kw(H, W, K, 0, D - 1)
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw))
    lt, rt = torch.from_numpy(l).cuda(), torch.from_numpy(r).cuda()
    plain = sm.compute_disparity_map(lt, rt).cpu().numpy().copy()
    sm.set_left_right_check(1.0, background_fill=True)
    filled = sm.compute_disparity_map(lt, rt).cpu().numpy().copy()
    right = sm.stage("right").cpu().numpy()
    assert mismatch(filled, reference_background_fill(plain, right, 1.0)) == 0
    cfg = O.make_config(**kw)
    assert mismatch(plain, O.run(cfg, l, r)["out"]) == 0
    assert mismatch(right, oracle_right_map(cfg, l, r)) == 0
    # the CPU test's quality numbers, at full size
    q = fill_quality(plain, right, gt, visible)
    print("1080p layered:", {k: round(v, 4) for k, v in q.items()})
    assert q["occluded_filled"] >= q["occluded_plain"] + 0.15, q
    assert q["all_filled"] >= q["all_plain"] + 0.005, q
    assert q["visible_filled"] >= q["visible_plain"] - 0.012, q
    # the check alone: filled pixels are exactly the rejected ones
    checked = reference_check(plain, right, 1.0, np.nan)
    assert same_bits(filled[~np.isnan(checked)], plain[~np.isnan(checked)])
