"""Left-right check and background fill in the peer-memory row-band mode (-m gpu): the band outputs and the band rows of
the right view's map are bit-identical to a single-GPU StereoMatching with the same settings on the whole frame, on one
GPU (world 1) and on 2-4 GPUs (spawned ranks, as tests/test_multi_gpu.py); the refusals of the other band paths stay;
guard bands stay clean and memory comes back."""
import ctypes as C
import gc
import os
import socket

import numpy as np
import pytest

from oracle import oracle as O
from test_lr_check_cpu import oracle_right_map
from test_lr_fill_cpu import keep_mask

pytestmark = pytest.mark.gpu

TOL, INVALID = 1.0, -1.0
MiB = 1 << 20


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _same(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


def _tensors(l, r, dtype):
    import torch
    lt, rt = torch.from_numpy(np.ascontiguousarray(l)).cuda(), torch.from_numpy(np.ascontiguousarray(r)).cuda()
    if dtype == "f32":
        lt, rt = lt.float(), rt.float()
    return lt.contiguous(), rt.contiguous()


def _single(kw, frames, dtype, fill):
    """Outputs and right maps of a single-GPU matcher with the same settings on the whole frames."""
    from stereo_depth_b200 import cuda_depth
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=2)
    sm.set_compat(False)
    sm.set_left_right_check(TOL, INVALID, background_fill=fill)
    outs, rights = [], []
    for l, r in frames:
        lt, rt = _tensors(l, r, dtype)
        outs.append(sm.compute_disparity_map(lt, rt).cpu().numpy().copy())
        rights.append(sm.stage("right").cpu().numpy().copy())
    return outs, rights


def _banded(kw, fill):
    """The band matcher with the check (relative-index secondary reads, as _single: the empty-band scene has
    min_disparity != 0, where the reference-compat default is on)."""
    from stereo_depth_b200 import cuda_depth
    from stereo_depth_b200.bands import BandedStereoMatching
    sm = BandedStereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), p2p=True, left_right_check=TOL,
                              invalid_disparity=INVALID, background_fill=fill)
    sm.handle.set_compat(False)
    return sm


def _band_frames(sm, frames, dtype):
    """Band outputs and band rows of the right map of consecutive compute() calls (this rank's rows)."""
    p = sm.plan
    outs, rights = [], []
    for l, r in frames:
        lt, rt = _tensors(l[:, p.x0 * p.K:p.x1 * p.K], r[:, p.x0 * p.K:p.x1 * p.K], dtype)
        outs.append(sm.compute(lt, rt).cpu().numpy().copy())
        rights.append(sm.right_map().cpu().numpy().copy())
    return outs, rights


def _layered(H, W, D, seeds):
    from stereo_depth_b200.synthetic import make_layered_pair
    return [make_layered_pair(H, W, D, s)[:2] for s in seeds]


# ---- a scene whose rows without a kept pixel lie on another rank than the first / last non-empty row ---------------
# Random texture with a circular horizontal shift s per row: s = 12 in the middle, s = 36 >= W = 32 in the `edge`
# rows.  min_disparity 8 rules out the alias 36 - 32 = 4, so those rows match at d = 36, and every left pixel's partner
# c - 36 lies outside the image: the check keeps nothing there.  K = 1 keeps the bands short (12 halo rows).
EMPTY_BAND = 16   # rows per rank


def empty_band_kw(world):
    return dict(height=EMPTY_BAND * world, width=32, downscale_factor=1, min_disparity=8, max_disparity=40)


def empty_band_scene(world, seed, bottom=False):
    H, W = EMPTY_BAND * world, 32
    rng = np.random.default_rng(seed)
    left = rng.integers(0, 256, (3, H, W), dtype=np.uint8)
    s = np.where(np.arange(H) < EMPTY_BAND + 8, 36, 12)   # all of rank 0's band and 8 rows of rank 1's
    cols = (np.arange(W)[None, :] + s[:, None]) % W
    right = np.take_along_axis(left, np.broadcast_to(cols, left.shape), axis=2)
    if bottom:   # the same upside down: the last rank's band is empty
        left, right = left[:, ::-1], right[:, ::-1]
    return np.ascontiguousarray(left), np.ascontiguousarray(right)


def empty_band_frames(world):
    return [empty_band_scene(world, 7), empty_band_scene(world, 8, bottom=True), empty_band_scene(world, 9)]


def _assert_empty_band_case(world):
    """From the oracle's maps: rank 0's (or the last rank's) rows keep no pixel, and the first (last) non-empty row lies
    on another rank -- so the column pass must copy a row published by another rank."""
    from stereo_depth_b200.bands import BandPlan
    kw = empty_band_kw(world)
    cfg = O.make_config(**kw)
    plans = [BandPlan.make(kw["height"], kw["width"], 1, world, q, 12) for q in range(world)]
    for i, (l, r) in enumerate(empty_band_frames(world)):
        dl = O.run(cfg, l, r)["out"]
        rows = keep_mask(dl, oracle_right_map(cfg, l, r), TOL).any(axis=1)
        nz = np.flatnonzero(rows)
        assert nz.size > 0
        if i == 1:   # bottom: rows below the last non-empty row, which lies on an earlier rank
            assert not rows[plans[-1].x0:].any() and nz[-1] < plans[-1].x0, (i, rows.astype(int))
        else:
            assert not rows[:plans[0].x1].any() and nz[0] >= plans[0].x1, (i, rows.astype(int))


# ---- one GPU, world 1 -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("fill", [False, True])
@pytest.mark.parametrize("dtype", ["u8", "f32"])
@pytest.mark.parametrize("K", [1, 2])
def test_world1_equals_single_gpu(K, dtype, fill):
    import torch
    H, W, D = 256, 512, 64
    kw = dict(height=H, width=W, downscale_factor=K, min_disparity=0, max_disparity=D - 1)
    frames = _layered(H, W, D, (1, 2, 3))
    checked, checked_right = _single(kw, frames, dtype, False)
    want, want_right = _single(kw, frames, dtype, True) if fill else (checked, checked_right)
    for c, w in zip(checked, want):   # the check rejects a few percent of the pixels, and the fill changes them
        rejected = c == np.float32(INVALID)
        assert 0.03 < rejected.mean() < 0.12, rejected.mean()
        if fill:
            assert np.all(w[rejected] != np.float32(INVALID))
    sm = _banded(kw, fill)
    assert sm.handle.frames_per_launch == 2 and sm.background_fill == fill
    # several calls with different scenes: both parities of the published gray planes and fill areas
    order = [0, 1, 2, 0, 2]
    got, got_right = _band_frames(sm, [frames[i] for i in order], dtype)
    for j, i in enumerate(order):
        assert _same(got[j], want[i]), (j, i)
        assert _same(got_right[j], want_right[i]), ("right", j, i)
    sm.close()
    torch.cuda.synchronize()


def test_world1_rows_without_kept_pixels():
    """World 1 on the empty-band scene: the column pass takes the frame's first / last non-empty row from the rank's
    own published copy."""
    _assert_empty_band_case(2)
    kw, frames = empty_band_kw(2), empty_band_frames(2)
    for fill in (False, True):
        want, want_right = _single(kw, frames, "u8", fill)
        sm = _banded(kw, fill)
        got, got_right = _band_frames(sm, frames, "u8")
        for j in range(len(frames)):
            assert _same(got[j], want[j]) and _same(got_right[j], want_right[j]), (fill, j)
        if fill:
            assert not np.any(want[0][:EMPTY_BAND] == np.float32(INVALID))
        sm.close()


# ---- refusals -------------------------------------------------------------------------------------------------------

def test_refusals():
    import torch
    from stereo_depth_b200 import _native as N
    from stereo_depth_b200 import cuda_depth
    from stereo_depth_b200.bands import BandedStereoMatching
    from stereo_depth_b200.synthetic import make_pair
    H, W, D = 64, 128, 32
    kw = dict(height=H, width=W, downscale_factor=2, min_disparity=0, max_disparity=D - 1)
    cfg = cuda_depth.StereoMatchingConfiguration(**kw)
    with pytest.raises(RuntimeError, match="peer-memory"):
        BandedStereoMatching(cfg, p2p=False, left_right_check=1.0)
    for bad in (-1.0, float("nan"), float("inf")):
        with pytest.raises(ValueError):
            BandedStereoMatching(cfg, p2p=True, left_right_check=bad)
    with pytest.raises(RuntimeError, match="needs left_right_check"):
        BandedStereoMatching(cfg, p2p=True, background_fill=True)
    lib = N.lib()
    # the check and the fill are fixed at sd_band_p2p_init: refused afterwards, on or off, with the check on or off
    l, r, _ = make_pair(H, W, D, seed=3)
    lt, rt = _tensors(l, r, "u8")
    for tol in (None, TOL):
        sm = BandedStereoMatching(cfg, p2p=True, left_right_check=tol)
        sm.compute(lt, rt)
        h = sm.handle._h
        for on in (0, 1):
            assert lib.sd_set_lr_check(h, on, 1.0, -1.0) == N.SD_ERR_UNSUPPORTED
            assert b"before sd_band_p2p_init" in lib.sd_last_error(h)
            assert lib.sd_set_lr_fill(h, on) == N.SD_ERR_UNSUPPORTED
            assert b"before sd_band_p2p_init" in lib.sd_last_error(h)
        if tol is None:
            with pytest.raises(RuntimeError, match="left_right_check"):
                sm.right_map()
        # rectification with a band handle
        m = torch.zeros((sm.plan.local_rows, W), device="cuda")
        assert lib.sd_set_rectification(h, m.data_ptr(), m.data_ptr(), m.data_ptr(), m.data_ptr(), None) == \
            N.SD_ERR_UNSUPPORTED
        sm.close()
    # the NCCL transport with the check, in either order, and rectification before sd_band_p2p_init
    sm = cuda_depth.StereoMatching(cfg, frames_per_launch=2)
    sm.set_left_right_check(TOL)
    h = sm._handle._h
    gray = torch.zeros((H, W), device="cuda")
    dst = torch.zeros((H, W), device="cuda")
    assert lib.sd_set_band(h, 0, H, gray.data_ptr()) == N.SD_ERR_UNSUPPORTED
    assert lib.sd_compute_range(h, dst.data_ptr(), dst.data_ptr(), N.SD_U8, 1, dst.data_ptr(), None, 0, 3) == \
        N.SD_ERR_UNSUPPORTED
    sm.set_left_right_check(None)
    assert lib.sd_set_band(h, 0, H, gray.data_ptr()) == N.SD_OK
    assert lib.sd_set_lr_check(h, 1, 1.0, -1.0) == N.SD_ERR_UNSUPPORTED
    assert lib.sd_set_band(h, 0, 0, None) == N.SD_OK
    local = N.SdConfig(*[getattr(cfg._as_struct(), f) for f in N.CONFIG_FIELDS])
    local.height = H + 2 * 24
    hb = N.Handle(local, torch.cuda.current_device(), 2)
    m = torch.zeros((H + 48, W), device="cuda")
    hb.set_rectification(m.data_ptr(), m.data_ptr(), m.data_ptr(), m.data_ptr(), None)
    rows = (C.c_int32 * 2)(0, H)
    buf = C.create_string_buffer(64)
    assert lib.sd_band_p2p_init(hb._h, 1, 0, rows, 24, N.SD_U8, buf) == N.SD_ERR_UNSUPPORTED
    hb.close()


# ---- hygiene --------------------------------------------------------------------------------------------------------

def _free_bytes(torch):
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return torch.cuda.mem_get_info()[0]


def test_guard_bands_and_memory(monkeypatch):
    import torch
    from stereo_depth_b200 import cuda_depth
    from stereo_depth_b200.bands import BandedStereoMatching
    monkeypatch.setenv("SD_DEBUG_GUARDS", "1")
    H, W, D = 256, 512, 64
    kw = dict(height=H, width=W, downscale_factor=2, min_disparity=0, max_disparity=D - 1)
    frames = _layered(H, W, D, (1, 2, 3))
    ins = [_tensors(l, r, "u8") for l, r in frames]

    def cycle(check_guards):
        sm = BandedStereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), p2p=True, left_right_check=TOL,
                                  background_fill=True)
        for lt, rt in ins:
            sm.compute(lt, rt)
            sm.right_map()
        torch.cuda.synchronize()
        if check_guards:
            assert sm.handle.check_guards() == 0
        sm.close()

    cycle(False)   # (first launches load the library's modules)
    base = _free_bytes(torch)
    cycle(True)
    assert base - _free_bytes(torch) <= MiB


# ---- 2-4 GPUs -------------------------------------------------------------------------------------------------------

MULTI_H, MULTI_W, MULTI_K, MULTI_D = 288, 512, 2, 64


def _multi_cases():
    """(name, kw, dtype, fill, frames): even and uneven bands, both dtypes, check and check + fill."""
    cases = []
    for H in (MULTI_H, MULTI_H + 2 * MULTI_K):   # (uneven: pooled rows not divisible by the world size)
        kw = dict(height=H, width=MULTI_W, downscale_factor=MULTI_K, min_disparity=0, max_disparity=MULTI_D - 1)
        frames = _layered(H, MULTI_W, MULTI_D, (1, 2, 3))
        for dtype in ("u8", "f32"):
            for fill in (False, True):
                cases.append((f"h{H}_{dtype}_{'fill' if fill else 'check'}", kw, dtype, fill, frames))
    return cases


def _lr_band_worker(rank, world, port, outdir):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        cases = _multi_cases()
        cases += [(f"empty_{'fill' if f else 'check'}", empty_band_kw(world), "u8", f, empty_band_frames(world))
                  for f in (False, True)]
        for name, kw, dtype, fill, frames in cases:
            sm = _banded(kw, fill)
            for j, (l, r) in enumerate(frames):
                p = sm.plan
                lt, rt = _tensors(l[:, p.x0 * p.K:p.x1 * p.K], r[:, p.x0 * p.K:p.x1 * p.K], dtype)
                full = sm.gather(sm.compute(lt, rt))
                right = sm.gather(sm.right_map())
                torch.cuda.synchronize()
                np.save(os.path.join(outdir, f"{name}_{j}_{rank}.npy"), full.cpu().numpy())
                np.save(os.path.join(outdir, f"{name}_{j}_{rank}_right.npy"), right.cpu().numpy())
            sm.close()
    finally:
        dist.destroy_process_group()


def test_multi_gpu_equals_single_gpu(tmp_path):
    import torch
    import torch.multiprocessing as mp
    world = min(torch.cuda.device_count(), 4)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    _assert_empty_band_case(world)   # before the GPUs run: the scene really puts empty rows on another rank
    mp.spawn(_lr_band_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    cases = _multi_cases()
    cases += [(f"empty_{'fill' if f else 'check'}", empty_band_kw(world), "u8", f, empty_band_frames(world))
              for f in (False, True)]
    for name, kw, dtype, fill, frames in cases:
        want, want_right = _single(kw, frames, dtype, fill)
        for j in range(len(frames)):
            for r in range(world):
                got = np.load(tmp_path / f"{name}_{j}_{r}.npy")
                assert _same(got, want[j]), (name, j, r)
                assert _same(np.load(tmp_path / f"{name}_{j}_{r}_right.npy"), want_right[j]), ("right", name, j, r)
