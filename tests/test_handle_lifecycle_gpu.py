"""A closed handle gives its device memory back (-m gpu), also after the switches that allocate and free buffers of
their own (left-right check, background fill, reference-compat mode) and after the host path was rebuilt for a second
dtype, with and without debug guard bands.

Free device memory is compared with a tolerance of 1 MiB.  A 1080p handle's scratch is gigabytes, so a leaked scratch
plane, volume, right map or host-path slot shows; the smallest buffers (the fill's per-row flags, a few KB) would not."""
import gc

import pytest

pytestmark = pytest.mark.gpu

MiB = 1 << 20


def _free_bytes(torch):
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return torch.cuda.mem_get_info()[0]


def _cycle(torch, cuda_depth, guards):
    sm = cuda_depth.StereoMatching()   # default configuration: 1080p, min_disparity 75, so reference-compat mode is on
    gen = torch.Generator().manual_seed(11)
    shape = (2, 3, sm.height, sm.width)
    left = torch.randint(0, 256, shape, dtype=torch.uint8, generator=gen)
    right = torch.randint(0, 256, shape, dtype=torch.uint8, generator=gen)
    sm.profile(True)
    sm.set_left_right_check(1.0, background_fill=True)
    sm.compute_disparity_batch(left.cuda(), right.cuda())
    sm.compute_disparity_host(left, right)
    sm.compute_disparity_host(left.float(), right.float())   # rebuilds the host pipeline for float32
    assert sm.profile_read()["fill"][1] > 0
    sm.set_left_right_check(None)
    sm.set_compat(False)
    if guards:
        assert sm._handle.check_guards() == 0
    sm._handle.close()


@pytest.mark.parametrize("guards", [False, True], ids=["plain", "guards"])
def test_closed_handle_returns_its_device_memory(guards, monkeypatch):
    import torch
    from stereo_depth_b200 import cuda_depth
    if guards:
        monkeypatch.setenv("SD_DEBUG_GUARDS", "1")
    else:
        monkeypatch.delenv("SD_DEBUG_GUARDS", raising=False)
    _cycle(torch, cuda_depth, guards)   # warm-up: module load, torch's caching allocator
    base = _free_bytes(torch)
    for _ in range(3):
        _cycle(torch, cuda_depth, guards)
    drift = base - _free_bytes(torch)
    assert abs(drift) <= MiB, f"free device memory changed by {drift / MiB:.2f} MiB over 3 handle lifetimes"
