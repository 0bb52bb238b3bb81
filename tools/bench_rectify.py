#!/usr/bin/env python
"""Cost of rectification (StereoMatching.set_rectification): off and on, alternated in the same process on the same
handle.  Inputs resident in HBM, CUDA events, warm-up, median of 5 repeats, best of 2 alternations.  With it on the
handle gets the raw views of synthetic.make_unrectified_pair (cameras rotated by about a degree: realistic gather
strides); with it off it gets the same raw views rectified beforehand by consumers.rectify, so both states match the
same rectified scene bit for bit and differ only by the remap (the level screen's pruning, and so the fused kernel's
time, depends on the scene).

    python tools/bench_rectify.py [--out profiles/rectify_b200.json]

Legs: C3 (1080p, D=128, 64 frames per step) batches in uint8 and float32; C5 (720p) uint8; one frame per call at 1080p;
the per-kernel split (profile_read_detail) at C3, where the remap counts in the gray_pool bucket; the host path end to
end at C3; the remap alone through consumers.rectify.  Records the GPU name and power limit beside the numbers."""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
from bench_lr import REPEATS, WORKLOADS, gpu_info, timed  # noqa: E402
from stereo_depth_b200 import consumers, cuda_depth  # noqa: E402
from stereo_depth_b200.synthetic import make_unrectified_pair, rotated_rig_maps  # noqa: E402

STATES = ("off", "on")
_maps = {}


def maps(H, W):
    if (H, W) not in _maps:
        _maps[(H, W)] = rotated_rig_maps(H, W)
    return _maps[(H, W)]


_raw = {}


def inputs(H, W, D, n, distinct=8):
    """(raw, rectified) [n,3,H,W] uint8 batches of both views on the device."""
    if (H, W) not in _raw:
        pairs = [make_unrectified_pair(H, W, D, seed=70 + f)[:2] for f in range(distinct)]
        _raw[(H, W)] = [torch.from_numpy(np.stack(v)).cuda() for v in zip(*pairs)]
    reps = -(-n // distinct)
    raw = [torch.cat([v] * reps)[:n].contiguous() for v in _raw[(H, W)]]
    dev = [tuple(torch.from_numpy(m).cuda() for m in p) for p in maps(H, W)]
    rect = [consumers.rectify(v, *m) for v, m in zip(raw, dev)]
    return raw, rect


def matcher(name):
    H, W, K, D = WORKLOADS[name]
    return cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(height=H, width=W, downscale_factor=K,
                                                                            min_disparity=0, max_disparity=D - 1))


def set_state(sm, state):
    if state == "on":
        sm.set_rectification(*maps(sm.height, sm.width))
    else:
        sm.set_rectification(None, None)


def alternate(sm, fn, iters, warm):
    """fn(state) runs one step of `state`; returns the best of 2 alternations of timed(..., iters) per state."""
    for state in STATES:
        set_state(sm, state)
        for _ in range(warm):
            fn(state)
    res = {s: [] for s in STATES}
    for _ in range(2):
        for state in STATES:
            set_state(sm, state)
            res[state].append(timed(lambda: fn(state), iters))
    return {s: min(v) for s, v in res.items()}


def pick(raw, rect, state):
    return raw if state == "on" else rect


def batch_leg(name, frames, iters, dtype):
    H, W, K, D = WORKLOADS[name]
    sm = matcher(name)
    raw, rect = inputs(H, W, D, frames)
    if dtype == "f32":
        raw, rect = [v.float() for v in raw], [v.float() for v in rect]
    out = torch.empty((frames, H, W), dtype=torch.float32, device="cuda")
    t = alternate(sm, lambda s: sm.compute_disparity_batch(*pick(raw, rect, s), out), iters, 3)
    return {"workload": name, "dtype": dtype, "frames_per_step": frames, "frames_per_launch": sm.frames_per_launch,
            "ms_per_step_off": t["off"], "ms_per_step_on": t["on"], "frames_per_s_off": frames / t["off"] * 1e3,
            "frames_per_s_on": frames / t["on"] * 1e3, "rate_on_over_off": t["off"] / t["on"]}


def single_frame_leg(name, iters=200):
    H, W, K, D = WORKLOADS[name]
    sm = matcher(name)
    raw, rect = inputs(H, W, D, 1)
    raw, rect = [v[0].contiguous() for v in raw], [v[0].contiguous() for v in rect]
    t = alternate(sm, lambda s: sm.compute_disparity_map(*pick(raw, rect, s)), iters, 10)
    return {"workload": name, "one_frame_per_call": True, "ms_per_frame_off": t["off"], "ms_per_frame_on": t["on"],
            "on_minus_off_ms": t["on"] - t["off"]}


def profile_leg(name="C3", frames=64, iters=10):
    H, W, K, D = WORKLOADS[name]
    sm = matcher(name)
    raw, rect = inputs(H, W, D, frames)
    out = torch.empty((frames, H, W), dtype=torch.float32, device="cuda")
    res = {}
    for state in STATES:
        set_state(sm, state)
        L, R = pick(raw, rect, state)
        for _ in range(3):
            sm.compute_disparity_batch(L, R, out)
        torch.cuda.synchronize()
        sm.profile(True)
        sm.profile_read_detail()
        for _ in range(iters):
            sm.compute_disparity_batch(L, R, out)
        d = sm.profile_read_detail()
        sm.profile(False)
        res[state] = {k: {"us_per_frame": ms * 1e3 / (frames * iters), "launches": n} for k, (ms, n) in d.items()}
    res["derived"] = {"remap_us_per_frame": res["on"]["gray_pool"]["us_per_frame"] -
                      res["off"]["gray_pool"]["us_per_frame"]}
    return {"workload": name, "frames_per_step": frames, "per_kernel": res}


def host_leg(name="C3", frames=64):
    H, W, K, D = WORKLOADS[name]
    sm = matcher(name)
    raw, rect = [[v.cpu().pin_memory() for v in x] for x in inputs(H, W, D, frames)]
    out = torch.empty((frames, H, W), dtype=torch.float32).pin_memory()
    t = alternate(sm, lambda s: sm.compute_disparity_host(*pick(raw, rect, s), out), 2, 1)
    return {"workload": name, "host_path": True, "frames_per_call": frames, "frames_per_s_off": frames / t["off"] * 1e3,
            "frames_per_s_on": frames / t["on"] * 1e3, "rate_on_over_off": t["off"] / t["on"]}


def remap_leg(name="C3", frames=29, iters=20):
    """consumers.rectify of both views of `frames` frames (two launches, one per view), against the compulsory bytes."""
    H, W, K, D = WORKLOADS[name]
    (L, R), _ = inputs(H, W, D, frames)
    (lx, ly), (rx, ry) = [tuple(torch.from_numpy(m).cuda() for m in p) for p in maps(H, W)]
    rows = []
    for dtype in ("u8", "f32"):
        a, b = (L, R) if dtype == "u8" else (L.float(), R.float())
        oa, ob = torch.empty_like(a), torch.empty_like(b)

        def fn():
            consumers.rectify(a, lx, ly, out=oa)
            consumers.rectify(b, rx, ry, out=ob)
        for _ in range(3):
            fn()
        ms = timed(fn, iters)
        frame_bytes = 2 * 3 * H * W * a.element_size()
        compulsory = frames * 2 * frame_bytes + 4 * H * W * 4      # read + write the frames, read the maps once
        rows.append({"dtype": dtype, "frames": frames, "us_per_frame": ms * 1e3 / frames,
                     "compulsory_bytes_per_frame": compulsory / frames, "achieved_TB_per_s": compulsory / (ms * 1e-3) / 1e12})
    return {"workload": name, "remap_alone": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_rectify.py needs a CUDA device")
    rec = {"gpu": gpu_info(), "repeats": REPEATS, "statistic": "median of repeats, best of 2 alternations", "legs": []}
    legs = [lambda: batch_leg("C3", 64, 5, "u8"), lambda: batch_leg("C3", 64, 5, "f32"),
            lambda: batch_leg("C5", 64, 10, "u8"), lambda: single_frame_leg("C3"), profile_leg, host_leg, remap_leg]
    for leg in legs:
        rec["legs"].append(leg())
        print(json.dumps(rec["legs"][-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
