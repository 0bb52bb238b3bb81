#!/usr/bin/env python
"""Cost of the left-right consistency check (StereoMatching.set_left_right_check): check off, on, and on with the
background fill, alternated in the same process on the same handle.  Inputs resident in HBM, CUDA events, warm-up,
median of 5 repeats.

    python tools/bench_lr.py [--out profiles/lr_fill_b200.json]

Legs: C3 (1080p, D=128, 64 frames per step), C5 (720p) and C1 (480p) batches; one frame per call at 1080p and 720p; the
per-kernel split (profile_read_detail) at C3; the host path end to end at C3; the natural pair when data/_ref has it.
Records the GPU name and power limit beside the numbers."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from stereo_depth_b200 import cuda_depth  # noqa: E402
from stereo_depth_b200.synthetic import load_natural_pair, make_batch  # noqa: E402

WORKLOADS = {"C3": (1080, 1920, 2, 128), "C5": (720, 1280, 2, 128), "C1": (480, 640, 2, 64)}
REPEATS = 5


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # the numbers are still device-timed; say what is missing
        q = f"nvidia-smi unavailable: {e}"
    return {"torch_device_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def timed(fn, iters):
    """Median over REPEATS of the device time of `iters` calls (CUDA events), in ms per call."""
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = []
    for _ in range(REPEATS):
        start.record()
        for _ in range(iters):
            fn()
        stop.record()
        stop.synchronize()
        res.append(start.elapsed_time(stop) / iters)
    return float(np.median(res))


def inputs(H, W, D, n, distinct=8):
    l, r = make_batch(distinct, H, W, D, seed=70)
    reps = -(-n // distinct)
    return (torch.from_numpy(np.concatenate([l] * reps)[:n]).cuda(), torch.from_numpy(np.concatenate([r] * reps)[:n]).cuda())


STATES = ("off", "on", "fill")   # no check, check, check + background fill


def set_check(sm, state):
    sm.set_left_right_check(None if state == "off" else 1.0, background_fill=state == "fill")


def batch_leg(name, frames, iters):
    H, W, K, D = WORKLOADS[name]
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(height=H, width=W, downscale_factor=K,
                                                                          min_disparity=0, max_disparity=D - 1))
    L, R = inputs(H, W, D, frames)
    out = torch.empty((frames, H, W), dtype=torch.float32, device="cuda")
    fn = lambda: sm.compute_disparity_batch(L, R, out)   # noqa: E731
    res = {s: [] for s in STATES}
    for state in STATES:        # warm-up of every path
        set_check(sm, state)
        for _ in range(3):
            fn()
    for _ in range(2):          # alternated
        for state in STATES:
            set_check(sm, state)
            res[state].append(timed(fn, iters))
    set_check(sm, "on")
    fn()
    invalid = float((out == -1.0).float().mean().item())
    off, on, fill = min(res["off"]), min(res["on"]), min(res["fill"])
    return {"workload": name, "frames_per_step": frames, "frames_per_launch": sm.frames_per_launch,
            "ms_per_step_off": off, "ms_per_step_on": on, "ms_per_step_fill": fill,
            "frames_per_s_off": frames / off * 1e3, "frames_per_s_on": frames / on * 1e3,
            "frames_per_s_fill": frames / fill * 1e3, "on_over_off": on / off,
            "fill_rate_over_check_rate": on / fill, "invalid_fraction": invalid}


def single_frame_leg(name, iters=200):
    H, W, K, D = WORKLOADS[name]
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(height=H, width=W, downscale_factor=K,
                                                                          min_disparity=0, max_disparity=D - 1))
    L, R = inputs(H, W, D, 1)
    l0, r0 = L[0].contiguous(), R[0].contiguous()
    fn = lambda: sm.compute_disparity_map(l0, r0)   # noqa: E731
    res = {}
    for state in STATES:
        set_check(sm, state)
        for _ in range(10):
            fn()
    for _ in range(2):
        for state in STATES:
            set_check(sm, state)
            res.setdefault(state, []).append(timed(fn, iters))
    t = {s: min(v) for s, v in res.items()}
    return {"workload": name, "one_frame_per_call": True, "ms_per_frame_off": t["off"], "ms_per_frame_on": t["on"],
            "ms_per_frame_fill": t["fill"], "on_over_off": t["on"] / t["off"], "fill_over_on": t["fill"] / t["on"]}


def profile_leg(name="C3", frames=64, iters=10):
    H, W, K, D = WORKLOADS[name]
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(height=H, width=W, downscale_factor=K,
                                                                          min_disparity=0, max_disparity=D - 1))
    L, R = inputs(H, W, D, frames)
    out = torch.empty((frames, H, W), dtype=torch.float32, device="cuda")
    res = {}
    for state in STATES:
        set_check(sm, state)
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
    # kernel A with the check runs forward + mirrored frames in one launch: mirrored / forward = on / off - 1
    a_off, a_on = res["off"]["gray_pool"]["us_per_frame"], res["on"]["gray_pool"]["us_per_frame"]
    f_off, f_on = res["off"]["fill"]["us_per_frame"], res["on"]["fill"]["us_per_frame"]
    res["derived"] = {"mirrored_over_forward_kernel_a": a_on / a_off - 1.0,
                      "fill_plus_check_minus_plain_fill_us_per_frame": f_on - 2.0 * f_off,
                      "fill_bucket_background_fill_minus_check_us_per_frame":
                          res["fill"]["fill"]["us_per_frame"] - f_on}
    return {"workload": name, "frames_per_step": frames, "per_kernel": res}


def host_leg(name="C3", frames=64):
    H, W, K, D = WORKLOADS[name]
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(height=H, width=W, downscale_factor=K,
                                                                          min_disparity=0, max_disparity=D - 1))
    L, R = inputs(H, W, D, frames)
    Lh, Rh = L.cpu().pin_memory(), R.cpu().pin_memory()
    out = torch.empty((frames, H, W), dtype=torch.float32).pin_memory()
    fn = lambda: sm.compute_disparity_host(Lh, Rh, out)   # noqa: E731
    res = {}
    for state in STATES:
        set_check(sm, state)
        fn()
    for _ in range(2):
        for state in STATES:
            set_check(sm, state)
            res.setdefault(state, []).append(timed(fn, 2))
    t = {s: min(v) for s, v in res.items()}
    return {"workload": name, "host_path": True, "frames_per_call": frames, "frames_per_s_off": frames / t["off"] * 1e3,
            "frames_per_s_on": frames / t["on"] * 1e3, "frames_per_s_fill": frames / t["fill"] * 1e3,
            "on_over_off": t["on"] / t["off"], "fill_over_on": t["fill"] / t["on"]}


def natural_leg():
    nat = load_natural_pair()
    if nat is None:
        return {"natural_pair": "not available (data/_ref)"}
    l, r, vmin, vmax = nat
    H, W = l.shape[1:]
    rows = []
    for mn, mx in ((vmin, vmax), (0, 127)):
        sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(height=H, width=W, downscale_factor=2,
                                                                              min_disparity=mn, max_disparity=mx))
        lt, rt = torch.from_numpy(l).cuda(), torch.from_numpy(r).cuda()
        fn = lambda: sm.compute_disparity_map(lt, rt)   # noqa: E731
        res = {}
        for state in STATES:
            set_check(sm, state)
            for _ in range(5):
                fn()
        for _ in range(2):
            for state in STATES:
                set_check(sm, state)
                res.setdefault(state, []).append(timed(fn, 50))
        set_check(sm, "on")
        inv = float((fn() == -1.0).float().mean().item())
        t = {s: min(v) for s, v in res.items()}
        rows.append({"natural_pair": f"{W}x{H} {mn}..{mx}", "ms_per_frame_off": t["off"], "ms_per_frame_on": t["on"],
                     "ms_per_frame_fill": t["fill"], "on_over_off": t["on"] / t["off"],
                     "fill_over_on": t["fill"] / t["on"], "invalid_fraction": inv})
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_lr.py needs a CUDA device")
    rec = {"gpu": gpu_info(), "repeats": REPEATS, "statistic": "median of repeats, best of 2 alternations",
           "legs": []}
    for name, frames, iters in (("C3", 64, 5), ("C5", 64, 10), ("C1", 64, 20)):
        rec["legs"].append(batch_leg(name, frames, iters))
        print(json.dumps(rec["legs"][-1]), flush=True)
    for name in ("C3", "C5"):
        rec["legs"].append(single_frame_leg(name))
        print(json.dumps(rec["legs"][-1]), flush=True)
    rec["legs"].append(profile_leg())
    print(json.dumps(rec["legs"][-1]), flush=True)
    rec["legs"].append(host_leg())
    print(json.dumps(rec["legs"][-1]), flush=True)
    rec["legs"].append(natural_leg())
    print(json.dumps(rec["legs"][-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
