#!/usr/bin/env python
"""Cost of the reprojection to 3-D (consumers.reproject_image_to_3d, sd_reproject): the pass alone on batches of
disparity maps, handleMissingValues off and on, against its compulsory bytes and a device-to-device copy measured in the
same process; and C3 frames/s of compute_disparity_batch with and without the reprojection after it, alternated.
Everything resident in HBM, CUDA events, warm-up, median of 5 repeats, best of 2 alternations.  The batches (240 MB of
maps and 720 MB of points at 29 x 1080p) are far larger than the 126 MB L2, so every pass reads from and writes to HBM.

    python tools/bench_reproject.py [--out profiles/reproject_b200.json]

Bytes per pixel: 4 read + 12 written, plus 4 read by the minimum pass with handleMissingValues.  Records the GPU name
and power limit beside the numbers."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_lr import REPEATS, WORKLOADS, gpu_info, inputs, timed  # noqa: E402
from stereo_depth_b200 import consumers, cuda_depth  # noqa: E402

DATASHEET_TB_S = 7.7


def rig_q(H, W, baseline=0.12):
    return np.array([[1, 0, 0, -(W - 1) / 2], [0, 1, 0, -(H - 1) / 2], [0, 0, 0, float(W)], [0, 0, 1 / baseline, 0]])


def copy_rate(nbytes=1 << 30, iters=20):
    """TB/s of a device-to-device copy of nbytes (read + write counted)."""
    a = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda").uniform_()
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    ms = timed(lambda: b.copy_(a), iters)
    return 2 * nbytes / (ms * 1e-3) / 1e12


def alone_leg(n, H, W, copy_tb_s, iters=20):
    gen = torch.Generator(device="cuda").manual_seed(5)
    d = torch.rand((n, H, W), device="cuda", generator=gen) * 127 + 1
    d[:, ::7, ::5] = -1.0
    out = torch.empty((n, H, W, 3), dtype=torch.float32, device="cuda")
    Q = rig_q(H, W)
    rows = []
    for hm in (False, True):
        fn = lambda: consumers.reproject_image_to_3d(d, Q, handle_missing_values=hm, out=out)   # noqa: E731
        for _ in range(3):
            fn()
        ms = timed(fn, iters)
        px = n * H * W
        nbytes = px * (16 + (4 if hm else 0))
        tb_s = nbytes / (ms * 1e-3) / 1e12
        rows.append({"frames": n, "H": H, "W": W, "handle_missing_values": hm, "us_per_frame": ms * 1e3 / n,
                     "bytes_per_frame": nbytes / n, "achieved_TB_per_s": tb_s,
                     "fraction_of_measured_copy_rate": tb_s / copy_tb_s,
                     "fraction_of_datasheet_7.7_TB_per_s": tb_s / DATASHEET_TB_S,
                     "copy_time_of_the_same_bytes_us_per_frame": nbytes / n / (copy_tb_s * 1e12) * 1e6})
    rows[1]["handle_missing_values_adds_us_per_frame"] = rows[1]["us_per_frame"] - rows[0]["us_per_frame"]
    return rows


def c3_leg(frames=64, iters=5):
    H, W, K, D = WORKLOADS["C3"]
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(height=H, width=W, downscale_factor=K,
                                                                          min_disparity=0, max_disparity=D - 1))
    L, R = inputs(H, W, D, frames)
    out = torch.empty((frames, H, W), dtype=torch.float32, device="cuda")
    pts = torch.empty((frames, H, W, 3), dtype=torch.float32, device="cuda")
    Q = rig_q(H, W)

    def step(state):
        sm.compute_disparity_batch(L, R, out)
        if state == "on":
            consumers.reproject_image_to_3d(out, Q, out=pts)
    states = ("off", "on")
    for s in states:
        for _ in range(3):
            step(s)
    res = {s: [] for s in states}
    for _ in range(2):
        for s in states:
            res[s].append(timed(lambda: step(s), iters))
    t = {s: min(v) for s, v in res.items()}
    return {"workload": "C3", "frames_per_step": frames, "frames_per_launch": sm.frames_per_launch,
            "ms_per_step_off": t["off"], "ms_per_step_on": t["on"], "frames_per_s_off": frames / t["off"] * 1e3,
            "frames_per_s_on": frames / t["on"] * 1e3, "rate_on_over_off": t["off"] / t["on"],
            "reprojection_us_per_frame_in_step": (t["on"] - t["off"]) * 1e3 / frames}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_reproject.py needs a CUDA device")
    copy = copy_rate()
    rec = {"gpu": gpu_info(), "repeats": REPEATS, "statistic": "median of repeats (C3: best of 2 alternations)",
           "device_copy_TB_per_s": copy, "datasheet_TB_per_s": DATASHEET_TB_S, "legs": []}
    print(json.dumps({"device_copy_TB_per_s": copy}), flush=True)
    for n, H, W in ((29, 1080, 1920), (64, 720, 1280)):
        rec["legs"].append({"reprojection_alone": alone_leg(n, H, W, copy)})
        print(json.dumps(rec["legs"][-1]), flush=True)
    rec["legs"].append(c3_leg())
    print(json.dumps(rec["legs"][-1]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
