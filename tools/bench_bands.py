#!/usr/bin/env python
"""Row-band mode benchmark (BASELINE config C4: one 3840x2160 frame, D=256, K=2, split over the GPUs of a box).

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P tools/bench_bands.py
        [--left-right-check TOL [--background-fill]] [--steps S] [--warmup W] [--repeats R]

Every rank owns one band of the raw frame on its GPU; a step = halo ring exchange (NCCL send/recv over NVLink) +
gray/pool + all-gather of the left gray bands + fused matching + secondary + fill on the band.  Prints one JSON line
(frames/s of the whole frame, max over ranks) and checks the gathered result against a single-GPU run on rank 0.

With --left-right-check (peer-memory transport only) the same run also times the band frame with the left-right check,
and with --background-fill additionally with the check and its background fill: the legs alternate within one run
(R repeats of S steps each, median per leg), each is checked bit for bit against a single-GPU matcher with the same
settings, and the line records the card name and power limit."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from stereo_depth_b200 import cuda_depth  # noqa: E402
from stereo_depth_b200.bands import BandedStereoMatching  # noqa: E402
from stereo_depth_b200.synthetic import make_pair  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--left-right-check", type=float, default=None, help="tolerance in pixels: also time the checked frame")
ap.add_argument("--background-fill", action="store_true", help="also time the checked frame with the background fill")
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--repeats", type=int, default=None, help="alternations of the legs (default 1, 5 with the check)")
args = ap.parse_args()
if args.background_fill and args.left_right_check is None:
    ap.error("--background-fill needs --left-right-check")

H, W, K, D = 2160, 3840, 2, 256
steps, warmup = args.steps, args.warmup
rank = int(os.environ.get("RANK", "0"))
world = int(os.environ.get("WORLD_SIZE", "1"))
local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
left, right, _ = make_pair(H, W, D, seed=1234)
kw = dict(height=H, width=W, downscale_factor=K, min_disparity=0, max_disparity=D - 1)
P2P = os.environ.get("SD_BANDS_P2P", "1") == "1"
if args.left_right_check is not None and not P2P:
    sys.exit("the left-right check on row bands needs the peer-memory transport (SD_BANDS_P2P=1)")
VARIANT = os.environ.get("SD_BANDS_VARIANT")
# legs: (name, tolerance, background fill)
legs = [("off", None, False)]
if args.left_right_check is not None:
    legs.append(("check", args.left_right_check, False))
    if args.background_fill:
        legs.append(("check_fill", args.left_right_check, True))
repeats = args.repeats or (5 if len(legs) > 1 else 1)
sms = {name: BandedStereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), p2p=P2P, variant=VARIANT,
                                  left_right_check=tol, background_fill=fill) for name, tol, fill in legs}
p = sms["off"].plan
lb = torch.from_numpy(left[:, p.x0 * K:p.x1 * K].copy()).cuda()
rb = torch.from_numpy(right[:, p.x0 * K:p.x1 * K].copy()).cuda()
for sm in sms.values():
    for _ in range(warmup):
        sm.compute(lb, rb)
torch.cuda.synchronize()
times = {name: [] for name, _, _ in legs}
for _ in range(repeats):
    for name, _, _ in legs:
        sm = sms[name]
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            sm.compute(lb, rb)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / steps], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        times[name].append(float(ms.item()))
fulls = {name: sms[name].gather(sms[name].compute(lb, rb)) for name, _, _ in legs}


def card():
    """(name, power limit) of this rank's GPU as nvidia-smi reports them (read-only query)."""
    name, limit = torch.cuda.get_device_name(local), None
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        limit = q.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        pass
    return name, limit


if rank == 0:
    l, r = torch.from_numpy(left).cuda(), torch.from_numpy(right).cuda()
    res = {}
    for name, tol, fill in legs:
        plain = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw),
                                          frames_per_launch=1 if tol is None else 2)
        if tol is not None:
            plain.set_left_right_check(tol, background_fill=fill)
        want = plain.compute_disparity_map(l, r)
        torch.cuda.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(5):
            plain.compute_disparity_map(l, r)
        s1.record()
        torch.cuda.synchronize()
        res[name] = {"ms_per_frame": round(float(np.median(times[name])), 4),
                     "ms_runs": [round(t, 4) for t in times[name]],
                     "single_gpu_ms_per_frame": round(s0.elapsed_time(s1) / 5, 4),
                     "bit_identical_to_single_gpu": bool(torch.equal(fulls[name], want))}
    off = res["off"]
    sm = sms["off"]
    line = {"metric": "frames/s (single 3840x2160 frame, D=256, K=2, row bands)", "n_gpus": world,
            "ms_per_frame": off["ms_per_frame"], "value": round(1000.0 / off["ms_per_frame"], 2),
            "single_gpu_ms_per_frame": off["single_gpu_ms_per_frame"],
            "fused_kernel": sm.handle.active_variant + ("+screen" if sm.handle.screen_active else ""),
            "band_rows": p.band_rows, "halo_rows": p.halo_rows,
            "bit_identical_to_single_gpu": off["bit_identical_to_single_gpu"],
            "exchange": ("peer-memory stores of 2x24 raw rows per view + left gray bands read in place over NVLink (flags, no NCCL)"
                         if P2P else "ring send/recv of 2x24 raw rows per view + all-gather of left gray bands (NCCL)")}
    if len(legs) > 1:
        name, limit = card()
        line.update({"legs": res, "left_right_check": args.left_right_check, "repeats": repeats, "steps": steps,
                     "check_over_off": round(res["check"]["ms_per_frame"] / off["ms_per_frame"], 3),
                     "gpu": name, "power_limit": limit})
        if "check_fill" in res:
            line["fill_minus_check_us"] = round(1000.0 * (res["check_fill"]["ms_per_frame"] - res["check"]["ms_per_frame"]), 1)
    print(json.dumps(line), flush=True)
for sm in sms.values():
    sm.close()
if world > 1:
    dist.destroy_process_group()
