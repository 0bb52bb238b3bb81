#!/usr/bin/env python
"""Benchmark of the stereo-matching hot path (BASELINE.json metric: frames/s at 1920x1080, D=128, K=2).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the whole hot path (gray+pool, fused cost+aggregation+WTA, secondary matching,
upscale+fill) over a batch of `--frames` synthetic random-dot frames per GPU.  Frames are sharded over
GPUs (one process per GPU, no collective on the data path) => weak scaling.  Prints ONE JSON line.
The timed loops run exactly K steps in all, split into `--repeats` windows.

--dump-outputs DIR writes the disparity maps of the last timed step's distinct frames (the first `--distinct`) as
DIR/disparity.npy (float32; with N GPUs, disparity_rank<r>.npy per rank): all of their rows when they fit in 48 MiB,
else a fixed, seeded sample of whole image rows (of the [n*H, W] rows, in ascending order).  Inputs are seeded,
so two builds can be compared output for output.

  value      frames/s, inputs (uint8 CHW, what a camera delivers) already resident in HBM, CUDA events
  e2e        frames/s through CudaStereoMatchingBackend.process_batch with pinned HOST tensors: every step
             copies its inputs host->device and its disparity maps device->host (pipelined by the library)
  roofline   dominant kernel (fused cost+aggregation+WTA): algorithmic fp32 lane-ops / measured launch time
             vs the measured fp32-add peak of the CUDA cores (not HBM, not tensor cores: SURVEY 8-d)
  cpu_baseline  the CPU oracle (order-faithful port of the reference kernels) on this box's host cores
  reference_cuda  the reference's own CUDA kernels (oracle/_ref build) on the same B200, same run

--impl reference times the reference itself: its CUDA kernels when oracle/_ref/cuda_depth.so loads (the
reference has no CPU implementation), else the oracle port on the host cores.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[2]: the configuration the metric is quoted on
    "C3": dict(H=1080, W=1920, K=2, D=128, name="1920x1080 synthetic random-dot video, D=128, K=2"),
    "C5": dict(H=720, W=1280, K=2, D=128, name="1280x720 synthetic random-dot video, D=128, K=2"),
    "C1": dict(H=480, W=640, K=2, D=64, name="640x480 synthetic random-dot pair, D=64, K=2"),
}
FADD_PEAK_TOPS = 37.0  # measured on this pool's B200: tools/microbench/fadd_bench (profiles/r01_fadd_microbench.txt)
SMI_QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=50)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--frames", type=int, default=64, help="frames per step per GPU")
    p.add_argument("--workload", default="C3", choices=sorted(WORKLOADS))
    p.add_argument("--frames-per-launch", type=int, default=0, help="0 = library default (fills whole waves of the fused kernel)")
    p.add_argument("--distinct", type=int, default=8, help="distinct synthetic frames generated (tiled to --frames)")
    p.add_argument("--no-extras", action="store_true", help="skip cpu_baseline / reference_cuda / natural / multi-GPU legs")
    p.add_argument("--repeats", type=int, default=5,
                   help="the K timed steps are split into this many windows; value = median window")
    p.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's disparity maps here (.npy)")
    args = p.parse_args()
    if args.steps < 1 or args.repeats < 1:
        p.error("--steps and --repeats must be positive")
    if args.dump_outputs and args.impl != "ours":
        p.error("--dump-outputs applies to --impl ours")
    return args


def windows(steps, repeats):
    """Sizes of the timed windows: `steps` steps in all, over at most `repeats` windows."""
    n = min(steps, repeats)
    return [steps // n + (i < steps % n) for i in range(n)]


DUMP_BYTES = 48 << 20   # per dump, over all ranks


def dump_outputs(out, directory, rank, world):
    """Writes the [F,H,W] float32 disparity maps `out` (a CUDA tensor) as rows of [F*H, W]: all of them, or a
    seeded sample of whole rows (same rows in every run with the same arguments) when they exceed the budget."""
    import numpy as np
    import torch
    rows = out.reshape(-1, out.shape[-1])
    n = min(rows.shape[0], DUMP_BYTES // world // (rows.shape[1] * 4))
    if n < rows.shape[0]:
        pick = np.sort(np.random.default_rng(0).choice(rows.shape[0], size=n, replace=False))
        rows = rows.index_select(0, torch.from_numpy(pick).to(rows.device))
    os.makedirs(directory, exist_ok=True)
    name = "disparity.npy" if world == 1 else f"disparity_rank{rank}.npy"
    np.save(os.path.join(directory, name), rows.cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.path = gpu_index, None, f"/tmp/bench_clocks_{os.getpid()}.csv"

    def start(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={SMI_QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.f.close()
        sm, mx, power, reasons = [], [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for line in open(self.path):
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2])); power.append(float(parts[3]))
            except ValueError:
                continue
            for n, v in zip(names, parts[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        try:
            os.remove(self.path)
        except OSError:
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # "under load": samples drawing clearly more than idle power
        load = [c for c, p in zip(sm, power) if p >= 0.6 * max(power)] or sm
        return {"sm_mhz": statistics.median(load), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power)}


def pin_to_gpu_numa_node(local):
    """Run this process (and first-touch its pinned buffers) on the CPUs closest to its GPU: with one process per
    GPU the host<->device copies of the e2e leg otherwise cross the socket interconnect."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        n = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n)
        cpus = [64 * i + b for i, w in enumerate(mask) for b in range(64) if (w >> b) & 1]
        if cpus:
            os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:  # noqa: BLE001
        return 0


def dist_setup(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    pin_to_gpu_numa_node(local)   # also with one GPU: the pinned buffers of the e2e leg should be first-touched near it
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(local)
    return rank, world, local


def barrier(world):
    import torch
    import torch.distributed as dist
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, world):
    import torch
    import torch.distributed as dist
    if world == 1:
        return x
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def make_inputs(wl, frames, distinct, rank):
    import numpy as np
    import torch
    from stereo_depth_b200.synthetic import make_batch
    distinct = max(1, min(distinct, frames))
    l, r = make_batch(distinct, wl["H"], wl["W"], wl["D"], seed=1234, first_frame=rank * frames)
    reps = (frames + distinct - 1) // distinct
    l = np.concatenate([l] * reps)[:frames]
    r = np.concatenate([r] * reps)[:frames]
    return torch.from_numpy(l), torch.from_numpy(r)


def workload_config(args, wl, world):
    """The workload description both arms print as `config` (identical keys and values: the driver compares them).
    Everything implementation-specific goes to `impl_config`."""
    F = args.frames
    in_bytes = 2 * F * 3 * wl["H"] * wl["W"]
    return {"workload": f"{args.workload}: {wl['name']}, {F} frames per GPU per step, frame-sharded",
            "H": wl["H"], "W": wl["W"], "D": wl["D"], "K": wl["K"], "frames_per_gpu_per_step": F,
            "distinct_frames": max(1, min(args.distinct, F)),
            "input": "uint8 CHW frames as a camera delivers them (an arm that needs float32 converts with .float(), as "
                     "cuda_stereo_matching_backend.py:14-15 does)",
            "l2": f"inputs {in_bytes / 1e6:.0f} MB per step > 126 MB L2 (no flush needed)",
            "parallelism": f"frame-batch x{world}, no collective"}


def cpu_baseline_leg(wl):
    """Bounded sample: one frame of the workload through the oracle on the host cores."""
    import numpy as np
    from oracle import oracle as O
    from stereo_depth_b200.synthetic import make_pair
    l, r, _ = make_pair(wl["H"], wl["W"], wl["D"], seed=1234)
    cfg = O.make_config(height=wl["H"], width=wl["W"], downscale_factor=wl["K"], min_disparity=0,
                        max_disparity=wl["D"] - 1)
    lf, rf = l.astype(np.float32), r.astype(np.float32)
    best = 1e30
    for _ in range(2):
        t = time.perf_counter()
        O.run(cfg, lf, rf, want=("out",))
        best = min(best, time.perf_counter() - t)
    return {"value": 1.0 / best, "unit": "frames/s", "cores": O.num_threads(), "kind": "port",
            "sample": f"1 frame of {wl['name']} (best of 2), oracle/stereo_oracle.c with OpenMP over all host cores"}


SCREEN_OPS_PER_CELL = 45.0   # lane-ops the level screen executes per (pixel, level) cell (header of csrc/mbm_screen.cu)


def copy_ceiling_leg(lh, rh, out_h, steps, world, chunk=8):
    """The e2e leg's byte pattern with bare cudaMemcpyAsync and NO kernels: per step, every chunk of `chunk` frames
    is copied host->device (both views) on one stream while a chunk of disparity maps goes device->host on another,
    all ranks concurrently.  This is what the box's PCIe / host-memory system can carry at this duplex mix."""
    import torch
    F = lh.shape[0]
    dl = torch.empty((chunk,) + tuple(lh.shape[1:]), dtype=lh.dtype, device="cuda")
    dr = torch.empty_like(dl)
    do = torch.zeros((chunk,) + tuple(out_h.shape[1:]), dtype=out_h.dtype, device="cuda")
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()

    def step():
        for f0 in range(0, F, chunk):
            n = min(chunk, F - f0)
            with torch.cuda.stream(s_in):
                dl[:n].copy_(lh[f0:f0 + n], non_blocking=True)
                dr[:n].copy_(rh[f0:f0 + n], non_blocking=True)
            with torch.cuda.stream(s_out):
                out_h[f0:f0 + n].copy_(do[:n], non_blocking=True)

    step()
    barrier(world)
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    torch.cuda.synchronize()
    dt = max_over_ranks(time.perf_counter() - t0, world)
    barrier(world)
    return world * F * steps / dt


def natural_leg(args, wl):
    """The reference's own natural stereo pair (src/python/data/im0.png, im1.png via data/_ref/natural_pair.npz)
    through the same path, next to the random-dot headline: the level screen's gain is scene dependent."""
    import numpy as np
    import torch
    from stereo_depth_b200 import cuda_depth
    from stereo_depth_b200.synthetic import load_natural_pair
    pair = load_natural_pair()
    if pair is None:
        return {"unavailable": "data/_ref/natural_pair.npz not present (oracle/make_natural.py needs /root/reference)"}
    left, right, vmin, vmax = pair
    H, W = left.shape[1:]
    F, distinct = 32, 16
    # 16 distinct frames (the pair rolled horizontally by 8 columns per frame: 199 MB of inputs > L2), tiled to 32
    ls = np.stack([np.roll(left, 8 * i, axis=2) for i in range(distinct)] * (F // distinct))
    rs = np.stack([np.roll(right, 8 * i, axis=2) for i in range(distinct)] * (F // distinct))
    ld, rd = torch.from_numpy(ls).cuda(), torch.from_numpy(rs).cuda()
    out = torch.empty((F, H, W), dtype=torch.float32, device="cuda")
    res = {"frames_per_step": F, "distinct_frames": distinct,
           "data": "the reference's shipped Middlebury-format pair, rolled by 8 columns per frame"}
    for name, mn, mx in (("headline_range_0_127", 0, wl["D"] - 1), ("reference_default_75_262", vmin, vmax)):
        sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(
            height=H, width=W, downscale_factor=2, min_disparity=mn, max_disparity=mx))
        one = {"min_disparity": mn, "max_disparity": mx, "levels": sm.dims[2], "screen_active": bool(sm.screen_active)}
        for screen in ((True, False) if sm.screen_active else (None,)):
            if screen is not None:
                sm.set_screen(screen)
            for _ in range(3):
                sm.compute_disparity_batch(ld, rd, out=out)
            sm.screen_stats(reset=True)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                sm.compute_disparity_batch(ld, rd, out=out)
            e1.record()
            torch.cuda.synchronize()
            fps = F * 5 / (e0.elapsed_time(e1) * 1e-3)
            if screen is None or screen:
                one.update(fps=round(fps, 1), ms_per_frame=round(1e3 / fps, 4),
                           evaluated_fraction=round(sm.screen_stats(reset=True), 4), screen_paused=int(sm.screen_paused))
            else:
                one.update(fps_screen_off=round(fps, 1), ms_per_frame_screen_off=round(1e3 / fps, 4))
        res[name] = one
        del sm
    return res


def c5_leg(world, rank, steps=5):
    """BASELINE configs[4]: 256 frames of 1280x720 (D=128, K=2), full pipeline, frame-sharded over the GPUs."""
    import torch
    from stereo_depth_b200 import cuda_depth
    from stereo_depth_b200.bands import shard_frames
    wl = WORKLOADS["C5"]
    total = 256
    a, b = shard_frames(total, world, rank)
    F = b - a
    ns = argparse.Namespace(distinct=8)
    lh, rh = make_inputs(wl, F, ns.distinct, rank)
    ld, rd = lh.cuda(), rh.cuda()
    sm = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(
        height=wl["H"], width=wl["W"], downscale_factor=wl["K"], min_disparity=0, max_disparity=wl["D"] - 1))
    out = torch.empty((F, wl["H"], wl["W"]), dtype=torch.float32, device="cuda")
    for _ in range(3):
        sm.compute_disparity_batch(ld, rd, out=out)
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        sm.compute_disparity_batch(ld, rd, out=out)
    e1.record()
    barrier(world)
    ms = max_over_ranks(e0.elapsed_time(e1), world)
    return {"fps": round(total * steps / (ms * 1e-3), 1), "frames_total": total, "frames_per_gpu": F, "steps": steps,
            "workload": wl["name"], "timer": "CUDA events, max over ranks"}


def bands_c4_leg(world, rank, steps=20):
    """BASELINE configs[3]: ONE 3840x2160 frame (D=256, K=2) split into row bands over the GPUs, halos and left-gray rows
    exchanged through peer memory over NVLink (sd_band_p2p_*).  Checked bit for bit against the single-GPU result."""
    import torch
    from stereo_depth_b200 import cuda_depth
    from stereo_depth_b200.bands import BandedStereoMatching
    from stereo_depth_b200.synthetic import make_pair
    H, W, K, D = 2160, 3840, 2, 256
    left, right, _ = make_pair(H, W, D, seed=1234)
    kw = dict(height=H, width=W, downscale_factor=K, min_disparity=0, max_disparity=D - 1)
    sm = BandedStereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), p2p=True)
    p = sm.plan
    lb = torch.from_numpy(left[:, p.x0 * K:p.x1 * K].copy()).cuda()
    rb = torch.from_numpy(right[:, p.x0 * K:p.x1 * K].copy()).cuda()
    for _ in range(3):
        out = sm.compute(lb, rb)
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = sm.compute(lb, rb)
    e1.record()
    barrier(world)
    ms = max_over_ranks(e0.elapsed_time(e1), world) / steps
    full = sm.gather(out)
    res = None
    if rank == 0:
        plain = cuda_depth.StereoMatching(cuda_depth.StereoMatchingConfiguration(**kw), frames_per_launch=1)
        l, r = torch.from_numpy(left).cuda(), torch.from_numpy(right).cuda()
        want = plain.compute_disparity_map(l, r)
        torch.cuda.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(5):
            plain.compute_disparity_map(l, r)
        s1.record()
        torch.cuda.synchronize()
        single = s0.elapsed_time(s1) / 5
        res = {"ms_per_frame": round(ms, 4), "single_gpu_ms": round(single, 4), "speedup": round(single / ms, 3),
               "efficiency": round(single / ms / world, 3), "bit_identical": bool(torch.equal(full, want)),
               "transport": "peer-memory stores + system-scope flags over NVLink (sd_band_p2p_*), no NCCL on the data path",
               "band_rows": p.band_rows, "halo_rows": p.halo_rows, "level_split": getattr(sm.handle, "level_split", 1),
               "fused_kernel": sm.handle.active_variant + ("+screen" if sm.handle.screen_active else "")}
    sm.close()
    barrier(world)
    return res


def run_ours(args):
    import torch
    from stereo_depth_b200 import backend, cuda_depth
    rank, world, local = dist_setup(args)
    wl = WORKLOADS[args.workload]
    H, W, K, D = wl["H"], wl["W"], wl["K"], wl["D"]
    F = args.frames
    cfg = cuda_depth.StereoMatchingConfiguration(height=H, width=W, downscale_factor=K, min_disparity=0,
                                                 max_disparity=D - 1)
    be = backend.CudaStereoMatchingBackend(cfg, frames_per_launch=args.frames_per_launch)
    sm = be.native
    Hd, Wd, L = sm.dims
    lh, rh = make_inputs(wl, F, args.distinct, rank)
    lh, rh = lh.pin_memory(), rh.pin_memory()
    ld, rd = lh.cuda(), rh.cuda()
    out_d = torch.empty((F, H, W), dtype=torch.float32, device="cuda")
    out_h = torch.empty((F, H, W), dtype=torch.float32).pin_memory()
    in_bytes = 2 * F * 3 * H * W
    out_bytes = F * H * W * 4

    # ---- device-resident throughput: exactly K steps in REPEATS windows, each bracketed by barrier + synchronize;
    #      the reported value is the median window (max over ranks per window) -------------------------------------
    for _ in range(max(args.warmup, 3)):
        sm.compute_disparity_batch(ld, rd, out=out_d)
    sampler = ClockSampler(local)
    barrier(world)
    if rank == 0:
        sampler.start()
    win = windows(args.steps, args.repeats)
    rep_ms = []
    for n in win:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(world)
        e0.record()
        for _ in range(n):
            sm.compute_disparity_batch(ld, rd, out=out_d)
        e1.record()
        barrier(world)
        rep_ms.append(max_over_ranks(e0.elapsed_time(e1), world))
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # frame i repeats frame i % distinct: sample the distinct ones
        dump_outputs(out_d[:max(1, min(args.distinct, F))], args.dump_outputs, rank, world)
    rep_fps = sorted(world * F * n / (t * 1e-3) for n, t in zip(win, rep_ms))
    value = statistics.median(rep_fps)
    ms_per_step = world * F / value * 1e3   # at the median window's rate

    # ---- end to end from pinned host memory through the plugin API (K steps in up to 3 windows, median window) -------
    for _ in range(2):
        be.process_batch(lh, rh, out=out_h)
    e2e_win = windows(args.steps, 3)
    e2e_runs = []
    for n in e2e_win:
        barrier(world)
        t0 = time.perf_counter()
        for _ in range(n):
            be.process_batch(lh, rh, out=out_h)   # synchronous: returns when out_h is complete
        torch.cuda.synchronize()
        e2e_runs.append(world * F * n / max_over_ranks(time.perf_counter() - t0, world))
    barrier(world)
    e2e = statistics.median(e2e_runs)
    same = bool(torch.equal(out_h[:2], out_d[:2].cpu()))
    keep = out_h[:2].clone()
    ceiling = copy_ceiling_leg(lh, rh, out_h, max(2, args.steps // 2), world)
    out_h[:2].copy_(keep)

    # ---- single-frame latency through the reference-shaped call (one frame per process() call) --------
    one_l, one_r = lh[0], rh[0]
    for _ in range(3):
        be.process(one_l, one_r)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(20):
        o = be.process(one_l, one_r)
        o.cpu()
    latency_ms = (time.perf_counter() - t0) / 20 * 1e3

    # ---- per-kernel device times (CUDA events inside the library, on the launching stream) ----------
    screened = sm.screen_active
    sm.screen_stats(reset=True)
    sm.profile(True)
    for _ in range(2):
        sm.compute_disparity_batch(ld, rd, out=out_d)
    prof = sm.profile_read_detail()
    sm.profile(False)
    evaluated_fraction = sm.screen_stats(reset=True)
    b_n = prof["cost_agg_wta"][1]
    # "kernel B" = everything between the pooled images and the WTA records: plane padding, level screen, exact kernel
    b_ms = prof["pad_planes"][0] + prof["level_screen"][0] + prof["cost_agg_wta"][0]
    frames_per_launch = sm.frames_per_launch
    # SURVEY 8-d: 237 lane-ops per cell; the 2 profiled passes processed 2*F frames in b_n launches (the last chunk
    # of a pass may be shorter, so work per launch is the average)
    ops_per_launch = 237.0 * Hd * Wd * L * (2.0 * F / b_n)
    achieved = ops_per_launch / (b_ms / b_n * 1e-3) / 1e12
    # what the hardware actually executed: the screen's ~45 lane-ops on every cell + 237 on the flagged fraction
    exec_ops_per_launch = ((SCREEN_OPS_PER_CELL + 237.0 * evaluated_fraction) if screened else 237.0) * Hd * Wd * L * (2.0 * F / b_n)
    hw_achieved = exec_ops_per_launch / (b_ms / b_n * 1e-3) / 1e12
    kernel_ms = {k: round(v[0] / max(v[1], 1), 4) for k, v in prof.items()}
    total_prof = sum(v[0] for v in prof.values())
    # hardware efficiency of the exact kernel itself: the same launches with the screen switched off (all levels)
    exact_all = None
    if screened:
        sm.set_screen(False)
        sm.compute_disparity_batch(ld, rd, out=out_d)
        sm.profile(True)
        for _ in range(2):
            sm.compute_disparity_batch(ld, rd, out=out_d)
        p2 = sm.profile_read_detail()
        sm.profile(False)
        sm.set_screen(True)
        x_ms, x_n = p2["cost_agg_wta"]
        x_ach = 237.0 * Hd * Wd * L * (2.0 * F / x_n) / (x_ms / x_n * 1e-3) / 1e12
        exact_all = {"achieved": round(x_ach, 3), "frac": round(x_ach / FADD_PEAK_TOPS, 4), "launch_ms": round(x_ms / x_n, 4),
                     "how": "mbm_wta_fast_kernel alone with the screen switched off (every level evaluated), profiled after the timed region"}
    traffic, screen_ncu = None, None
    tpath = os.path.join(ROOT, "profiles", "kernelB_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            per_frame = tj.get(args.workload + ("_screened" if screened else "") + "_per_frame")
            traffic = None if per_frame is None else int(per_frame * 2.0 * F / b_n)
            screen_ncu = tj.get("screen_kernel_ncu") if args.workload == "C3" else None
        except (OSError, ValueError):
            traffic = None

    # ---- BASELINE configs[3] and [4]: every rank takes part --------------------------------------------------------
    multi = {}
    if not args.no_extras:
        del ld, rd, out_d, lh, rh, out_h
        torch.cuda.empty_cache()
        try:
            multi["c5"] = c5_leg(world, rank)
        except Exception as e:  # noqa: BLE001
            multi["c5"] = {"error": str(e)[:300]}
        if world > 1:
            try:
                multi["bands_c4"] = bands_c4_leg(world, rank)
            except Exception as e:  # noqa: BLE001
                multi["bands_c4"] = {"error": str(e)[:300]}
    if rank != 0:
        return
    line = {
        "metric": "frames/s", "value": round(value, 2), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms_per_step, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, wl, world),
        "impl_config": {"frames_per_launch": frames_per_launch, "fused_kernel_variant": sm.active_variant,
                        "level_screen": screened},
        "repeats": {"n": len(win), "steps_each": win, "value": "median", "fps_min": round(rep_fps[0], 1),
                    "fps_median": round(value, 1), "fps_max": round(rep_fps[-1], 1),
                    "timed_seconds_total": round(sum(rep_ms) * 1e-3, 3)},
        "e2e": {"value": round(e2e, 2), "unit": "frames/s", "h2d_bytes_per_step": in_bytes,
                "d2h_bytes_per_step": out_bytes, "api": "CudaStereoMatchingBackend.process_batch (sd_compute_host)",
                "timer": "wall clock around the synchronous calls, max over ranks, median of up to 3 windows of the K steps",
                "fps_min": round(min(e2e_runs), 1), "fps_max": round(max(e2e_runs), 1),
                "matches_device_path": same,
                "single_frame_latency_ms": round(latency_ms, 3),
                "copy_ceiling_fps": round(ceiling, 1), "frac_of_copy_ceiling": round(e2e / ceiling, 4),
                "copy_ceiling_how": "the same H2D + D2H bytes per step as bare cudaMemcpyAsync in 8-frame chunks on two "
                                    "streams, no kernels, all ranks concurrently (wall clock, max over ranks)"},
        "gpu_launches": sm.launches_per_call(F) * args.steps * world,
        "clocks": clocks,
        "roofline": {"bound": "fp32_alu",
                     "kernel": ("mbm_screen_kernel + mbm_wta_fast_kernel (certified level screen + exact cost/aggregation/WTA of the flagged level pairs)"
                                if screened else ("mbm_wta_ws_kernel" if sm.active_variant == "ws" else "mbm_wta_fast_kernel") +
                                " (fused cost + aggregation + WTA)"),
                     "achieved": round(achieved, 3), "peak": FADD_PEAK_TOPS, "unit": "TFLOP/s",
                     "frac": round(achieved / FADD_PEAK_TOPS, 4), "traffic": traffic,
                     "traffic_source": "static: one ncu --set full capture (profiles/kernelB_traffic.json), scaled to this launch size; not measured in this run",
                     "hw_achieved": round(hw_achieved, 3), "hw_frac": round(hw_achieved / FADD_PEAK_TOPS, 4),
                     "hw_frac_how": "EXECUTED lane-ops (level screen: 45 per cell on every cell + exact kernel: 237 per cell on the "
                                    "evaluated fraction of the level pairs) / the same time / the same peak; `frac` counts the "
                                    "ALGORITHMIC 237 per cell",
                     "peak_source": "measured fp32 add peak of the CUDA cores (128 lane-adds/clk/SM x 148 SM x 1.955 GHz, "
                                    "tools/microbench/fadd_bench; MEASURED_PEAKS.json has no ALU figure); 1 lane-op = 1 'FLOP'",
                     "algorithmic_ops_per_launch": ops_per_launch, "frames_per_launch_avg": round(2.0 * F / b_n, 3),
                     "launch_ms": round(b_ms / b_n, 4),
                     "share_of_step": round(b_ms / total_prof, 4), "kernel_ms_per_launch": kernel_ms},
    }
    if screened:
        line["roofline"]["certified_screen"] = {
            "evaluated_fraction": round(evaluated_fraction, 4),
            "note": "achieved/frac count the ALGORITHMIC 237 lane-ops per cell (SURVEY 8-d) over the time of padding + screen + "
                    "exact kernel; the screen proves most level pairs cannot hold the arg-max, so fewer are executed and frac may "
                    "exceed the hardware fraction (and 1).  Results are bit-identical with the screen off.",
            "exact_kernel_all_levels": exact_all,
            # the screen kernel itself is bound by the shared-memory crossbar, not by the adders: its ncu figures
            # (one --set full capture, profiles/r01_ncu_screen_summary.txt), not measured live
            "screen_kernel": None if screen_ncu is None else dict(screen_ncu, bound="shared-memory crossbar (128 B/clk/SM)",
                                                                 launch_ms=kernel_ms.get("level_screen"))}
    extra = {}
    if world == 1 and not args.no_extras:
        try:
            line["cpu_baseline"] = cpu_baseline_leg(wl)
        except Exception as e:  # noqa: BLE001
            line["cpu_baseline"] = {"error": str(e)[:200]}
        line["reference_cuda"] = reference_subprocess(args, frames=4, steps=3)
        try:
            extra["natural"] = natural_leg(args, wl)
        except Exception as e:  # noqa: BLE001
            extra["natural"] = {"error": str(e)[:300]}
    extra.update(multi or {})
    line["extra"] = extra
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# reference arm
# ------------------------------------------------------------------------------------------------

def load_reference_module():
    import importlib.util
    import torch  # noqa: F401  (libtorch symbols must be loaded first)
    path = os.path.join(ROOT, "oracle", "_ref", "cuda_depth.so")
    if not os.path.exists(path):
        return None
    spec = importlib.util.spec_from_file_location("cuda_depth", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def run_reference_gpu(args, wl):
    """The reference's own CUDA kernels (unmodified algorithm; sm_100 build of a patched copy, see
    oracle/build_ref.py) through its public class cuda_depth.StereoMatching."""
    import torch
    mod = load_reference_module()
    if mod is None:
        return None
    H, W, K, D = wl["H"], wl["W"], wl["K"], wl["D"]
    F = args.frames
    torch.cuda.set_device(0)
    lh, rh = make_inputs(wl, F, min(args.distinct, F), 0)
    lh, rh = lh.pin_memory(), rh.pin_memory()
    # one large cached segment so the reference's out-of-bounds reads stay inside mapped memory (SURVEY 8-c)
    # and keep a pre-guard at its start: secondary_matching reads up to 5 rows BEFORE left_grayscaled
    guard = torch.empty(2 << 30, dtype=torch.uint8, device="cuda")
    del guard
    pre_guard = torch.zeros(64 << 20, dtype=torch.uint8, device="cuda")  # noqa: F841  (carved from the cached 2 GiB block)
    sm = mod.StereoMatching(mod.StereoMatchingConfiguration(height=H, width=W, downscale_factor=K, min_disparity=0,
                                                            max_disparity=D - 1))
    nd = max(1, min(args.distinct, F))   # frames repeat with this period: keep one float32 device copy of each
    lf = [lh[i].cuda().float().contiguous() for i in range(nd)]
    rf = [rh[i].cuda().float().contiguous() for i in range(nd)]

    def step():
        for i in range(F):
            sm.compute_disparity_map(lf[i % nd], rf[i % nd])

    for _ in range(max(args.warmup, 1)):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    value = F * args.steps / (ms * 1e-3)
    # end to end as CudaStereoMatchingBackend.process does it (cuda_stereo_matching_backend.py:13-17) + D2H
    out_h = torch.empty((H, W), dtype=torch.float32).pin_memory()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        for i in range(F):
            o = sm.compute_disparity_map(lh[i].cuda().float().contiguous(), rh[i].cuda().float().contiguous())
            out_h.copy_(o)
    torch.cuda.synchronize()
    e2e = F * args.steps / (time.perf_counter() - t0)
    return {"value": value, "ms_per_step": ms / args.steps, "e2e": e2e, "frames": F,
            "h2d": 2 * F * 3 * H * W, "d2h": F * H * W * 4}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # rank 0 alone runs the reference arm
    wl = WORKLOADS[args.workload]
    base = {"metric": "frames/s", "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "impl": "reference",
            "config": workload_config(args, wl, int(os.environ.get("WORLD_SIZE", args.gpus)))}
    res = None
    try:
        import torch
        if torch.cuda.is_available():
            res = run_reference_gpu(args, wl)
    except Exception as e:  # noqa: BLE001
        base["reference_gpu_error"] = str(e)[:300]
    if res is not None:
        base.update({"value": round(res["value"], 2), "ms_per_step": round(res["ms_per_step"], 3),
                     "impl_config": {"device": "the reference's own CUDA kernels on 1 B200 (it has no CPU or multi-GPU path)",
                                     "value_input": "float32 CHW on device (what compute_disparity_map accepts)",
                                     "e2e_input": "uint8 CHW pinned host frames -> .cuda().float().contiguous()"},
                     "cpu_baseline": {"value": round(res["value"], 2), "unit": "frames/s", "cores": 0, "kind": "reference",
                                      "sample": f"{res['frames']} frames per step, reference CUDA kernels (oracle/_ref/cuda_depth.so) "
                                                "on one B200; cores=0: runs on the GPU, not on host cores"},
                     "e2e": {"value": round(res["e2e"], 2), "unit": "frames/s", "h2d_bytes_per_step": res["h2d"],
                             "d2h_bytes_per_step": res["d2h"],
                             "api": "uint8 host -> .cuda().float().contiguous() -> compute_disparity_map -> host"}})
    else:
        cb = cpu_baseline_leg(wl)
        cb["kind"] = "port"
        base.update({"value": round(cb["value"], 4), "ms_per_step": round(1000.0 / cb["value"], 1), "cpu_baseline": cb,
                     "e2e": {"value": round(cb["value"], 4), "unit": "frames/s", "h2d_bytes_per_step": 0,
                             "d2h_bytes_per_step": 0}})
    print(json.dumps(base), flush=True)


def reference_subprocess(args, frames, steps):
    """Times the reference CUDA kernels in a child process (its out-of-bounds reads must not be able to
    take this process's CUDA context down) and returns the parsed result."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", args.workload,
           "--frames", str(frames), "--steps", str(steps), "--warmup", "1"]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env).stdout.strip().splitlines()
        j = json.loads(out[-1])
        return {"value": j.get("value"), "unit": "frames/s", "e2e": j.get("e2e", {}).get("value"),
                "kind": j.get("cpu_baseline", {}).get("kind"), "sample": j.get("cpu_baseline", {}).get("sample")}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)[:200]}


def main():
    args = parse_args()
    if args.gpus > 1 and "RANK" not in os.environ:
        import socket
        s = socket.socket()
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
        s.close()
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
