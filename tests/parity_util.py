"""Shared helpers for the parity tests (CUDA path vs oracle vs reference fixtures)."""
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def mismatch(a, b, mask=None):
    """Number of cells whose fp32 bit patterns differ (NaN-safe, -0/+0 distinguished)."""
    d = bits(a) != bits(b)
    if mask is not None:
        d &= mask
    return int(d.sum())


def max_abs(a, b, mask=None):
    d = np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64))
    if mask is not None:
        d = d[mask]
    return float(d.max()) if d.size else 0.0


def golden_cases():
    if not os.path.isdir(GOLDEN_DIR):
        return []
    return sorted(f[:-4] for f in os.listdir(GOLDEN_DIR) if f.endswith(".npz") and not f.endswith(".volumes.npz"))


def load_golden(name):
    """A case is <name>.npz, plus <name>.volumes.npz (cost, agg) where the volumes are kept apart to keep files small."""
    g = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz")))
    vol = os.path.join(GOLDEN_DIR, name + ".volumes.npz")
    if os.path.exists(vol):
        g.update(np.load(vol))
    return g


def oracle_config_from_array(O, arr):
    from oracle.oracle import CONFIG_FIELDS
    return O.make_config(**{f: int(v) for f, v in zip(CONFIG_FIELDS, arr)})


def run_cuda_all_stages(left_u8, right_u8, cfg_kwargs, variant="auto", dtype="u8", volumes=True, frames_per_launch=0,
                        compat=None, screen=None, info=None):
    """Runs the CUDA path on one frame and returns every intermediate as numpy arrays."""
    import torch
    from stereo_depth_b200 import cuda_depth
    cfg = cuda_depth.StereoMatchingConfiguration(**cfg_kwargs)
    sm = cuda_depth.StereoMatching(cfg, frames_per_launch=frames_per_launch)
    sm.set_variant(variant)
    if compat is not None:
        sm.set_compat(compat)
    if screen is not None:
        sm.set_screen(screen)
    vols = sm.debug_volumes(True) if volumes else None
    if info is not None:
        info["screen_active"] = sm.screen_active
    l = torch.from_numpy(left_u8).cuda()
    r = torch.from_numpy(right_u8).cuda()
    if dtype == "f32":
        l, r = l.float(), r.float()
    out = sm.compute_disparity_map(l.contiguous(), r.contiguous())
    torch.cuda.synchronize()
    res = {"out": out.cpu().numpy().copy()}
    for st in ("gray_l", "gray_r", "pool_l", "pool_r", "wta", "agg3", "refined"):
        res[st] = sm.stage(st).cpu().numpy()
    if vols:
        res["cost"], res["agg"] = vols[0].cpu().numpy(), vols[1].cpu().numpy()
    if info is not None:
        info["evaluated_fraction"] = sm.screen_stats()
    return res


def agg3_from_volume(agg, wta, min_ds=0):
    """The three aggregated values secondary matching reads: A[d*-1], A[d*], A[d*+1], circular in d."""
    Hd, Wd, L = agg.shape
    bd = (wta.astype(np.int64) - min_ds)
    idx = np.stack([(bd - 1) % L, bd % L, (bd + 1) % L], axis=-1)
    return np.take_along_axis(agg, idx, axis=2)


def must_flag_fraction(agg, tile_h=32, tile_w=64):
    """Lower bound of the level screen's `evaluated_fraction` (mbm_screen.cu): whatever its error bound admits, a tile's
    pass mask has to contain the level PAIRS of every pixel's exact arg-max d* and of d*-1, d*+1 (circular in L,
    secondary_matching.cu:28-31).  Returns (sum over tiles of those pairs) / (tiles * ceil(L/2)) -- the same ratio
    sd_screen_stats reports."""
    Hd, Wd, L = agg.shape
    M = (L + 1) // 2
    best = agg.argmax(axis=2)            # first maximum, like the reference's strict '>' scan
    need = np.zeros((Hd, Wd, M), bool)
    ii, jj = np.mgrid[0:Hd, 0:Wd]
    for off in (-1, 0, 1):
        need[ii, jj, ((best + off) % L) // 2] = True
    ty, tx = (Hd + tile_h - 1) // tile_h, (Wd + tile_w - 1) // tile_w
    pad = np.zeros((ty * tile_h, tx * tile_w, M), bool)
    pad[:Hd, :Wd] = need
    tiles = pad.reshape(ty, tile_h, tx, tile_w, M).any(axis=(1, 3))
    return float(tiles.sum()) / float(ty * tx * M)
