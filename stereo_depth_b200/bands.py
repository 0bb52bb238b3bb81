"""Multi-GPU partitioning of the stereo-matching hot path (no counterpart in the reference, which is single-GPU).

Two modes (SURVEY.md section 8-e):

* frame-batch sharding (video): frames are independent -> `shard_frames` gives each rank a contiguous chunk;
  no collective on the data path.

* row bands (one very large frame, BASELINE config C4): every rank owns a contiguous band of pooled rows and
  the matching raw image rows.  One exchange step moves the halos over NVLink (NCCL send/recv in a ring -- the
  ring is closed because the reference's row padding is circular, device_functions.cuh:13-14):
      top halo    12 pooled rows (11 for cost+aggregation of the row above the band, whose refined disparity the
                  vertical fill reads, upscale_disparity_vertical_fill.cu:34)
      bottom halo 12 pooled rows (10 aggregation + 1 cost + the next row's column 0 read by the horizontal fill,
                  horizontal_disparity_fill.cu:27)
  Each rank then runs the unchanged kernels on its local window [top halo | band | bottom halo].  Only the fill
  kernel needs global knowledge (the reference's `x == 0` rule, the `(k+1)*x` colour row and the last-row rule),
  which it gets from `sd_set_band` plus an all-gather of the left gray bands (the second exchange step).
  Band results are bit-identical to the single-GPU result (tests/test_multi_gpu.py).

  `BandedStereoMatching(..., p2p=True)` runs the same two exchange steps over PEER MEMORY instead of NCCL: the library
  stores the halo rows straight into the neighbours' HBM while it copies the band into its own window, publishes its
  left gray band for the other ranks' fill kernels to read in place, and synchronises with system-scope flags
  (stereo_depth_b200/csrc/band_p2p.cu).  torch.distributed is then only used once, to exchange the CUDA IPC handles.

  Over peer memory the left-right check (and its background fill) runs on the bands too, bit-identical to a
  single-GPU `StereoMatching.set_left_right_check` on the whole frame: the mirrored pair is read from the same raw
  window, the mirrored frame's left gray band is published next to the forward one, and with the fill a third exchange
  step shares every band's first / last row that kept a pixel (DESIGN.md section 8).
"""
import math
from dataclasses import dataclass

import torch
import torch.distributed as dist

HALO_POOLED = 12   # the halo of the reference's default radii (large_mbm_radius 10, cost radius 1, sad radius 5, K >= 1)


def halo_pooled_rows(cfg):
    """Pooled halo rows a band needs above and below for configuration `cfg` (an sd_config / SdConfig):
    aggregation (large_mbm_radius) + cost (ncc_patch_radius) + 1 row (top: the row above the band, whose refined
    disparity the vertical fill reads; bottom: the next row's column 0 read by the horizontal fill), and enough
    full-resolution rows for the secondary matching window of those rows: halo * K >= K + sad_patch_radius."""
    K = cfg.downscale_factor
    return max(cfg.large_mbm_radius + cfg.ncc_patch_radius + 1, -(-(K + cfg.sad_patch_radius) // K))


def shard_frames(n_frames, world, rank):
    """Contiguous [start, stop) chunk of rank `rank`; sizes differ by at most one frame."""
    base, extra = divmod(n_frames, world)
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


@dataclass(frozen=True)
class BandPlan:
    """Host-side geometry of one rank's band (all row counts in FULL-RESOLUTION rows unless noted)."""
    H: int
    W: int
    K: int
    world: int
    rank: int
    x0: int          # first pooled row of the band
    x1: int          # one past the last pooled row
    halo: int        # halo in pooled rows (top and bottom)

    @staticmethod
    def make(H, W, K, world, rank, halo=HALO_POOLED):
        if H % K != 0:
            raise ValueError("row-band mode needs height divisible by downscale_factor")
        Hd = H // K
        x0, x1 = shard_frames(Hd, world, rank)
        if world > 1 and min(shard_frames(Hd, world, r)[1] - shard_frames(Hd, world, r)[0] for r in range(world)) < halo:
            raise ValueError("bands must be at least as tall as the halo (halos come from the ring neighbours only)")
        return BandPlan(H, W, K, world, rank, x0, x1, halo)

    @property
    def band_rows(self):
        return (self.x1 - self.x0) * self.K

    @property
    def halo_rows(self):
        return self.halo * self.K

    @property
    def local_rows(self):
        return self.band_rows + 2 * self.halo_rows

    @property
    def pooled_row_offset(self):
        """Global pooled row of local pooled row 0 (negative for the first band: circular)."""
        return self.x0 - self.halo

    def global_rows_of_local_window(self):
        r0 = self.K * (self.x0 - self.halo)
        return [(r0 + i) % self.H for i in range(self.local_rows)]


def exchange_halos(band, halo_rows, group=None):
    """band: [C, rows, W] tensor owned by this rank.  Returns [C, halo + rows + halo, W] with the top halo
    received from the previous rank's last rows and the bottom halo from the next rank's first rows (ring).
    NCCL send/recv (NVLink) on CUDA tensors, gloo on CPU tensors (tests)."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    C, rows, W = band.shape
    out = torch.empty((C, rows + 2 * halo_rows, W), dtype=band.dtype, device=band.device)
    out[:, halo_rows:halo_rows + rows] = band
    if world == 1:
        out[:, :halo_rows] = band[:, rows - halo_rows:]
        out[:, halo_rows + rows:] = band[:, :halo_rows]
        return out
    prev, nxt = (rank - 1) % world, (rank + 1) % world
    send_top = band[:, :halo_rows].contiguous()            # becomes prev's bottom halo
    send_bot = band[:, rows - halo_rows:].contiguous()     # becomes next's top halo
    recv_top = torch.empty_like(send_top)
    recv_bot = torch.empty_like(send_bot)
    # Order matters when prev == next (world 2): the peer's first message (its top rows, sent to ITS prev) is our
    # BOTTOM halo, so the first receive posted for that peer must be the bottom one.
    ops = [dist.P2POp(dist.isend, send_top, prev, group), dist.P2POp(dist.isend, send_bot, nxt, group),
           dist.P2POp(dist.irecv, recv_bot, nxt, group), dist.P2POp(dist.irecv, recv_top, prev, group)]
    for req in dist.batch_isend_irecv(ops):
        req.wait()
    out[:, :halo_rows] = recv_top
    out[:, halo_rows + rows:] = recv_bot
    return out


def gather_rows(band, rows_per_rank, group=None):
    """All-gather of row bands [rows_r, W] (possibly unequal heights) into the global [sum rows, W] tensor."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return band.contiguous()
    mx = max(rows_per_rank)
    padded = torch.zeros((mx, band.shape[1]), dtype=band.dtype, device=band.device)
    padded[:band.shape[0]] = band
    parts = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(parts, padded, group=group)
    return torch.cat([p[:n] for p, n in zip(parts, rows_per_rank)], dim=0)


class BandedStereoMatching:
    """One very large frame split into row bands over the ranks of a torch.distributed (NCCL) group.

        sm = BandedStereoMatching(cuda_depth.StereoMatchingConfiguration(height=2160, width=3840, ...))
        out_band = sm.compute(left_band, right_band)     # [3, band_rows, W] each -> [band_rows, W]
        full = sm.gather(out_band)                       # optional: [H, W] on every rank

    left_right_check (a tolerance in pixels, peer-memory transport only) runs the left-right check of
    `StereoMatching.set_left_right_check` on the bands, with `invalid_disparity` and `background_fill` as there; the
    band outputs are bit-identical to it on the whole frame.  It is fixed for the object's lifetime (every rank must run
    the same exchange steps on every frame).
    """

    def __init__(self, configuration, group=None, p2p=False, variant=None, left_right_check=None, invalid_disparity=-1.0,
                 background_fill=False):
        from . import _native as N
        self._N = N
        self.group = group
        self.p2p = bool(p2p)
        if left_right_check is not None:
            left_right_check = float(left_right_check)
            if not math.isfinite(left_right_check) or left_right_check < 0:
                raise ValueError(f"tolerance must be finite and >= 0, got {left_right_check}")
            if not self.p2p:
                raise RuntimeError("the left-right check on row bands needs the peer-memory transport (p2p=True); the "
                                   "NCCL transport does not support it")
        elif background_fill:
            raise RuntimeError("background_fill needs left_right_check (a tolerance in pixels)")
        self.left_right_check = left_right_check
        self.background_fill = bool(background_fill) if left_right_check is not None else False
        self._p2p_dtype = None
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        g = configuration._as_struct()
        halo = halo_pooled_rows(g)   # 12 for the default radii; grows with large_mbm_radius / sad_patch_radius
        self.plan = BandPlan.make(g.height, g.width, g.downscale_factor, self.world, self.rank, halo)
        self.rows_per_rank = [BandPlan.make(g.height, g.width, g.downscale_factor, self.world, r, halo).band_rows
                              for r in range(self.world)]
        local = N.SdConfig(*[getattr(g, f) for f in N.CONFIG_FIELDS])
        local.height = self.plan.local_rows
        self.device = torch.cuda.current_device()
        # (with the check a launch carries the frame and its mirrored pair; set before band_p2p_init, which sizes the
        #  exported buffer for it)
        self.handle = N.Handle(local, self.device, 1 if left_right_check is None else 2)
        if variant is not None:   # e.g. "fast" pins the screened two-phase kernel (auto decides per launch size)
            self.handle.set_variant({"auto": 0, "generic": 1, "fast": 2, "ws": 3}.get(variant, variant))
        if left_right_check is not None:
            self.handle.set_lr_check(True, left_right_check, float(invalid_disparity))
            self.handle.set_lr_fill(self.background_fill)
        self.H, self.W = g.height, g.width
        self._out = torch.empty((self.plan.local_rows, self.W), dtype=torch.float32, device="cuda")
        self._gray = torch.empty((self.plan.local_rows, self.W), dtype=torch.float32, device="cuda")
        self._gl_glob = None

    def compute(self, left_band, right_band):
        N, p = self._N, self.plan
        for t in (left_band, right_band):
            if not t.is_cuda or tuple(t.shape) != (3, p.band_rows, self.W):
                raise RuntimeError(f"band must be a CUDA tensor of shape [3,{p.band_rows},{self.W}], got {list(t.shape)}")
        if left_band.dtype != right_band.dtype:
            raise RuntimeError("left and right bands must have the same dtype")
        code = N.SD_U8 if left_band.dtype == torch.uint8 else N.SD_F32
        if self.p2p:
            return self._compute_p2p(left_band, right_band, code)
        # exchange step 1: raw halo rows of both views in ONE ring send/recv over NVLink
        both = exchange_halos(torch.cat([left_band, right_band], dim=0), p.halo_rows, self.group)
        left, right = both[:3], both[3:]
        stream = torch.cuda.current_stream().cuda_stream
        self.handle.set_band(0, 0, None)
        self.handle.compute_range(left.data_ptr(), right.data_ptr(), code, 1, None, stream, 0, 0)   # gray + pool
        # exchange step 2: the fill kernel's colour reference row (k+1)*x can be anywhere in the image
        self.handle.get_stage("gray_l", 0, self._gray.data_ptr(), stream)
        mine = self._gray[p.halo_rows:p.halo_rows + p.band_rows]
        if self.world > 1 and len(set(self.rows_per_rank)) == 1:
            if self._gl_glob is None:
                self._gl_glob = torch.empty((self.H, self.W), dtype=torch.float32, device="cuda")
            dist.all_gather_into_tensor(self._gl_glob, mine, group=self.group)
        else:
            self._gl_glob = gather_rows(mine, self.rows_per_rank, self.group)
        self.handle.set_band(p.pooled_row_offset, self.H, self._gl_glob.data_ptr())
        self.handle.compute_range(None, None, code, 1, self._out.data_ptr(), stream, 1, 3)
        return self._out[p.halo_rows:p.halo_rows + p.band_rows]

    def _compute_p2p(self, left_band, right_band, code):
        p = self.plan
        if self._p2p_dtype is None:
            K = p.K
            row0 = [0]
            for r in self.rows_per_rank:
                row0.append(row0[-1] + r)
            assert row0[self.rank] == p.x0 * K
            mine = self.handle.band_p2p_init(self.world, self.rank, row0, p.halo_rows, code)
            if self.world > 1:
                t = torch.frombuffer(bytearray(mine), dtype=torch.uint8).cuda()
                allh = torch.empty(64 * self.world, dtype=torch.uint8, device="cuda")
                dist.all_gather_into_tensor(allh, t, group=self.group)
                self.handle.band_p2p_connect(bytes(allh.cpu().numpy().tobytes()))
                dist.barrier(group=self.group)   # every rank has mapped every buffer before anyone stores into one
            self._p2p_dtype = code
        elif self._p2p_dtype != code:
            raise RuntimeError("peer-memory band mode was initialised for the other input dtype")
        if not (left_band.is_contiguous() and right_band.is_contiguous()):
            raise RuntimeError("bands must be contiguous")
        stream = torch.cuda.current_stream().cuda_stream
        self.handle.band_p2p_compute(left_band.data_ptr(), right_band.data_ptr(), self._out.data_ptr(), stream)
        return self._out[p.halo_rows:p.halo_rows + p.band_rows]

    def right_map(self):
        """The right view's disparity map (right-image columns) on this rank's band rows, of the last compute() call;
        needs left_right_check."""
        if self.left_right_check is None:
            raise RuntimeError("the right view's map exists only with left_right_check")
        p = self.plan
        dst = torch.empty((p.local_rows, self.W), dtype=torch.float32, device="cuda")
        self.handle.get_stage("right", 0, dst.data_ptr(), torch.cuda.current_stream().cuda_stream)
        return dst[p.halo_rows:p.halo_rows + p.band_rows]

    def gather(self, out_band):
        return gather_rows(out_band, self.rows_per_rank, self.group)

    def close(self):
        """COLLECTIVE in peer-memory mode: every rank's exported buffer may still be written (halo stores) or read (gray
        rows) by its neighbours' kernels, so all ranks finish their work and meet at a barrier before anyone frees."""
        if self.handle is None:
            return
        torch.cuda.synchronize()
        if self.p2p and self._p2p_dtype is not None and self.world > 1 and dist.is_initialized():
            dist.barrier(group=self.group)
        self.handle.close()
        self.handle = None
