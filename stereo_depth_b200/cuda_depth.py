"""Drop-in for the reference's `cuda_depth` extension module
(src/csrc/depth/torch_extension_module.cc:6-27): same class names, keyword arguments and defaults.

    cfg = cuda_depth.StereoMatchingConfiguration(height=1080, width=1920, downscale_factor=2,
                                                 min_disparity=0, max_disparity=127)
    sm = cuda_depth.StereoMatching(cfg)
    disp = sm.compute_disparity_map(left_cuda, right_cuda)   # [H,W] float32, aliases an internal buffer

Differences from the reference, all additive:
  * inputs may be uint8 as well as float32 (the reference needs the caller's `.float()`);
  * shape / dtype / device are validated (the reference silently reads out of bounds);
  * kernels run on PyTorch's current stream (the reference uses the legacy default stream);
  * `compute_disparity_batch` processes [N,3,H,W] in one call;
  * `set_left_right_check` marks occluded and mismatched pixels with an invalid value, or fills them from the
    background (off by default);
  * `set_rectification` takes raw frames from an unrectified rig and remaps them on the GPU first (off by default).
"""
import math

import torch

from . import _native as N


class StereoMatchingConfiguration:
    """Opaque configuration object; argument order and defaults of torch_extension_module.cc:8-19
    (note the pybind default width=1980, which differs from the C++ struct's 1920)."""

    def __init__(self, height=1080, width=1980, downscale_factor=2, min_disparity=75, max_disparity=262,
                 ncc_patch_radius=1, sad_patch_radius=5, threshold=5, small_mbm_radius=1, mid_mbm_radius=4,
                 large_mbm_radius=10):
        vals = (height, width, downscale_factor, min_disparity, max_disparity, ncc_patch_radius, sad_patch_radius,
                threshold, small_mbm_radius, mid_mbm_radius, large_mbm_radius)
        for name, v in zip(N.CONFIG_FIELDS, vals):
            if not isinstance(v, int) or isinstance(v, bool):
                # pybind11 rejects non-integers for these uint32_t/int32_t parameters with a TypeError
                raise TypeError(f"StereoMatchingConfiguration(): incompatible constructor argument {name}={v!r}")
        self._c = N.SdConfig(*vals)

    def _as_struct(self):
        return self._c

    def _key(self):
        return tuple(getattr(self._c, f) for f in N.CONFIG_FIELDS)


def _check_input(t, name):
    # same two checks and messages as CHECK_INPUT in stereo_matching.cc:13-15,23-24
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"compute_disparity_map(): incompatible function arguments ({name} is not a torch.Tensor)")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor")
    if not t.is_contiguous():
        raise RuntimeError(f"{name} must be contiguous")


class StereoMatching:
    def __init__(self, configuration=None, frames_per_launch=0, device=None):
        if configuration is None:
            # C++ default argument: stereo_matching_configuration{} -> the struct's defaults (width 1920)
            configuration = StereoMatchingConfiguration(width=1920)
        if not torch.cuda.is_available():
            raise RuntimeError("stereo_depth_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self._cfg = configuration._as_struct()
        self._device = torch.cuda.current_device() if device is None else torch.device(device).index
        self._handle = N.Handle(self._cfg, self._device, frames_per_launch)
        self.height, self.width = self._cfg.height, self._cfg.width
        self.dims = N.dims(self._cfg)
        # persistent output, like device_buffer.output_disparity (buffer/device_buffer.cc:12):
        # compute_disparity_map returns this same storage on every call
        self._out = torch.empty((self.height, self.width), dtype=torch.float32, device=self._dev())
        self._lr_tolerance = None
        self._lr_fill = False
        self._rectification = False

    def _dev(self):
        return torch.device("cuda", self._device)

    def _dtype_code(self, left, right):
        if left.dtype != right.dtype:
            raise RuntimeError("left_image and right_image must have the same dtype")
        if left.dtype == torch.uint8:
            return N.SD_U8
        if left.dtype == torch.float32:
            return N.SD_F32
        raise RuntimeError(f"images must be uint8 or float32, got {left.dtype}")

    def _check_shape(self, t, name, batch):
        want = (3, self.height, self.width)
        got = tuple(t.shape[1:]) if batch else tuple(t.shape)
        if got != want or (batch and t.dim() != 4):
            raise RuntimeError(f"{name} must have shape {'[N,' if batch else '['}3,{self.height},{self.width}], "
                               f"got {list(t.shape)}")
        if t.device.index != self._device:
            raise RuntimeError(f"{name} is on {t.device}, the matcher was created on cuda:{self._device}")

    def compute_disparity_map(self, left_image, right_image):
        _check_input(left_image, "left_image")
        _check_input(right_image, "right_image")
        self._check_shape(left_image, "left_image", False)
        self._check_shape(right_image, "right_image", False)
        code = self._dtype_code(left_image, right_image)
        stream = torch.cuda.current_stream(self._dev()).cuda_stream
        self._handle.compute(left_image.data_ptr(), right_image.data_ptr(), code, 1, self._out.data_ptr(), stream)
        return self._out

    def compute_disparity_batch(self, left_images, right_images, out=None):
        """[N,3,H,W] x2 -> [N,H,W] float32 (caller-owned, or written into `out`)."""
        _check_input(left_images, "left_image")
        _check_input(right_images, "right_image")
        self._check_shape(left_images, "left_image", True)
        self._check_shape(right_images, "right_image", True)
        if left_images.shape[0] != right_images.shape[0]:
            raise RuntimeError("left and right batches differ in length")
        n = left_images.shape[0]
        if n == 0:
            raise RuntimeError("empty batch: n_frames must be positive")
        code = self._dtype_code(left_images, right_images)
        if out is None:
            out = torch.empty((n, self.height, self.width), dtype=torch.float32, device=self._dev())
        elif (tuple(out.shape) != (n, self.height, self.width) or out.dtype != torch.float32
              or not out.is_cuda or not out.is_contiguous()):
            raise RuntimeError("out must be a contiguous float32 CUDA tensor of shape [N,H,W]")
        stream = torch.cuda.current_stream(self._dev()).cuda_stream
        self._handle.compute(left_images.data_ptr(), right_images.data_ptr(), code, n, out.data_ptr(), stream)
        return out

    def compute_disparity_host(self, left_images, right_images, out=None):
        """Host tensors in, host tensor out ([N,3,H,W] -> [N,H,W]); copies pipelined with the kernels."""
        for t, name in ((left_images, "left_image"), (right_images, "right_image")):
            if t.is_cuda:
                raise RuntimeError(f"{name} must be a CPU tensor for the host path")
            if not t.is_contiguous():
                raise RuntimeError(f"{name} must be contiguous")
            if t.dim() != 4 or tuple(t.shape[1:]) != (3, self.height, self.width):
                raise RuntimeError(f"{name} must have shape [N,3,{self.height},{self.width}], got {list(t.shape)}")
        n = left_images.shape[0]
        if right_images.shape[0] != n:
            raise RuntimeError("left and right batches differ in length")
        if n == 0:
            raise RuntimeError("empty batch: n_frames must be positive")
        code = self._dtype_code(left_images, right_images)
        if out is None:
            out = torch.empty((n, self.height, self.width), dtype=torch.float32).pin_memory()
        elif (not isinstance(out, torch.Tensor) or out.is_cuda or out.dtype != torch.float32 or not out.is_contiguous()
              or tuple(out.shape) != (n, self.height, self.width)):
            raise RuntimeError("out must be a contiguous float32 CPU tensor of shape [N,H,W]")
        self._handle.compute_host(left_images.data_ptr(), right_images.data_ptr(), code, n, out.data_ptr())
        return out

    def set_left_right_check(self, tolerance=1.0, invalid_disparity=-1.0, background_fill=False):
        """Left-right consistency check on every entry point of this matcher (default off).

        Each frame is also matched as the mirrored pair (flip(right), flip(left)), which gives the right view's disparity
        map; a left pixel with disparity d at column c keeps d only if d is finite, c - rint(d) is inside the image and
        the right map there differs from d by at most `tolerance` full-resolution pixels, else it becomes
        `invalid_disparity`.  Costs about twice the device time.  `set_left_right_check(None)` switches it off.
        Needs a matcher created with frames_per_launch != 1 (a launch carries a frame and its mirrored pair).

        background_fill=True instead gives each run of rejected pixels in a row the smaller of the two kept values that
        bound it (occluded pixels lie on the background), a run at the image border its one kept neighbour; rows with
        no kept pixel copy the nearest non-empty row above the first / below the last one (DESIGN.md §13).  Only rows
        between non-empty rows, and frames without any kept pixel, keep `invalid_disparity`."""
        if tolerance is None:
            self._handle.set_lr_check(False)
            self._lr_tolerance = None
            self._lr_fill = False
            return
        tolerance = float(tolerance)
        if not math.isfinite(tolerance) or tolerance < 0:
            raise ValueError(f"tolerance must be finite and >= 0, got {tolerance}")
        self._handle.set_lr_check(True, tolerance, float(invalid_disparity))
        self._lr_tolerance = tolerance
        self._handle.set_lr_fill(bool(background_fill))
        self._lr_fill = bool(background_fill)

    @property
    def left_right_check(self):
        """The left-right check's tolerance in pixels, or None while the check is off."""
        return self._lr_tolerance

    @property
    def background_fill(self):
        """True while the left-right check fills the pixels it rejects instead of marking them invalid."""
        return self._lr_fill

    def _map_tensor(self, m, name):
        if isinstance(m, torch.Tensor):
            t = m
        else:
            import numpy as np
            if not isinstance(m, np.ndarray):
                raise TypeError(f"{name} must be a numpy array or a torch tensor, got {type(m).__name__}")
            t = torch.from_numpy(m)
        if t.dtype != torch.float32 or tuple(t.shape) != (self.height, self.width):
            raise RuntimeError(f"{name} must be a float32 [{self.height},{self.width}] map (cv2.initUndistortRectifyMap "
                               f"with m1type=cv2.CV_32FC1), got {t.dtype} {list(t.shape)}")
        return t.to(self._dev()).contiguous()

    def set_rectification(self, left_maps, right_maps):
        """Rectify raw frames on the GPU before matching, on every entry point of this matcher (default off).

        left_maps / right_maps: (map_x, map_y) of each view as cv2.initUndistortRectifyMap returns them with
        m1type=cv2.CV_32FC1 -- float32 [H,W] numpy arrays or tensors giving, for every rectified pixel, the raw image's
        sampling coordinate.  Every view is then remapped exactly as cv2.remap(raw, map_x, map_y, cv2.INTER_LINEAR,
        borderMode=cv2.BORDER_CONSTANT, borderValue=0) would (DESIGN.md §14), and the outputs are in rectified (left)
        coordinates.  The maps are copied to the matcher's device, so the caller may change theirs afterwards.
        `set_rectification(None, None)` switches it off."""
        if left_maps is None and right_maps is None:
            self._handle.set_rectification(None, None, None, None, None)
            self._rectification = False
            return
        maps = []
        for pair, view in ((left_maps, "left"), (right_maps, "right")):
            if pair is None or len(pair) != 2:
                raise RuntimeError(f"{view}_maps must be a (map_x, map_y) pair, or both maps None to switch off")
            maps += [self._map_tensor(m, f"{view} map_{a}") for m, a in zip(pair, "xy")]
        stream = torch.cuda.current_stream(self._dev()).cuda_stream
        self._handle.set_rectification(*[m.data_ptr() for m in maps], stream)
        self._rectification = True

    @property
    def rectification(self):
        """True while this matcher rectifies its input frames (set_rectification)."""
        return self._rectification

    # ---- parity / debugging hooks (not part of the reference API) -------------------------------
    def stage(self, name, frame=0):
        H, W = self.height, self.width
        Hd, Wd, _ = self.dims
        # ("right": the right view's disparity map of the left-right check, right-image columns)
        shape = {"gray_l": (H, W), "gray_r": (H, W), "pool_l": (Hd, Wd), "pool_r": (Hd, Wd), "wta": (Hd, Wd),
                 "agg3": (Hd, Wd, 3), "refined": (Hd, Wd), "right": (H, W)}[name]
        dst = torch.empty(shape, dtype=torch.float32, device=self._dev())
        stream = torch.cuda.current_stream(self._dev()).cuda_stream
        self._handle.get_stage(name, frame, dst.data_ptr(), stream)
        return dst

    def debug_volumes(self, enable=True):
        """Allocate [Hd,Wd,L] cost / aggregated volumes that the fused kernel fills for frame 0."""
        if not enable:
            self._handle.set_debug_volumes(None, None)
            self._dbg = None
            return None
        Hd, Wd, L = self.dims
        self._dbg = (torch.zeros((Hd, Wd, L), dtype=torch.float32, device=self._dev()),
                     torch.zeros((Hd, Wd, L), dtype=torch.float32, device=self._dev()))
        self._handle.set_debug_volumes(self._dbg[0].data_ptr(), self._dbg[1].data_ptr())
        return self._dbg

    def debug_screen(self, enable=True):
        """Allocate an [Hd,Wd,L] volume that the level screen fills with its APPROXIMATE aggregated costs of frame 0."""
        if not enable:
            self._handle.set_debug_screen(None)
            self._dbg_screen = None
            return None
        Hd, Wd, L = self.dims
        self._dbg_screen = torch.zeros((Hd, Wd, L), dtype=torch.float32, device=self._dev())
        self._handle.set_debug_screen(self._dbg_screen.data_ptr())
        return self._dbg_screen

    def set_compat(self, on=True):
        """Reproduce (True) or fix (False) the reference's absolute-index read for min_disparity != 0."""
        self._handle.set_compat(on)

    def set_variant(self, v):
        self._handle.set_variant({"auto": 0, "generic": 1, "fast": 2, "ws": 3}.get(v, v))

    def set_level_split(self, on=True):
        """Level split of launches too small to fill the GPU (default on; results identical)."""
        self._handle.set_level_split(on)

    def level_split(self, n_frames=1):
        return self._handle.level_split_for(n_frames)

    def set_screen(self, on=True):
        """Certified level screen in front of the fused kernel (default on where supported; results identical)."""
        self._handle.set_screen(on)

    @property
    def screen_active(self):
        return self._handle.screen_active

    @property
    def screen_paused(self):
        """Chunks left in the current pause of the adaptive screen policy (0 = screening)."""
        return self._handle.screen_paused

    def screen_stats(self, reset=True):
        return self._handle.screen_stats(reset)

    def profile(self, on=True):
        self._handle.profile_enable(on)

    def profile_read(self):
        """{kernel: (milliseconds, launches)} accumulated since the last read (device time, CUDA events)."""
        return self._handle.profile_read()

    def profile_read_detail(self):
        return self._handle.profile_read_detail()

    def launches_per_call(self, n_frames=1):
        return self._handle.launches_per_call(n_frames)

    @property
    def frames_per_launch(self):
        return self._handle.frames_per_launch

    @property
    def active_variant(self):
        return self._handle.active_variant
