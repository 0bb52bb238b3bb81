"""ctypes binding of libstereo_b200.so (C ABI: include/stereo_b200.h).

Fails loudly when the library is missing -- there is no fallback path.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libstereo_b200.so")

SD_OK, SD_ERR_BAD_ARG, SD_ERR_SHAPE, SD_ERR_CUDA, SD_ERR_NOMEM, SD_ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5
SD_U8, SD_F32 = 0, 1
STAGES = dict(gray_l=0, gray_r=1, pool_l=2, pool_r=3, wta=4, agg3=5, refined=6, right=7)

CONFIG_FIELDS = ("height", "width", "downscale_factor", "min_disparity", "max_disparity",
                 "ncc_patch_radius", "sad_patch_radius", "threshold",
                 "small_mbm_radius", "mid_mbm_radius", "large_mbm_radius")

# every symbol include/stereo_b200.h declares
EXPORTS = ("sd_abi_version", "sd_config_default", "sd_dims", "sd_create", "sd_destroy", "sd_compute",
           "sd_compute_range", "sd_set_band", "sd_band_p2p_init", "sd_band_p2p_connect", "sd_band_p2p_compute", "sd_compute_host", "sd_get_stage", "sd_set_debug_volumes", "sd_set_compat", "sd_set_variant",
           "sd_launches_per_call", "sd_frames_per_launch", "sd_active_variant", "sd_set_screen", "sd_screen_active", "sd_screen_stats", "sd_screen_paused", "sd_profile_enable", "sd_profile_read", "sd_profile_read_detail", "sd_metrics", "sd_point_cloud", "sd_check_guards", "sd_stage_pointer", "sd_set_debug_screen", "sd_set_level_split", "sd_level_split",
           "sd_set_lr_check", "sd_set_lr_fill", "sd_lr_fill", "sd_set_rectification", "sd_rectify", "sd_reproject", "sd_last_error", "sd_last_cuda_error")


class SdConfig(C.Structure):
    _fields_ = [(f, C.c_int32) for f in CONFIG_FIELDS]


def build(force=False):
    """Compile the library in-tree with nvcc (sm_100a).  Works without a GPU."""
    import subprocess
    cmd = ["make", "-C", os.path.join(HERE, "csrc"), "-j8"] + (["-B"] if force else [])
    subprocess.check_call(cmd, stdout=subprocess.DEVNULL)
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  stereo_depth_b200 has no CPU/PyTorch fallback.")
    L = C.CDLL(LIB_PATH)
    vp, ip, fp = C.c_void_p, C.c_int, C.POINTER(C.c_float)
    i32p = C.POINTER(C.c_int32)
    L.sd_abi_version.restype = ip
    L.sd_config_default.argtypes = [C.POINTER(SdConfig)]
    L.sd_dims.argtypes = [C.POINTER(SdConfig), i32p, i32p, i32p]
    L.sd_create.argtypes = [C.POINTER(SdConfig), ip, ip, C.POINTER(vp)]
    L.sd_destroy.argtypes = [vp]
    L.sd_compute.argtypes = [vp, vp, vp, ip, ip, vp, vp]
    L.sd_compute_host.argtypes = [vp, vp, vp, ip, ip, vp]
    L.sd_compute_range.argtypes = [vp, vp, vp, ip, ip, vp, vp, ip, ip]
    L.sd_set_band.argtypes = [vp, ip, ip, vp]
    L.sd_band_p2p_init.argtypes = [vp, ip, ip, i32p, ip, ip, vp]
    L.sd_band_p2p_connect.argtypes = [vp, vp]
    L.sd_band_p2p_compute.argtypes = [vp, vp, vp, vp, vp]
    L.sd_get_stage.argtypes = [vp, ip, ip, vp, vp]
    L.sd_set_debug_volumes.argtypes = [vp, vp, vp]
    L.sd_set_debug_screen.argtypes = [vp, vp]
    L.sd_set_variant.argtypes = [vp, ip]
    L.sd_set_compat.argtypes = [vp, ip]
    L.sd_launches_per_call.argtypes = [vp, ip]
    L.sd_frames_per_launch.argtypes = [vp]
    L.sd_active_variant.argtypes = [vp]
    L.sd_set_screen.argtypes = [vp, ip]
    L.sd_screen_active.argtypes = [vp]
    L.sd_screen_stats.argtypes = [vp, C.POINTER(C.c_double), ip]
    L.sd_screen_paused.argtypes = [vp]
    L.sd_profile_enable.argtypes = [vp, ip]
    L.sd_profile_read.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_int)]
    L.sd_profile_read_detail.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_int)]
    L.sd_metrics.argtypes = [vp, vp, C.c_longlong, C.c_float, C.c_float, vp, vp]
    L.sd_point_cloud.argtypes = [vp, ip, ip, C.c_float, C.c_float, vp, vp, vp]
    L.sd_set_level_split.argtypes = [vp, ip]
    L.sd_level_split.argtypes = [vp, ip]
    L.sd_stage_pointer.argtypes = [vp, ip, ip, C.POINTER(vp)]
    L.sd_set_lr_check.argtypes = [vp, ip, C.c_float, C.c_float]
    L.sd_set_lr_fill.argtypes = [vp, ip]
    L.sd_lr_fill.argtypes = [vp, vp, ip, ip, ip, C.c_float, C.c_float, vp, vp]
    L.sd_set_rectification.argtypes = [vp, vp, vp, vp, vp, vp]
    L.sd_rectify.argtypes = [vp, vp, vp, vp, ip, ip, ip, ip, vp]
    L.sd_reproject.argtypes = [vp, ip, ip, ip, C.POINTER(C.c_double), ip, vp, vp]
    L.sd_check_guards.argtypes = [vp, C.POINTER(C.c_longlong)]
    L.sd_last_error.argtypes = [vp]
    L.sd_last_error.restype = C.c_char_p
    L.sd_last_cuda_error.argtypes = [vp]
    for n in EXPORTS:
        getattr(L, n)  # AttributeError if the header and the library ever disagree
    _lib = L
    return L


def default_config():
    c = SdConfig()
    lib().sd_config_default(C.byref(c))
    return c


def dims(cfg):
    hd, wd, l = C.c_int32(), C.c_int32(), C.c_int32()
    rc = lib().sd_dims(C.byref(cfg), C.byref(hd), C.byref(wd), C.byref(l))
    if rc != SD_OK:
        raise RuntimeError(f"invalid stereo matching configuration (sd_dims -> {rc})")
    return hd.value, wd.value, l.value


class Handle:
    """Owns one sd_handle (device scratch for `frames_per_launch` frames)."""

    def __init__(self, cfg, device, frames_per_launch=0):
        self._h = C.c_void_p()
        self.cfg = cfg
        self.device = device
        rc = lib().sd_create(C.byref(cfg), device, frames_per_launch, C.byref(self._h))
        if rc != SD_OK:
            msg = lib().sd_last_error(self._h).decode() if self._h else "allocation failed"
            if self._h:
                lib().sd_destroy(self._h)
                self._h = C.c_void_p()
            raise RuntimeError(f"sd_create failed ({rc}): {msg}")

    def check(self, rc):
        if rc != SD_OK:
            raise RuntimeError(f"libstereo_b200 error {rc}: {lib().sd_last_error(self._h).decode()}")

    def compute(self, left_ptr, right_ptr, dtype, n_frames, out_ptr, stream_ptr):
        self.check(lib().sd_compute(self._h, left_ptr, right_ptr, dtype, n_frames, out_ptr, stream_ptr))

    def compute_range(self, left_ptr, right_ptr, dtype, n_frames, out_ptr, stream_ptr, first, last):
        self.check(lib().sd_compute_range(self._h, left_ptr, right_ptr, dtype, n_frames, out_ptr, stream_ptr, first, last))

    def set_band(self, pooled_row_offset, global_height, global_left_gray_ptr):
        self.check(lib().sd_set_band(self._h, pooled_row_offset, global_height, global_left_gray_ptr))

    def band_p2p_init(self, world, rank, band_row0, halo_rows, dtype):
        """Returns this rank's 64-byte CUDA IPC handle (bytes)."""
        rows = (C.c_int32 * len(band_row0))(*band_row0)
        buf = C.create_string_buffer(64)
        self.check(lib().sd_band_p2p_init(self._h, world, rank, rows, halo_rows, dtype, buf))
        return buf.raw

    def band_p2p_connect(self, all_handles):
        self.check(lib().sd_band_p2p_connect(self._h, C.c_char_p(all_handles)))

    def band_p2p_compute(self, left_ptr, right_ptr, out_ptr, stream_ptr):
        self.check(lib().sd_band_p2p_compute(self._h, left_ptr, right_ptr, out_ptr, stream_ptr))

    def compute_host(self, left_ptr, right_ptr, dtype, n_frames, out_ptr):
        self.check(lib().sd_compute_host(self._h, left_ptr, right_ptr, dtype, n_frames, out_ptr))

    def get_stage(self, stage, frame, dst_ptr, stream_ptr):
        self.check(lib().sd_get_stage(self._h, STAGES[stage], frame, dst_ptr, stream_ptr))

    def set_debug_volumes(self, cost_ptr, agg_ptr):
        self.check(lib().sd_set_debug_volumes(self._h, cost_ptr, agg_ptr))

    def set_debug_screen(self, ptr):
        self.check(lib().sd_set_debug_screen(self._h, ptr))

    def set_compat(self, on):
        self.check(lib().sd_set_compat(self._h, 1 if on else 0))

    def set_variant(self, v):
        self.check(lib().sd_set_variant(self._h, v))

    def set_screen(self, on):
        self.check(lib().sd_set_screen(self._h, 1 if on else 0))

    @property
    def screen_active(self):
        return bool(lib().sd_screen_active(self._h))

    @property
    def screen_paused(self):
        return lib().sd_screen_paused(self._h)

    def screen_stats(self, reset=True):
        """Fraction of level pairs the fused kernel evaluated since the last reset (1.0 without the screen)."""
        f = C.c_double(1.0)
        self.check(lib().sd_screen_stats(self._h, C.byref(f), 1 if reset else 0))
        return f.value

    def launches_per_call(self, n_frames):
        return lib().sd_launches_per_call(self._h, n_frames)

    def profile_enable(self, on=True):
        self.check(lib().sd_profile_enable(self._h, 1 if on else 0))

    def profile_read(self):
        ms, n = (C.c_double * 4)(), (C.c_int * 4)()
        self.check(lib().sd_profile_read(self._h, ms, n))
        names = ("gray_pool", "cost_agg_wta", "secondary", "fill")
        return {k: (ms[i], n[i]) for i, k in enumerate(names)}

    def profile_read_detail(self):
        ms, n = (C.c_double * 6)(), (C.c_int * 6)()
        self.check(lib().sd_profile_read_detail(self._h, ms, n))
        names = ("gray_pool", "pad_planes", "level_screen", "cost_agg_wta", "secondary", "fill")
        return {k: (ms[i], n[i]) for i, k in enumerate(names)}

    def set_lr_check(self, on, tolerance=1.0, invalid_disparity=-1.0):
        self.check(lib().sd_set_lr_check(self._h, 1 if on else 0, tolerance, invalid_disparity))

    def set_lr_fill(self, on):
        self.check(lib().sd_set_lr_fill(self._h, 1 if on else 0))

    def set_rectification(self, left_map_x, left_map_y, right_map_x, right_map_y, stream_ptr):
        """Device pointers of the four float32 [H][W] maps, or four None to switch rectification off."""
        self.check(lib().sd_set_rectification(self._h, left_map_x, left_map_y, right_map_x, right_map_y, stream_ptr))

    def set_level_split(self, on):
        self.check(lib().sd_set_level_split(self._h, 1 if on else 0))

    def level_split_for(self, n_frames=1):
        return lib().sd_level_split(self._h, n_frames)

    @property
    def level_split(self):
        """Level split of a one-frame launch (1 = none)."""
        return lib().sd_level_split(self._h, 1)

    @property
    def frames_per_launch(self):
        return lib().sd_frames_per_launch(self._h)

    @property
    def active_variant(self):
        return {1: "generic", 2: "fast", 3: "ws"}.get(lib().sd_active_variant(self._h), "?")

    def stage_pointer(self, stage, frame=0):
        """Device address of a plain-float scratch plane (gray_l/r, pool_l/r, refined) of the last chunk."""
        p = C.c_void_p()
        self.check(lib().sd_stage_pointer(self._h, STAGES[stage], frame, C.byref(p)))
        return p.value

    def check_guards(self):
        """Guard-band bytes changed by stray stores (handle created with SD_DEBUG_GUARDS=1); synchronises."""
        n = C.c_longlong(0)
        self.check(lib().sd_check_guards(self._h, C.byref(n)))
        return n.value

    def close(self):
        if self._h:
            lib().sd_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
