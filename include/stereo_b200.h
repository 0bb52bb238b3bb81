/* stereo_b200.h -- C ABI of libstereo_b200.so, the sm_100a stereo-matching backend.
 *
 * Drop-in boundary for the reference's `cuda_depth` pybind module
 * (reference: src/csrc/depth/torch_extension_module.cc:6-27) and the C++ class behind it
 * (src/csrc/depth/stereo_matching.hh:8-34, stereo_matching.cc:17-43).  Plain pointers and
 * sizes only; no torch types.  The Python shim stereo_depth_b200/cuda_depth.py binds these
 * entry points with ctypes (see INTEGRATION.md for the reference-side stub).
 *
 * All image pointers of sd_compute are DEVICE pointers on the handle's device.
 * All functions return SD_OK (0) or a negative sd_status; sd_last_error() gives the text.
 * A handle is not thread-safe; distinct handles are independent.
 */
#ifndef STEREO_B200_H
#define STEREO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SD_ABI_VERSION 3   /* 2: level screen, peer-memory row bands, detailed profile read; 3: guard bands (additions only) */

/* Replaces struct stereo_matching_configuration
 * (src/csrc/depth/stereo_matching_configuration.hh:5-17); field order = the pybind ctor's
 * argument order (torch_extension_module.cc:8-19). */
typedef struct sd_config {
    int32_t height;            /* 1080 */
    int32_t width;             /* 1920 (the pybind default is 1980, torch_extension_module.cc:10) */
    int32_t downscale_factor;  /* 2    K */
    int32_t min_disparity;     /* 75 */
    int32_t max_disparity;     /* 262 */
    int32_t ncc_patch_radius;  /* 1    3x3 similarity cost on the pooled images */
    int32_t sad_patch_radius;  /* 5    11x11 secondary matching on the full-res images */
    int32_t threshold;         /* 5    bilateral-fill disparity threshold */
    int32_t small_mbm_radius;  /* 1 */
    int32_t mid_mbm_radius;    /* 4 */
    int32_t large_mbm_radius;  /* 10 */
} sd_config;

typedef struct sd_handle sd_handle;

typedef enum sd_status {
    SD_OK = 0,
    SD_ERR_BAD_ARG = -1,      /* null pointer, non-positive size, radius ordering ... */
    SD_ERR_SHAPE = -2,        /* n_frames / dtype / stage does not fit the handle */
    SD_ERR_CUDA = -3,         /* a CUDA call failed; sd_last_cuda_error() holds the cudaError_t */
    SD_ERR_NOMEM = -4,
    SD_ERR_UNSUPPORTED = -5
} sd_status;

typedef enum sd_dtype { SD_U8 = 0, SD_F32 = 1 } sd_dtype;

/* Intermediates kept in HBM for the LAST frame chunk processed (parity tests / debugging).
 * Replaces nothing in the reference API: its device_buffer (buffer/device_buffer.hh:12-19) is private. */
typedef enum sd_stage {
    SD_STAGE_GRAY_L = 0,   /* float [H,W]    rgb_to_grayscale.cu:24-28 */
    SD_STAGE_GRAY_R = 1,
    SD_STAGE_POOL_L = 2,   /* float [Hd,Wd]  mean_pool.cu:25-35 */
    SD_STAGE_POOL_R = 3,
    SD_STAGE_WTA = 4,      /* float [Hd,Wd]  wta_disparity_selection.cu:22-30 (disparity incl. min_d/K) */
    SD_STAGE_AGG3 = 5,     /* float [Hd,Wd,3] aggregated cost at d*-1, d*, d*+1 (circular), the three
                              values secondary_matching.cu:55-58 reads from the aggregated volume */
    SD_STAGE_REFINED = 6,  /* float [Hd,Wd]  secondary_matching.cu:55-70 */
    SD_STAGE_RIGHT = 7     /* float [H,W]    the right view's disparity map (right-image columns) of the left-right
                              check; frame < frames_per_launch / 2; only while the check is on */
} sd_stage;

int sd_abi_version(void);

/* Fills *cfg with the reference's defaults (stereo_matching_configuration.hh:6-16). */
int sd_config_default(sd_config *cfg);

/* Hd = ceil(H/K), Wd = ceil(W/K), L = max/K - min/K + 1 (buffer/device_buffer.cc:7-9). */
int sd_dims(const sd_config *cfg, int32_t *Hd, int32_t *Wd, int32_t *L);

/* Replaces stereo_matching::stereo_matching (stereo_matching.cc:17-20): validates the configuration
 * and allocates all scratch for `frames_per_launch` frames on `device` (<=0 selects a default).
 * Unlike the reference, no [Hd,Wd,L] cost volume is ever allocated. */
int sd_create(const sd_config *cfg, int device, int frames_per_launch, sd_handle **out);
int sd_destroy(sd_handle *h);

/* Replaces stereo_matching::compute_disparity_map (stereo_matching.cc:22-43) for a batch:
 * left/right: [n_frames,3,H,W] CHW, uint8 or float32 (values as the reference sees them after
 * `.float()`), contiguous, device memory.  out: float32 [n_frames,H,W] device memory.
 * Asynchronous on `cuda_stream` (a cudaStream_t; NULL = legacy default stream, which is the
 * stream the reference launches on).  No allocation, no host synchronisation. */
int sd_compute(sd_handle *h, const void *left, const void *right, int dtype, int n_frames,
               float *out, void *cuda_stream);

/* Runs only kernels first_kernel..last_kernel (0 gray+pool, 1 cost+aggregation+WTA, 2 secondary matching,
 * 3 upscale+fill) of one chunk (n_frames <= frames_per_launch), so a caller can place a collective between
 * stages.  Used by the row-band mode: kernel 0, all-gather of the left gray bands over NCCL, kernels 1..3. */
int sd_compute_range(sd_handle *h, const void *left, const void *right, int dtype, int n_frames,
                     float *out, void *cuda_stream, int first_kernel, int last_kernel);

/* Row-band mode for a single very large frame split across GPUs (no reference counterpart: the
 * reference is single-GPU).  The handle's image is a window of `global_height` rows of a larger image:
 * local pooled row 0 is global pooled row `pooled_row_offset` (may be negative: circular).  The
 * vertical/horizontal fill then applies the reference's row rules (upscale_disparity_vertical_fill.cu:26-31,
 * horizontal_disparity_fill.cu:26-27) with GLOBAL row numbers and reads its colour reference row from
 * `global_left_gray` ([global_height, W] floats, device).  global_height <= 0 switches back to normal mode. */
int sd_set_band(sd_handle *h, int pooled_row_offset, int global_height, const float *global_left_gray);

/* Row-band mode over PEER MEMORY (NVLink / NVSwitch), one process per GPU: the halo exchange and the left-gray exchange of
 * sd_set_band's mode as kernels that store directly into the other ranks' HBM and signal with system-scope flags (no NCCL
 * call, no host synchronisation on the data path).
 *   sd_band_p2p_init     the handle must have been created with height = band rows + 2 * halo_rows.  band_row0[world+1]:
 *                        first full-resolution row of every rank's band, band_row0[world] = global height.  Allocates the
 *                        exported buffers and writes this rank's 64-byte CUDA IPC handle to ipc_handle_out.
 *                        The left-right check and its background fill (sd_set_lr_check / sd_set_lr_fill) must be set
 *                        before this call and are then fixed for the handle (every rank runs the same exchange steps on
 *                        every frame): all ranks must use the same settings.  With the check the exported buffer also
 *                        holds the mirrored frame's left gray band; with the fill, two fill-bounds areas of
 *                        256 + 8 * W bytes (rounded up to 256) and a third exchange step per frame (DESIGN.md §8).
 *                        Without the check its size and layout are those of the unchecked mode.  Rectification is
 *                        refused (SD_ERR_UNSUPPORTED): the remap reads raw rows outside the halo, as far as the maps move
 *                        rows.
 *   sd_band_p2p_connect  ipc_handles: the world x 64 bytes of all ranks (exchanged by the caller, e.g. an all-gather).
 *   sd_band_p2p_compute  left_band / right_band: [3, band rows, W] of `dtype` (device); out: [band rows + 2 * halo_rows, W]
 *                        floats, rows halo_rows .. halo_rows + band rows - 1 are this rank's part of the disparity map.
 *                        With the check a call runs one pair (a 2-frame launch); those rows equal sd_compute with the
 *                        same settings on the whole frame bit for bit, and SD_STAGE_RIGHT (frame 0) returns the right
 *                        view's map of the window, likewise exact on the band rows.
 * Every rank must call sd_band_p2p_compute the same number of times: a wait that sees no peer for ~10 s gives up (the
 * CUDA context stays usable) and the next sd_band_p2p_compute returns SD_ERR_CUDA with a "timed out" message.
 * sd_destroy on such a handle is COLLECTIVE in effect: peers may still store into / read from the exported buffer, so
 * synchronise all ranks before any of them destroys its handle (BandedStereoMatching.close() does). */
int sd_band_p2p_init(sd_handle *h, int world, int rank, const int32_t *band_row0, int halo_rows, int dtype, void *ipc_handle_out);
int sd_band_p2p_connect(sd_handle *h, const void *ipc_handles);
int sd_band_p2p_compute(sd_handle *h, const void *left_band, const void *right_band, float *out, void *cuda_stream);

/* Same computation with HOST buffers (pinned memory recommended): host->device copies, the
 * kernels and device->host copies are pipelined over internal streams, chunk by chunk.
 * Synchronous: returns when `out` is complete.  This is the end-to-end call
 * CudaStereoMatchingBackend.process makes for CPU tensors
 * (src/python/pipeline/depth/cuda_stereo_matching_backend.py:13-17). */
int sd_compute_host(sd_handle *h, const void *left, const void *right, int dtype, int n_frames,
                    float *out);

/* Copies one intermediate of frame `frame` (index inside the last chunk) to device memory `dst`
 * on `cuda_stream`. */
int sd_get_stage(sd_handle *h, int stage, int frame, float *dst, void *cuda_stream);

/* Zero-copy variant for the stages that live in scratch as plain float planes (gray, pooled, refined): the device
 * address inside the handle's scratch, valid until the next call that processes a chunk (order your reads after it on
 * the same stream).  SD_ERR_UNSUPPORTED for SD_STAGE_WTA / SD_STAGE_AGG3 (stored as packed records). */
int sd_stage_pointer(sd_handle *h, int stage, int frame, const float **ptr);

/* Debug/parity hook: when non-NULL, the fused kernel additionally stores the cost and aggregated
 * volumes ([Hd,Wd,L] floats, d innermost, device memory) of frame 0 of each chunk -- the two
 * tensors the reference materialises (buffer/device_buffer.cc:9-10).  Pass NULLs to switch off. */
int sd_set_debug_volumes(sd_handle *h, float *cost_volume, float *aggregated_volume);

/* Parity hook for the level screen: when non-NULL, mbm_screen_kernel additionally stores its APPROXIMATE aggregated
 * costs of frame 0 of each chunk ([Hd,Wd,L] floats, d innermost, device memory), so that a test can hold the kernel's own
 * sums against the error bound the screen relies on (header of csrc/mbm_screen.cu).  NULL switches it off. */
int sd_set_debug_screen(sd_handle *h, float *approx_volume);

/* Reference-compat switch for min_disparity != 0.  The reference's secondary matching reads the aggregated
 * volume at pad_index(ABSOLUTE disparity, L) with unchecked flat addressing (secondary_matching.cu:28-31), which
 * for min_disparity/K != 0 is a different cell than the arg-max's neighbours (an upstream bug).  on = 1 (the
 * default whenever min_disparity/K != 0): reproduce it bit for bit; this materialises the aggregated volume
 * (frames_per_launch * Hd*Wd*L floats).  on = 0: use the relative index (what the algorithm intends; no volume).
 * With min_disparity/K == 0 both are identical and no volume is ever allocated unless on = 1 is forced. */
int sd_set_compat(sd_handle *h, int on);

/* Selects the fused-kernel variant: 0 = auto, 1 = generic (any radii), 2 = specialised
 * (radii 1/4/10, cost radius 1), 3 = warp-specialised producer/consumer schedule of the same arithmetic (experimental).  SD_ERR_UNSUPPORTED if the configuration does not allow it. */
int sd_set_variant(sd_handle *h, int variant);

/* Certified level screen in front of the specialised fused kernel (default: on wherever it is supported, i.e.
 * variant 0/2, radii 1/4/10, 3 <= L <= 128, no debug volumes, no reference-compat volume).  A cheap kernel bounds
 * every aggregated cost from separable sums and flags, per 32x64 tile, the level pairs that can still hold the
 * reference's arg-max (rigorous fp32 error bound, stereo_depth_b200/csrc/mbm_screen.cu); the fused kernel then
 * evaluates the reference's sequential chains (multi_block_matching_cost_aggregation.cu:56-87) only for those.
 * Results are bit-identical with the screen on or off; only the run time changes (and becomes scene dependent).
 * With variant 0 the screen is skipped for launches of less than about two waves of tiles (single small frames), where
 * the heaviest tile bounds the launch time; sd_screen_active / sd_active_variant answer for a full chunk.
 * sd_screen_stats: fraction of level pairs the fused kernel had to evaluate since the last reset (synchronises). */
int sd_set_screen(sd_handle *h, int on);
int sd_screen_active(sd_handle *h);
int sd_screen_stats(sd_handle *h, double *evaluated_fraction, int reset);
/* Adaptive policy: when a chunk's screen left more than 70 % of the level pairs to evaluate (flat or periodic scenes),
 * the screen is skipped for the next 32 chunks and then probed again.  Returns the chunks left in the current pause. */
int sd_screen_paused(sd_handle *h);

/* Number of kernels one sd_compute call launches for n_frames frames (with the left-right check: chunks of
 * frames_per_launch / 2 pairs, each counted as one launch of twice its frames plus the second fill launch, plus 2 more
 * -- the row and column passes -- with the background fill). */
int sd_launches_per_call(sd_handle *h, int n_frames);

int sd_frames_per_launch(sd_handle *h);

/* Left-right consistency check (OpenCV's disp12MaxDiff), off by default.  With on != 0 every frame is also matched
 * as the mirrored pair (flip(right), flip(left)) -- the same kernels and semantics -- whose output, mirrored back, is
 * the right view's disparity map dR (right-image columns).  Each left pixel with value d = out[r][c] is then kept bit
 * for bit if d is finite, yr = c - rint(d) (round half to even) lies in [0, W) and |d - dR[r][yr]| <= tolerance
 * (fp32 subtraction); otherwise it is set to invalid_disparity.  This marks most occluded pixels (no partner in the
 * right view); consistent errors such as foreground fattening at object edges remain.
 * tolerance: full-resolution pixels, finite and >= 0 (SD_ERR_BAD_ARG otherwise); invalid_disparity: any float.
 * Kernels A..C run once per frame and view in shared launches, so a chunk holds frames_per_launch / 2 pairs and a
 * call costs about twice the device time; the fill writes both maps and checks in its epilogue.  Allocates the right
 * maps of one chunk (frames_per_launch / 2 * H * W floats, readable as SD_STAGE_RIGHT); on = 0 frees them and
 * restores the unchecked path exactly.  SD_ERR_SHAPE for a handle created with frames_per_launch = 1.
 * Row bands: supported over peer memory when set BEFORE sd_band_p2p_init (any call on or off after it is
 * SD_ERR_UNSUPPORTED); the NCCL transport (sd_set_band, sd_compute_range) refuses it, in either order. */
int sd_set_lr_check(sd_handle *h, int on, float tolerance, float invalid_disparity);

/* Background fill of the pixels the left-right check rejects (KITTI devkit's interpolateBackground), off by default.
 * A hole is a pixel the check rejects -- never a pixel whose value merely equals invalid_disparity.  In each row with a
 * kept pixel, a run of holes gets the smaller of the two kept values that bound it (dR < dL ? dR : dL of its right and
 * left neighbour, so the left one on ties), a run at a border its one kept neighbour; kept pixels stay bit for bit.
 * Rows without a kept pixel above the first non-empty row copy that row, below the last one copy that row, and
 * otherwise stay invalid_disparity (all of them in a frame without a kept pixel).  Every output value is thus a kept
 * left value or invalid_disparity.  With on != 0 the second fill launch of a chunk writes the unchecked left maps and
 * two more launches check and fill them in place.  Allocates frames_per_launch / 2 * H bytes of row flags, freed with
 * the check.  SD_ERR_UNSUPPORTED while the check is off and after sd_band_p2p_init (set it before, like the check);
 * sd_set_lr_check(h, 0, ...) also switches the fill off, and sd_set_lr_check(h, 1, ...) with the check already on keeps
 * the fill setting. */
int sd_set_lr_fill(sd_handle *h, int on);

/* The left-right check plus the background fill (sd_set_lr_fill) without a handle: left_map = n unchecked [H][W] maps,
 * right_map = the right views' maps in right-image columns, out = n [H][W] maps, all float32 in device memory.  out
 * may be left_map (in place) but not right_map.  tolerance as in sd_set_lr_check.  Stream-ordered on cuda_stream
 * (allocates n * H bytes of scratch with cudaMallocAsync).  SD_ERR_BAD_ARG for null pointers, n, H or W <= 0,
 * n * H > INT_MAX, a tolerance that is not finite and >= 0, or out == right_map; SD_ERR_CUDA if a launch fails. */
int sd_lr_fill(const float *left_map, const float *right_map, int n, int H, int W, float tolerance, float invalid_disparity,
               float *out, void *cuda_stream);

/* Stereo rectification on the device, off by default: with it on, every entry point (sd_compute, sd_compute_host) takes
 * RAW frames and first remaps each view exactly as cv2.remap(src, map_x, map_y, INTER_LINEAR, BORDER_CONSTANT, 0) with
 * the CV_32FC1 maps of cv2.initUndistortRectifyMap (rule: DESIGN.md §14), then runs the unchanged pipeline on the
 * rectified frames.  Source and rectified images are both the handle's H x W.
 *   sd_set_rectification  the four maps: device float32 [H][W] each (output pixel -> source coordinate).  They are
 *                         copied into the handle, stream-ordered on cuda_stream, so the caller may reuse or free theirs
 *                         in that stream's order.  Allocates 4 * H * W floats of maps plus the rectified frames of one
 *                         chunk, frames_per_launch * 2 * 3 * H * W * 4 bytes (sized for float32 input; 1.44 GB at the
 *                         1080p default of 29 frames per launch).  All four maps NULL switches rectification off, frees
 *                         both and restores the unrectified path exactly; a partial set of NULLs is SD_ERR_BAD_ARG.
 *                         The remap is one more launch per chunk (sd_launches_per_call) and counts as kernel 0 in the
 *                         per-kernel profile.  SD_ERR_UNSUPPORTED for H or W >= 32768 and together with the row-band
 *                         modes (sd_set_band, sd_band_p2p_init, sd_compute_range), in either order.
 *   sd_rectify            the same remap without a handle: n_planes [H][W] planes of dtype (SD_U8 / SD_F32) at src,
 *                         each sampled with the same map, written to dst (device memory, must not overlap src).
 *                         Asynchronous on cuda_stream.  SD_ERR_BAD_ARG for null pointers, non-positive sizes, H or
 *                         W >= 32768, an unknown dtype or dst == src; SD_ERR_CUDA if the launch fails. */
int sd_set_rectification(sd_handle *h, const float *left_map_x, const float *left_map_y, const float *right_map_x,
                         const float *right_map_y, void *cuda_stream);
int sd_rectify(const float *map_x, const float *map_y, const void *src, void *dst, int dtype, int n_planes, int H, int W,
               void *cuda_stream);

/* Reprojection of disparity maps to metric 3-D points, exactly cv2.reprojectImageTo3D(disparity, Q, xyz,
 * handleMissingValues) with float32 maps (rule: DESIGN.md §15): n float32 [H][W] maps at `disparity` (device memory)
 * -> xyz = n float32 [H][W][3] point maps (X, Y, Z interleaved, OpenCV's CV_32FC3; device memory).  Q: the 4x4
 * reprojection matrix of cv2.stereoRectify as 16 row-major doubles in HOST memory, read during the call.  With
 * handle_missing_values != 0 every pixel whose disparity lies within FLT_EPSILON of its frame's minimum gets Z = 10000;
 * the minimum is taken over the non-NaN values (OpenCV's is undefined with NaN) and a frame that is all NaN has none.
 * Asynchronous on cuda_stream (handle_missing_values allocates n * 4 bytes of scratch with cudaMallocAsync and adds one
 * launch).  SD_ERR_BAD_ARG for null pointers, n, H or W <= 0, or xyz overlapping disparity; SD_ERR_CUDA if a launch
 * fails. */
int sd_reproject(const float *disparity, int n, int H, int W, const double *Q, int handle_missing_values, float *xyz,
                 void *cuda_stream);

/* Level split for launches that cannot fill the GPU (one small frame, a thin row band): the unscreened specialised
 * kernel then spreads every tile's disparity levels over several blocks and a small kernel merges the partial
 * winner-take-all records (identical results: the maximum is taken in ascending level order with strict '>').
 * sd_level_split: the split a launch of n_frames frames would use (1 = none); sd_set_level_split(h, 0) disables it. */
int sd_set_level_split(sd_handle *h, int on);
int sd_level_split(sd_handle *h, int n_frames);

/* The fused-kernel variant the next sd_compute will run: 1 generic, 2 specialised, 3 warp-specialised
 * (variant 0 = auto picks 2 or 3 per shape from a wave/tile cost model, see sd_create in api.cu). */
int sd_active_variant(sd_handle *h);

/* Per-kernel device timing for benchmarks: while enabled, sd_compute brackets each of its four
 * kernels (0 gray+pool, 1 cost+aggregation+WTA, 2 secondary matching, 3 upscale+fill) with CUDA
 * events on the launching stream.  sd_profile_read waits for the last event, returns the summed
 * milliseconds and launch counts per kernel ([4] each) since the previous read, and resets them. */
int sd_profile_enable(sd_handle *h, int on);
int sd_profile_read(sd_handle *h, double *ms_per_kernel, int *launches_per_kernel);
/* Same, with kernel 1 split into its launches: [6] each = gray+pool, plane padding, level screen, cost+aggregation+WTA
 * (exact evaluation), secondary matching, upscale+fill.  Either read resets the counters. */
int sd_profile_read_detail(sd_handle *h, double *ms_per_kernel, int *launches_per_kernel);
/* ---- consumers of the disparity map (stateless; device pointers; asynchronous on cuda_stream) --------------
 * Accuracy metrics of depth_estimation_pipeline_metrics.py:18-56 over the mask `0 < gt <= max_disparity`
 * (depth_estimation_pipeline_runner.py:85): metrics_out[4] doubles in device memory =
 * {masked pixels, D1 outliers (|e|>3 and |e|/|gt|>0.05), pixels with |e|>threshold, sum of |e|}. */
int sd_metrics(const float *disparity, const float *gt_disparity, long long n, float max_disparity, float threshold,
               double *metrics_out, void *cuda_stream);

/* Disparity -> depth -> point list of depth_estimation_pipeline_hooks.py:84-92 / helpers/point_cloud_helpers.py:5-13:
 * for every pixel with disparity != invalid_disparity, in row-major order, (column, row, focal*baseline/disparity).
 * xyz: [H*W,3] floats; scratch: ceil(H*W/1024)+1 ints, the point count is left in scratch[ceil(H*W/1024)]. */
int sd_point_cloud(const float *disparity, int H, int W, float focal_times_baseline, float invalid_disparity, float *xyz,
                   int *scratch, void *cuda_stream);

/* Debug aid standing in for a memory checker: with SD_DEBUG_GUARDS=1 in the environment at sd_create, every scratch
 * allocation of the handle is bracketed by 64 KB guard bands holding a known pattern.  sd_check_guards synchronises the
 * device and returns in *corrupted_bytes how many guard bytes (incl. the slack behind each payload) a stray store has
 * changed since sd_create.  SD_ERR_UNSUPPORTED when the handle was created without guards. */
int sd_check_guards(sd_handle *h, long long *corrupted_bytes);

const char *sd_last_error(sd_handle *h);
int sd_last_cuda_error(sd_handle *h);

#ifdef __cplusplus
}
#endif
#endif /* STEREO_B200_H */
