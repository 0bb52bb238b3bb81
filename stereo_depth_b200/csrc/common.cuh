// Shared declarations of libstereo_b200.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/stereo_b200.h"

namespace sd {

// std::numeric_limits<float>::min() -- the reference's WTA / secondary-matching initial "best"
// (wta_disparity_selection.cu:22, secondary_matching.cu:45).
constexpr float kFltMin = 1.17549435e-38f;

// True modulo: the SAFE definition of the reference's pad_index (device_functions.cuh:10-20).
// Identical to pad_index wherever pad_index stays inside the tensor (index in [-n, n]); for
// index > n, where the reference forms a negative flat offset, we wrap instead.
__host__ __device__ __forceinline__ int wrapm(int i, int n) {
    if ((unsigned)i < (unsigned)n) return i;
    i %= n;
    return i < 0 ? i + n : i;
}

// The reference's pad_index, verbatim (device_functions.cuh:10-20): may return a NEGATIVE index.
__host__ __device__ __forceinline__ int ref_pad_index(int index, int n) {
    if (index >= 0 && index < n) return index;
    if (index < 0) return n + index;
    if (index == n) return 0;
    return n - index;
}

// Geometry shared by all kernels of one handle.
struct Geom {
    int H, W, K, Hd, Wd, L;
    int min_ds;        // min_disparity / K   (stereo_matching.cc:61)
    int r_cost;        // ncc_patch_radius
    int r_sad;         // sad_patch_radius
    int rs, rm, rl;    // small / mid / large multi-block radii
    float threshold;
    // Row-band mode (single very large frame split over GPUs, bands.py): this handle processes a window of
    // the global image.  band_x_off = global pooled row of local pooled row 0 (may be negative: circular),
    // Hd_glob / H_glob = global heights.  Normal mode: 0, Hd, H.
    int band_x_off, Hd_glob, H_glob;
    // != 0: secondary matching indexes the aggregated volume with the ABSOLUTE disparity, like the reference
    // (secondary_matching.cu:28-31).  Default when min_disparity/K != 0.  Needs Scratch::agg_vol, which holds
    //   1: the whole volume, plane-major [F][L][Hd*Wd]  (written by the fused kernel while it evaluates every level)
    //   2: only the level pairs some pixel's absolute-index read asks for, per 32x64 tile:
    //      [F*tiles][rank of the pair in Scratch::gather_mask][level parity][32*64]  (gather pass, api.cu run_chunk)
    int abs_index;
};

// Wrap-padded copies of the pooled planes for the specialised fused kernel: every tile's left/right row band
// (with the reference's circular padding, pad_index / device_functions.cuh:10-20, already applied) is a set of
// contiguous, 16-byte aligned row segments, so the kernel stages it with TMA bulk copies (cp.async.bulk).
//   left  plane: [rows][pwl], padded col = virtual col + 15,       padded row = virtual row + 11
//   right plane: [rows][pwr], padded col = virtual col + shift_r   (shift_r = 10 + min_ds + Lp: a tile's band then
//                starts at padded column c0, a multiple of 64, whatever min_ds and L are)
constexpr int kTileH = 32, kTileW = 64;   // pixels per tile of the specialised kernel
constexpr int kBandRows = 56;             // band rows staged per tile (54 used + 2 only dead work items touch)
constexpr int kBandLW = 96;               // left band pitch in shared memory (floats)
constexpr int kScreenBuckets = 8;         // cost classes of the screened tiles (mbm_screen.cu -> mbm_wta_fast.cu)
constexpr int kScreenCtrlInts = 16;       // bucket counts [8] | per-chunk pair accumulator (u64) | finished-block counter | pad
struct PadGeom {
    int tiles_x, tiles_y, rows, pwl, pwr, rw, shift_r;
};
__host__ __device__ inline PadGeom make_pad_geom(int Hd, int Wd, int L, int min_ds) {
    PadGeom p;
    const int Lp = (L + 1) & ~1;
    p.tiles_x = (Wd + kTileW - 1) / kTileW;
    p.tiles_y = (Hd + kTileH - 1) / kTileH;
    p.rows = (p.tiles_y - 1) * kTileH + kBandRows;
    {   // the warp-specialised variant uses 64-row tiles and 86 band rows: allocate for whichever needs more
        const int rows64 = ((Hd + 63) / 64 - 1) * 64 + 86;
        if (rows64 > p.rows) p.rows = rows64;
    }
    p.shift_r = 10 + min_ds + Lp;
    p.rw = (Lp + 86 + 3) & ~3;
    p.pwl = (p.tiles_x - 1) * kTileW + kBandLW;
    p.pwr = (p.tiles_x - 1) * kTileW + p.rw;
    return p;
}

// Per-chunk scratch in HBM (frame-major; one chunk = frames_per_launch frames).
//   gray  : [F][2][H][W]    float   (side 0 = left, 1 = right)
//   pool  : [F][2][Hd][Wd]  float
//   wta4  : [F][Hd][Wd]     float4  (d* relative as float, A[d*-1], max A, A[d*+1]) -- raw, see secondary.cu
//   edge2 : [F][Hd][Wd]     float2  (A[0], A[L-1])  for the circular wrap of d*-1 / d*+1
//   refined:[F][Hd][Wd]     float
struct Scratch {
    float *gray;
    float *pool;
    float4 *wta4;
    float2 *edge2;
    float *refined;
    float4 *wta4_parts;   // [split][frames][Hd*Wd] part slots of a level-split launch (small launches only), else NULL
    float2 *edge2_parts;  // [split][frames][Hd*Wd]
    int2 *part_range;     // [split][frames*tiles] first / last level each part evaluated (-1: empty part)
    float *agg_vol;  // [F][L][Hd*Wd] (plane-major) aggregated volume, only in reference-compat mode (abs_index), else NULL
    float *padl, *padr;  // [F][rows][pwl], [F][rows][pwr] wrap-padded pooled planes (PadGeom), NULL if unsupported
    // Certified level screen (mbm_screen.cu), all NULL when unsupported:
    unsigned *pass_mask;              // [F][tiles_y][tiles_x][4] bit m = the fused kernel must run level pair m of that tile
    float *dbg_screen;                // parity hook: the screen's approximate aggregated costs of frame 0, [Hd][Wd][L], or NULL
    unsigned *gather_mask;            // same shape: level pairs whose aggregated values the absolute-index reads of
                                      // secondary matching need (reference-compat mode behind the screen), else NULL
    int *tile_order;                  // [kScreenBuckets][F*tiles] tile ids bucketed by flagged-pair count (heaviest bucket last)
    int *bucket_count;                // [kScreenCtrlInts] tiles per bucket + per-chunk counters (zeroed before every screen launch)
    unsigned long long *screen_host_word;  // device alias of a mapped host word: per-chunk screen outcome, or NULL
    unsigned long long *screen_stats; // [2] {level pairs flagged, level pairs screened} since the last reset
    int *range_flag;                  // == range_epoch when some pooled value of the current chunk lies outside [0,255]
    int range_epoch;                  // (or is NaN): the screen's error bound does not hold, masks are ignored
};

// Where the GLOBAL left gray image lives in row-band mode (the vertical fill's colour row (K+1)*x can be anywhere in
// the image, upscale_disparity_vertical_fill.cu:31).  n == 0: one flat [H_glob][W] image `flat` (NULL = the handle's
// own image, normal mode).  n > 0: rank q holds rows row0[q] .. row0[q+1]-1 at band[q] (peer memory over NVLink).
struct GrayView {
    const float *flat;
    const float *band[8];
    int row0[9];
    int n;
};

// kernel launchers (each returns cudaGetLastError())
// mirrored > 0 (left-right check): the last `mirrored` of the `frames` frames are the mirrored pairs (flip R, flip L) of
// caller frames 0..mirrored-1, read from the same left / right input
cudaError_t launch_gray_pool(const Geom &g, const void *left, const void *right, int dtype, int frames,
                             const Scratch &s, cudaStream_t st, int mirrored = 0);
cudaError_t launch_pad_pooled(const Geom &g, int frames, const Scratch &s, cudaStream_t st);
cudaError_t launch_mbm_wta_generic(const Geom &g, int frames, const Scratch &s, float *dbg_cost,
                                   float *dbg_agg, cudaStream_t st);
bool mbm_wta_fast_supported(const Geom &g);
// use_screen: run only the level pairs flagged in s.pass_mask (written by launch_mbm_screen for the same chunk)
// gather: no WTA; evaluate the level pairs flagged in s.gather_mask and store their aggregated values into s.agg_vol
// in the compact per-tile layout (Geom::abs_index == 2)
// split > 1 (unscreened, no volumes): every tile's level pairs are spread over `split` blocks (part slots in
// s.wta4_parts / s.edge2_parts), then merged into s.wta4 / s.edge2 -- for launches too small to fill the GPU otherwise
cudaError_t launch_mbm_wta_fast(const Geom &g, int frames, const Scratch &s, float *dbg_cost,
                                float *dbg_agg, cudaStream_t st, bool use_screen = false, bool gather = false, int split = 1);
// marks in s.gather_mask (zeroed by the caller) the level pairs the absolute-index reads of secondary matching need
cudaError_t launch_abs_targets(const Geom &g, int frames, const Scratch &s, cudaStream_t st);
// floats per frame of the compact layout (>= Hd*Wd*L)
inline size_t compact_volume_floats(const Geom &g) {
    const PadGeom pg = make_pad_geom(g.Hd, g.Wd, g.L, g.min_ds);
    return (size_t)pg.tiles_x * pg.tiles_y * (((size_t)g.L + 1) / 2) * 2 * kTileH * kTileW;
}
bool mbm_screen_supported(const Geom &g);
cudaError_t launch_mbm_screen(const Geom &g, int frames, const Scratch &s, cudaStream_t st);
bool mbm_wta_ws_supported(const Geom &g);
cudaError_t launch_mbm_wta_ws(const Geom &g, int frames, const Scratch &s, cudaStream_t st);
cudaError_t launch_secondary(const Geom &g, int frames, const Scratch &s, cudaStream_t st);
cudaError_t launch_fill(const Geom &g, int frames, const Scratch &s, const GrayView &gv, float *out, cudaStream_t st);
// Left-right consistency check (api.cu sd_set_lr_check) as the epilogue of the fill: right_mirrored = [frames][H][W]
// disparity maps of the mirrored pairs (flip R, flip L); a left pixel keeps its value d only if d is finite, its partner
// column yr = c - rint(d) lies in [0, W) and |d - right_mirrored[r][W-1-yr]| <= tolerance, else it gets `invalid`.
struct LrCheck {
    const float *right_mirrored;
    float tolerance, invalid;
};
cudaError_t launch_fill_lr(const Geom &g, int frames, const Scratch &s, const GrayView &gv, float *out, const LrCheck &lr,
                           cudaStream_t st);
// Left-right check plus background fill (DESIGN.md §13) of `frames` [H][W] maps: `left` unchecked, `right` in right-image
// columns or, with right_mirrored, stored mirrored (partner at W-1-yr).  Each rejected pixel gets the smaller of the
// kept values that bound its run in the row (the one neighbour at a border); rows without a kept pixel copy the nearest
// non-empty row above the first / below the last one and otherwise stay `invalid`.  out may alias left (not right);
// row_kept: frames*H bytes of scratch.  Two launches: the row pass and the column pass.
cudaError_t launch_lr_background_fill(const float *left, const float *right, bool right_mirrored, int frames, int H, int W,
                                      float tolerance, float invalid, float *out, unsigned char *row_kept,
                                      cudaStream_t st);
// The row pass of launch_lr_background_fill alone (right map mirrored): the peer-memory row-band mode runs its column
// pass only after the fill-bounds exchange (launch_lr_fill_cols_band).
cudaError_t launch_lr_fill_rows(const float *left, const float *right_mirrored, int frames, int H, int W, float tolerance,
                                float invalid, float *out, unsigned char *row_kept, cudaStream_t st);
// Fill-bounds area of one rank and frame parity (peer-memory row bands with the background fill, DESIGN.md §8 / §13):
//   int [0] / [1]: first / last GLOBAL row of the rank's band that kept a pixel (-1: none), padded to 256 bytes;
//   then floats [W]: that first row after the row pass, and [W]: that last row.
constexpr int kFillAreaHeaderFloats = 64;
inline size_t fill_area_bytes(int W) { return ((size_t)kFillAreaHeaderFloats * 4 + 8 * (size_t)W + 255) & ~(size_t)255; }
struct FillAreas {
    const float *area[8];   // every rank's area of this frame's parity, in rank (= row) order
    int n;
};
// Column pass of the background fill on the band rows [row_first, row_first + band_rows) of one local window `out`
// (row_kept: the row pass's flags of the same window; glob_row0: global row of local row row_first): a row without a
// kept pixel copies the frame's first non-empty row when it lies above it, the last one when below it, read from the
// published copy of the rank that owns it.  Writes nothing outside the band.
cudaError_t launch_lr_fill_cols_band(float *out, const unsigned char *row_kept, int row_first, int band_rows, int glob_row0,
                                     int W, const FillAreas &areas, cudaStream_t st);
// Rectification remap (rectify.cu, DESIGN.md §14), exactly cv2.remap with CV_32FC1 maps, INTER_LINEAR and a constant 0
// border: dst[p][r][c] = src[p] sampled at (map_x[r][c], map_y[r][c]) for `planes` [H][W] planes per view, uint8 or
// float32 by `dtype`; grid.y runs over the n_views (1 or 2) views.  H, W < 32768; dst must not overlap src.
struct RectifyView {
    const float *map_x, *map_y;
    const void *src;
    void *dst;
};
struct RectifyViews {
    RectifyView view[2];
};
cudaError_t launch_rectify(const RectifyViews &v, int n_views, int dtype, int planes, int H, int W, cudaStream_t st);
// Reprojection to 3-D (reproject.cu, DESIGN.md §15), exactly cv2.reprojectImageTo3D: n float32 [H][W] disparity maps ->
// xyz [n][H][W][3] float32 with the 4x4 row-major Q.  min_key: n unsigned of scratch for handleMissingValues (one more
// launch plus a memset), NULL without it.  xyz must not overlap disp.
struct ReprojectQ {
    double q[16];
};
cudaError_t launch_reproject(const float *disp, int n, int H, int W, const ReprojectQ &Q, unsigned *min_key, float *xyz,
                             cudaStream_t st);
// peer-memory row-band exchange (band_p2p.cu)
cudaError_t launch_band_scatter(const void *left, const void *right, void *own_l, void *own_r, void *prev_l, void *prev_r,
                                void *next_l, void *next_r, int row_bytes, int band_rows, int halo, int own_rows, int prev_rows,
                                int next_rows, unsigned *counter, unsigned *flag_at_prev, unsigned *flag_at_next, unsigned epoch,
                                cudaStream_t st);
// `planes` planes of n_floats each: plane i from src + i * src_plane to dst + i * dst_plane (floats)
cudaError_t launch_publish_gray(const float *src, float *dst, size_t n_floats, unsigned *counter, unsigned *const *peer_flags,
                                int n_peers, unsigned epoch, cudaStream_t st, int planes = 1, size_t src_plane = 0,
                                size_t dst_plane = 0);
// Fill-bounds exchange: finds the first / last kept row among the band's `band_rows` row flags, copies those two filled
// rows of `rows` ([band_rows][W]) and their global rows (glob_row0 + index) into `area` (my fill area, layout above),
// then releases one flag at every peer.
cudaError_t launch_publish_fill_bounds(const unsigned char *row_kept, const float *rows, int band_rows, int glob_row0, int W,
                                       float *area, unsigned *counter, unsigned *const *peer_flags, int n_peers,
                                       unsigned epoch, cudaStream_t st);
cudaError_t launch_wait_flags(const unsigned *flags, int first, int count, unsigned epoch, unsigned long long *timeout_word,
                              cudaStream_t st);

}  // namespace sd
