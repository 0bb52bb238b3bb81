// C ABI of libstereo_b200.so (include/stereo_b200.h): handle, scratch, launch orchestration and
// the pipelined host-buffer entry point.  Replaces the reference's host class
// (src/csrc/depth/stereo_matching.cc:17-114) and its device_buffer (buffer/device_buffer.cc:3-12).
#include <stdio.h>
#include <string.h>

#include <stdlib.h>

#include <memory>
#include <new>
#include <utility>
#include <vector>

#include "common.cuh"

using namespace sd;

namespace {
constexpr int kSlots = 4;  // host pipeline depth (H2D / compute / D2H in flight)
constexpr double kScreenGiveUp = 0.70;  // evaluated fraction above which the screen costs more than it saves
constexpr double kScreenGiveUpGather = 0.40;  // the same in reference-compat mode, where a second (gather) pass of about the
                                              // same density follows and the alternative only adds the volume stores
constexpr int kScreenPause = 32;        // chunks without the screen before it is probed again
constexpr size_t kGuardBytes = 64 << 10;  // per side, debug guard bands
constexpr unsigned char kGuardPattern = 0xA5;
constexpr int kProfMarks = 7;  // start | gray+pool | plane padding | level screen | cost+agg+WTA | secondary | fill

// Base of the resource owners below: a copy would free the same resources twice.
struct NoCopy {
    NoCopy() = default;
    NoCopy(const NoCopy &) = delete;
    NoCopy &operator=(const NoCopy &) = delete;
};

// The handle's device scratch: every live allocation as (raw base, payload bytes); the destructor frees what is left.
// With debug guard bands (SD_DEBUG_GUARDS=1 at sd_create) every payload is bracketed by kGuardBytes of a known pattern;
// sd_check_guards counts the bytes a stray store has changed (stands in for compute-sanitizer).
struct DeviceAllocs : NoCopy {
    bool guards = false;
    std::vector<std::pair<char *, size_t>> live;
    ~DeviceAllocs() { for (const auto &a : live) cudaFree(a.first); }

    template <typename T>
    cudaError_t alloc(T **p, size_t bytes) {
        const size_t total = guards ? ((bytes + 255) & ~(size_t)255) + 2 * kGuardBytes : bytes;
        char *raw = nullptr;
        cudaError_t e = cudaMalloc((void **)&raw, total);
        if (e != cudaSuccess) return e;
        live.push_back(std::make_pair(raw, bytes));
        if (guards && (e = cudaMemset(raw, kGuardPattern, total)) != cudaSuccess) return e;
        *p = (T *)(raw + (guards ? kGuardBytes : 0));
        return cudaSuccess;
    }

    // frees the allocation whose payload is p and sets p to null (no-op for null)
    template <typename T>
    void release(T *&p) {
        for (size_t i = 0; p && i < live.size(); i++)
            if (live[i].first + (guards ? kGuardBytes : 0) == (char *)p) {
                cudaFree(live[i].first);
                live.erase(live.begin() + i);
                break;
            }
        p = nullptr;
    }
};

// Streams, per-slot events and device slots of the pipelined host path (sd_compute_host) for one input dtype.  Every
// member starts null and the destructor frees whatever was created, so a construction that fails partway leaks nothing.
struct HostPipeline : NoCopy {
    int dtype = -1;
    cudaStream_t st_h2d = nullptr, st_comp = nullptr, st_d2h = nullptr;
    void *din_l[kSlots] = {}, *din_r[kSlots] = {};
    float *dout[kSlots] = {};
    cudaEvent_t ev_h2d[kSlots] = {}, ev_comp[kSlots] = {}, ev_d2h[kSlots] = {};
    ~HostPipeline() {
        // (destroying a null event or stream would leave an error behind for the next cudaGetLastError)
        for (int i = 0; i < kSlots; i++) {
            cudaFree(din_l[i]);
            cudaFree(din_r[i]);
            cudaFree(dout[i]);
            for (cudaEvent_t e : {ev_h2d[i], ev_comp[i], ev_d2h[i]})
                if (e) cudaEventDestroy(e);
        }
        for (cudaStream_t s : {st_h2d, st_comp, st_d2h})
            if (s) cudaStreamDestroy(s);
    }
};

// A pinned host word mapped into the device's address space: kernels post to `dev`, the host reads `host`.
struct MappedWord : NoCopy {
    unsigned long long *host = nullptr, *dev = nullptr;
    ~MappedWord() { if (host) cudaFreeHost(host); }

    cudaError_t alloc() {
        cudaError_t e = cudaHostAlloc((void **)&host, sizeof(*host), cudaHostAllocMapped);
        if (e != cudaSuccess) {
            host = nullptr;
            return e;
        }
        *host = 0;
        if ((e = cudaHostGetDevicePointer((void **)&dev, host, 0)) != cudaSuccess) dev = nullptr;
        return e;
    }
};
}  // namespace

struct sd_handle {
    sd_config cfg = {};
    Geom g = {};
    int device = 0;
    int chunk = 0;         // frames per launch
    int variant = 0;       // 0 auto, 1 generic, 2 specialised, 3 warp-specialised
    bool auto_ws = false;  // variant 0 picks the warp-specialised schedule for this shape (sd_create's cost model)
    int sms = 0, per_sm_fast = 0;  // SM count and resident blocks per SM of the specialised kernel (launch cost models)
    bool screen = false;   // certified level screen in front of the specialised kernel (default on where supported)
    int epoch = 0;         // chunk counter, tags the out-of-range flag of the screen
    size_t parts_capacity = 0;  // pixels the part slots of a level-split launch can hold (Scratch::wta4_parts)
    bool split_off = false;     // sd_set_level_split(h, 0): never split (tuning / tests)
    int abs_mode = 0;      // layout of Scratch::agg_vol for the chunk in flight: 0 none, 1 whole volume, 2 compact (gather pass)
    // Adaptive policy: the screen only pays off when it removes work.  The last block of every screen launch posts
    // {chunk tag, pairs screened, pairs flagged} as one 64-bit store to mapped host memory (no copy, no wait); the
    // next chunks look at the latest word that has arrived: if the fused kernel still had to evaluate more than
    // kScreenGiveUp of the level pairs, the screen is skipped for kScreenPause chunks and then probed again.
    // Results never depend on this -- the screen only changes the run time.
    MappedWord stats;      // (its device alias is Scratch::screen_host_word)
    unsigned long long stats_seen = 0;
    int screen_pause = 0;
    DeviceAllocs allocs;   // owns every device buffer of `s`, rmap, lr_rows, rect_maps and rect_frames
    Scratch s = {};
    float *dbg_cost = nullptr, *dbg_agg = nullptr;
    GrayView gv = {};      // band mode: where the left gray of the global image lives, else all zero
    GrayView gv_mir = {};  // peer-memory band mode with the left-right check: the same for the mirrored frames' left gray
    // peer-memory row bands (sd_band_p2p_*): one exported allocation per rank =
    //   [window L | window R | gray 0 | gray 1 | flags | fill 0 | fill 1]
    // gray p holds one plane per frame of a call (two with the left-right check: forward, mirrored); the fill areas
    // (FillAreas in common.cuh) exist only with the background fill
    struct P2P : NoCopy {
        bool on = false, connected = false;
        int world = 0, rank = 0, dtype = 0, halo_rows = 0;
        int row0[9] = {};            // full-resolution first row of every rank's band (+ total height)
        size_t win_bytes = 0, gray_bytes = 0;  // per window / per published gray buffer (sized for the tallest band)
        size_t gray_plane_bytes = 0, fill_bytes = 0;  // per plane of a gray buffer / per fill area (0 without the fill)
        char *base = nullptr;        // my allocation
        char *peer[8] = {};          // every rank's allocation (peer[rank] == base)
        unsigned epoch = 0;
        MappedWord timeout;          // a wait kernel posts {epoch, flag} here when a peer never shows up
        ~P2P() { close(); }
        void close() {   // unmaps the peers' allocations and frees my own
            for (int q = 0; q < world; q++)
                if (q != rank && peer[q]) cudaIpcCloseMemHandle(peer[q]);
            cudaFree(base);
            base = nullptr;
        }
    } p2p;
    std::unique_ptr<HostPipeline> host;   // lazily created by sd_compute_host
    // scratch is shared by every call on this handle: each call's stream first waits for the previous call's work
    cudaEvent_t ev_last = nullptr;
    bool ev_last_valid = false;
    // optional per-kernel timing (sd_profile_enable): kProfMarks events per chunk on the launching stream
    bool prof = false;
    std::vector<cudaEvent_t> prof_events;
    // left-right consistency check (sd_set_lr_check): a chunk holds chunk/2 frame PAIRS, each run forward and mirrored
    bool lr = false;
    float lr_tol = 0.f, lr_invalid = 0.f;
    float *rmap = nullptr;       // [chunk/2][H][W] right views' disparity maps of the last chunk, in mirrored orientation
    bool lr_fill = false;        // background fill of the rejected pixels (sd_set_lr_fill)
    unsigned char *lr_rows = nullptr;   // [chunk/2][H] per row: 1 if the check kept a pixel of it (the fill's column pass)
    // rectification (sd_set_rectification): both NULL while it is off
    float *rect_maps = nullptr;  // [4][H][W] left map_x, left map_y, right map_x, right map_y
    char *rect_frames = nullptr; // [2 views][chunk][3][H][W] rectified frames of the chunk in flight, uint8 or float32
    char err[640] = {};
    int last_cuda = 0;

    // (the members' destructors free the rest; sd_destroy runs this on the handle's device)
    ~sd_handle() {
        for (cudaEvent_t e : prof_events) cudaEventDestroy(e);
        if (ev_last) cudaEventDestroy(ev_last);
    }
};

namespace {

int fail(sd_handle *h, int code, const char *msg) {
    if (h) snprintf(h->err, sizeof(h->err), "%s", msg);
    return code;
}

int fail_cuda(sd_handle *h, cudaError_t e, const char *where) {
    if (h) {
        h->last_cuda = (int)e;
        snprintf(h->err, sizeof(h->err), "CUDA error at %s: %s (%d)", where, cudaGetErrorString(e), (int)e);
    }
    return SD_ERR_CUDA;
}

#define SD_CUDA(h, call)                                        \
    do {                                                        \
        cudaError_t e__ = (call);                               \
        if (e__ != cudaSuccess) return fail_cuda(h, e__, #call); \
    } while (0)

struct DeviceGuard {
    int prev;
    bool ok;
    explicit DeviceGuard(int dev) : prev(-1), ok(false) {
        if (cudaGetDevice(&prev) != cudaSuccess) return;
        ok = (prev == dev) || (cudaSetDevice(dev) == cudaSuccess);
    }
    ~DeviceGuard() {
        int cur = -1;
        if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
    }
};

const char *validate(const sd_config *c) {
    if (c->height <= 0 || c->width <= 0) return "height and width must be positive";
    if (c->downscale_factor <= 0) return "downscale_factor must be positive";
    if (c->min_disparity < 0) return "min_disparity must be >= 0";
    if (c->max_disparity < c->min_disparity) return "max_disparity must be >= min_disparity";
    if (c->ncc_patch_radius < 0 || c->sad_patch_radius < 0) return "patch radii must be >= 0";
    if (c->small_mbm_radius < 0 || c->mid_mbm_radius < 0 || c->large_mbm_radius < 0) return "mbm radii must be >= 0";
    if (c->small_mbm_radius > c->large_mbm_radius || c->mid_mbm_radius > c->large_mbm_radius)
        return "small/mid mbm radius must not exceed large_mbm_radius (the reference's tile only covers the large radius)";
    if (c->threshold < 0) return "threshold must be >= 0";
    return nullptr;
}

size_t in_bytes_per_frame(const sd_handle *h, int dtype) {
    return (size_t)3 * h->g.H * h->g.W * (dtype == SD_U8 ? 1 : 4);
}

__global__ void extract_wta(const float4 *__restrict__ w, float *__restrict__ dst, int n, float min_ds) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = __fadd_rn(w[i].x, min_ds);
}

// right view's map in right-image orientation from the mirrored one
__global__ void unmirror_rows(const float *__restrict__ src, float *__restrict__ dst, int H, int W) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
    if (c < W && r < H) dst[(size_t)r * W + c] = src[(size_t)r * W + (W - 1 - c)];
}

__global__ void extract_agg3(const float4 *__restrict__ w, const float2 *__restrict__ e, float *__restrict__ dst, int n,
                             int L) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 v = w[i];
    const float2 ed = e[i];
    const int bd = (int)v.x;
    dst[3 * i + 0] = (bd == 0) ? ed.y : v.y;
    dst[3 * i + 1] = (bd == 0) ? ed.x : v.z;
    dst[3 * i + 2] = (bd == L - 1) ? ed.x : v.w;
}

// Orders this call after the previous call on the same handle (possibly on another stream): they share scratch.
int order_after_previous(sd_handle *h, cudaStream_t st) {
    if (h->ev_last_valid) SD_CUDA(h, cudaStreamWaitEvent(st, h->ev_last, 0));
    return SD_OK;
}

int mark_last_use(sd_handle *h, cudaStream_t st) {
    SD_CUDA(h, cudaEventRecord(h->ev_last, st));
    h->ev_last_valid = true;
    return SD_OK;
}

int prof_mark(sd_handle *h, cudaStream_t st) {
    if (!h->prof) return SD_OK;
    cudaEvent_t e;
    SD_CUDA(h, cudaEventCreate(&e));
    h->prof_events.push_back(e);
    SD_CUDA(h, cudaEventRecord(e, st));
    return SD_OK;
}

// The level screen runs in front of the specialised kernel only: not with debug volumes (they need every level) and not
// with an explicitly selected generic or warp-specialised variant.  In reference-compat mode (absolute-index reads,
// Scratch::agg_vol) the screen stays on: instead of the whole volume, a gather pass then evaluates just the level pairs
// those reads ask for (Geom::abs_index == 2, see run_chunk).
bool screen_allowed(const sd_handle *h) {
    return h->screen && h->s.pass_mask && h->s.padl && (h->variant == 0 || h->variant == 2) && !h->dbg_cost &&
           !h->dbg_agg && (!h->s.agg_vol || h->s.gather_mask) && mbm_screen_supported(h->g);
}

// LEVEL SPLIT of the unscreened specialised kernel for launches that do not fill the GPU (single frames, thin row
// bands): a tile's L/2 level pairs go to `split` blocks, so a launch of T tiles has T*split blocks of L/(2 split)
// passes each instead of T blocks of L/2.  Cost model in pass-times of one block: rounds * (passes + ~1.5 for staging
// the bands and the part records).  Returns the best split (1 = off) and its cost.
constexpr int kMaxSplit = 16;
constexpr double kSplitOverhead = 1.5;
int plan_split(const sd_handle *h, int frames, bool need_buffers, double *cost_out) {
    const Geom &g = h->g;
    const int M = ((g.L + 1) & ~1) / 2;
    const long long tiles = (long long)((g.Wd + kTileW - 1) / kTileW) * ((g.Hd + kTileH - 1) / kTileH) * frames;
    const long long slots = (long long)h->sms * h->per_sm_fast;
    auto cost = [&](int S) { return (double)((tiles * S + slots - 1) / slots) * ((M + S - 1) / S + kSplitOverhead); };
    int best = 1;
    double best_cost = cost(1);
    const bool can = mbm_wta_fast_supported(g) && !h->dbg_cost && !h->dbg_agg && !h->s.agg_vol && (!need_buffers || h->s.wta4_parts);
    for (int S = 2; can && S <= kMaxSplit && S <= M; S++) {
        if (need_buffers && (size_t)S * frames * g.Hd * g.Wd > h->parts_capacity) break;
        if (cost(S) < 0.9 * best_cost && cost(S) < 0.9 * cost(1)) {
            best = S;
            best_cost = cost(S);
        }
    }
    if (cost_out) *cost_out = best_cost;
    return best;
}

// Level split behind the screen: a launch cannot finish before its heaviest tile has, and a tile that keeps all its level
// pairs costs as much as an unscreened one.  With fewer than about four waves of tiles every tile's flagged pairs are
// therefore spread over several blocks (by rank; mbm_wta_fast.cu), heaviest tiles first.
int screened_split(const sd_handle *h, int frames) {
    if (h->split_off || !h->s.wta4_parts) return 1;
    const PadGeom pg = make_pad_geom(h->g.Hd, h->g.Wd, h->g.L, h->g.min_ds);
    const long long tiles = (long long)pg.tiles_x * pg.tiles_y * frames, slots = (long long)h->sms * h->per_sm_fast;
    if (tiles >= 4 * slots) return 1;
    int S = (int)((4 * slots + tiles - 1) / tiles);
    const int M = ((h->g.L + 1) & ~1) / 2;
    if (S > 8) S = 8;
    if (S > M) S = M;
    while (S > 1 && (size_t)S * frames * h->g.Hd * h->g.Wd > h->parts_capacity) S--;
    return S < 1 ? 1 : S;
}

// Does the screen pay for a launch of `frames` frames?  Model in units of one full (unscreened) tile: unscreened = waves;
// screened = screen kernel (0.175 tile-times per tile and SM, at least one tile's worth) + exact kernel
// max(heaviest tile / split, 25 % of the work spread over all slots).  With variant 0 only; an explicit variant 2 always
// screens (tests, tuning).
bool screen_pays(const sd_handle *h, int frames) {
    if (h->variant == 2) return true;
    const PadGeom pg = make_pad_geom(h->g.Hd, h->g.Wd, h->g.L, h->g.min_ds);
    const double tiles = (double)pg.tiles_x * pg.tiles_y * frames, sms = h->sms, slots = (double)h->sms * h->per_sm_fast;
    // best unscreened alternative: the split two-phase kernel (plan_split) or whole waves
    double unscreened = (double)(long long)((tiles + slots - 1) / slots);
    {
        const int M = ((h->g.L + 1) & ~1) / 2;
        double c = 0.0;
        if (plan_split(h, frames, true, &c) > 1 && c / (M + kSplitOverhead) < unscreened) unscreened = c / (M + kSplitOverhead);
    }
    const double heavy = 1.0 / screened_split(h, frames) + 0.05;
    const double spread = 0.25 * tiles / slots;
    const double screen_kernel = tiles * 0.175 / sms > 0.175 ? tiles * 0.175 / sms : 0.175;
    return screen_kernel + (spread > heavy ? spread : heavy) < 0.95 * unscreened;
}

bool screen_active(const sd_handle *h, int frames) { return screen_allowed(h) && screen_pays(h, frames); }

// 1 generic, 2 specialised, 3 warp-specialised -- for a launch of `frames` frames
int active_variant(const sd_handle *h, int frames) {
    const bool fast = h->s.padl && ((h->variant >= 2) || (h->variant == 0 && mbm_wta_fast_supported(h->g)));
    bool ws = (h->variant == 3 || (h->variant == 0 && h->auto_ws && !screen_active(h, frames))) && h->s.padl &&
              !h->dbg_cost && !h->dbg_agg && mbm_wta_ws_supported(h->g);
    if (ws && h->variant == 0) {
        // the warp-specialised schedule (64x64 tiles, one block per SM, ~0.96 of the two-phase pass time) has no level
        // split: for small launches the split two-phase kernel can be the faster one
        const Geom &g = h->g;
        const long long tiles_ws = (long long)((g.Wd + kTileW - 1) / kTileW) * ((g.Hd + 63) / 64) * frames;
        const double cost_ws = (double)((tiles_ws + h->sms - 1) / h->sms) * (((g.L + 1) & ~1) / 2 + kSplitOverhead) * 0.96;
        double cost_split = 0.0;
        if (plan_split(h, frames, true, &cost_split) > 1 && cost_split < 0.9 * cost_ws) ws = false;
    }
    return ws ? 3 : (fast ? 2 : 1);
}

// level split of the next launch of `frames` frames (1 = off): only for the unscreened specialised kernel
int active_split(const sd_handle *h, int frames) {
    if (h->split_off || active_variant(h, frames) != 2) return 1;
    if (screen_active(h, frames)) return h->s.agg_vol ? 1 : screened_split(h, frames);   // (not in reference-compat mode)
    return plan_split(h, frames, true, nullptr);
}

// Frames per launch of the left-right check: every launch runs a pair's forward and mirrored frame
inline int lr_pairs(const sd_handle *h) { return h->chunk / 2 > 0 ? h->chunk / 2 : 1; }

// With the left-right check on, `frames` counts PAIRS: kernels A..C run over 2*frames frames (forward 0..frames-1, then
// the mirrored pairs), the fill writes the mirrored frames' maps into h->rmap and then the forward frames into `out`,
// checked against them (with the background fill: unchecked, then checked and filled in place by two more launches).
int run_chunk(sd_handle *h, const void *left, const void *right, int dtype, int pairs, float *out, cudaStream_t st,
              int k0 = 0, int k1 = 3) {
    int rc;
    const bool full = (k0 == 0 && k1 == 3);  // per-kernel profiling only brackets complete passes
    const int frames = h->lr ? 2 * pairs : pairs;
    if (full && (rc = prof_mark(h, st)) != SD_OK) return rc;
    if (k0 <= 0 && 0 <= k1) {
        if (h->rect_maps) {   // raw input: remap the chunk's caller frames (once, also with the check) into rect_frames
            const size_t n = (size_t)h->g.H * h->g.W, view_bytes = (size_t)h->chunk * 3 * n * (dtype == SD_U8 ? 1 : 4);
            RectifyViews v;
            v.view[0] = RectifyView{h->rect_maps, h->rect_maps + n, left, h->rect_frames};
            v.view[1] = RectifyView{h->rect_maps + 2 * n, h->rect_maps + 3 * n, right, h->rect_frames + view_bytes};
            SD_CUDA(h, launch_rectify(v, 2, dtype, 3 * pairs, h->g.H, h->g.W, st));
            left = v.view[0].dst;
            right = v.view[1].dst;
        }
        SD_CUDA(h, launch_gray_pool(h->g, left, right, dtype, frames, h->s, st, h->lr ? pairs : 0));
    }
    if (full && (rc = prof_mark(h, st)) != SD_OK) return rc;
    if (k0 <= 1 && 1 <= k1) {
        h->s.range_epoch = ++h->epoch;
        const int v = active_variant(h, frames);
        bool screen = (v == 2) && screen_active(h, frames);
        if (screen && h->stats.host) {
            const unsigned long long w = *(volatile unsigned long long *)h->stats.host;   // [tag:16][screened:24][flagged:24]
            if (w != h->stats_seen) {
                const double flagged = (double)(w & 0xffffffull), screened = (double)((w >> 24) & 0xffffffull);
                const double give_up = h->s.agg_vol ? kScreenGiveUpGather : kScreenGiveUp;
                if (screened > 0 && flagged > give_up * screened) h->screen_pause = kScreenPause;
                h->stats_seen = w;
            }
            if (h->screen_pause > 0) {
                h->screen_pause--;
                screen = false;
            }
        }
        // Reference-compat mode (min_disparity/K != 0): secondary matching reads the aggregated volume at ABSOLUTE
        // indices.  Without the screen the fused kernel evaluates every level anyway and stores the whole volume
        // (abs_index 1).  Behind the screen it does not: WTA first (no store), then a gather pass of the same kernel over
        // exactly the level pairs those reads will touch, into a compact per-tile volume (abs_index 2).
        const bool gather = screen && h->s.agg_vol != nullptr;
        h->abs_mode = h->s.agg_vol ? (gather ? 2 : 1) : 0;
        if (v == 2) SD_CUDA(h, launch_pad_pooled(h->g, frames, h->s, st));
        if (full && (rc = prof_mark(h, st)) != SD_OK) return rc;
        if (screen) SD_CUDA(h, launch_mbm_screen(h->g, frames, h->s, st));
        if (full && (rc = prof_mark(h, st)) != SD_OK) return rc;
        if (v == 3) SD_CUDA(h, launch_mbm_wta_ws(h->g, frames, h->s, st));   // (pads its planes itself)
        else if (v == 2 && gather) {
            Scratch wta_only = h->s;
            wta_only.agg_vol = nullptr;
            SD_CUDA(h, launch_mbm_wta_fast(h->g, frames, wta_only, nullptr, nullptr, st, true));
            SD_CUDA(h, launch_abs_targets(h->g, frames, h->s, st));
            SD_CUDA(h, launch_mbm_wta_fast(h->g, frames, h->s, nullptr, nullptr, st, false, true));
        } else if (v == 2) {
            // (a paused screen falls back to the unscreened plan for this launch)
            const int split = h->split_off ? 1 : (screen ? (h->s.agg_vol ? 1 : screened_split(h, frames))
                                                          : plan_split(h, frames, true, nullptr));
            SD_CUDA(h, launch_mbm_wta_fast(h->g, frames, h->s, h->dbg_cost, h->dbg_agg, st, screen, false, split));
        }
        else SD_CUDA(h, launch_mbm_wta_generic(h->g, frames, h->s, h->dbg_cost, h->dbg_agg, st));
    }
    if (full && (rc = prof_mark(h, st)) != SD_OK) return rc;
    if (k0 <= 2 && 2 <= k1) {
        Geom g2 = h->g;
        g2.abs_index = h->abs_mode;   // which layout Scratch::agg_vol holds for THIS chunk
        SD_CUDA(h, launch_secondary(g2, frames, h->s, st));
    }
    if (full && (rc = prof_mark(h, st)) != SD_OK) return rc;
    if (k0 <= 3 && 3 <= k1 && !h->lr) SD_CUDA(h, launch_fill(h->g, frames, h->s, h->gv, out, st));
    if (k0 <= 3 && 3 <= k1 && h->lr) {
        const size_t n = (size_t)h->g.H * h->g.W, nd = (size_t)h->g.Hd * h->g.Wd;
        Scratch mirrored = h->s;   // the fill of frames pairs..2*pairs-1
        mirrored.gray += (size_t)pairs * 2 * n;
        mirrored.refined += (size_t)pairs * nd;
        // (peer-memory row bands: the mirrored frame's colour rows come from the ranks' published mirrored gray bands)
        SD_CUDA(h, launch_fill(h->g, pairs, mirrored, h->gv.n > 0 ? h->gv_mir : h->gv, h->rmap, st));
        if (h->lr_fill) {   // unchecked left maps, then the check and the background fill in place
            SD_CUDA(h, launch_fill(h->g, pairs, h->s, h->gv, out, st));
            if (h->gv.n == 0)
                SD_CUDA(h, launch_lr_background_fill(out, h->rmap, true, pairs, h->g.H, h->g.W, h->lr_tol, h->lr_invalid,
                                                     out, h->lr_rows, st));
            else   // peer-memory row bands: the column pass follows the fill-bounds exchange (sd_band_p2p_compute)
                SD_CUDA(h, launch_lr_fill_rows(out, h->rmap, pairs, h->g.H, h->g.W, h->lr_tol, h->lr_invalid, out,
                                               h->lr_rows, st));
        } else {
            SD_CUDA(h, launch_fill_lr(h->g, pairs, h->s, h->gv, out, LrCheck{h->rmap, h->lr_tol, h->lr_invalid}, st));
        }
    }
    if (full && (rc = prof_mark(h, st)) != SD_OK) return rc;
    return SD_OK;
}

// Frames per chunk of the pipelined host path: copies of a chunk cannot overlap its own kernels, so the host path uses
// chunks of at most kHostChunk frames whatever the device path's chunk is.
constexpr int kHostChunk = 8;
int host_chunk(const sd_handle *h) { return h->chunk < kHostChunk ? h->chunk : kHostChunk; }

// frames (pairs with the left-right check) per host-path chunk: the slots hold host_chunk frames, scratch 2 * pairs
int host_chunk_frames(const sd_handle *h) {
    const int hc = host_chunk(h);
    return (h->lr && lr_pairs(h) < hc) ? lr_pairs(h) : hc;
}

int ensure_host_pipeline(sd_handle *h, int dtype) {
    if (h->host && h->host->dtype == dtype) return SD_OK;
    h->host.reset();
    std::unique_ptr<HostPipeline> p(new (std::nothrow) HostPipeline());
    if (!p) return fail(h, SD_ERR_NOMEM, "out of host memory");
    const size_t inb = in_bytes_per_frame(h, dtype) * host_chunk(h);
    const size_t outb = (size_t)h->g.H * h->g.W * sizeof(float) * host_chunk(h);
    SD_CUDA(h, cudaStreamCreateWithFlags(&p->st_h2d, cudaStreamNonBlocking));
    SD_CUDA(h, cudaStreamCreateWithFlags(&p->st_comp, cudaStreamNonBlocking));
    SD_CUDA(h, cudaStreamCreateWithFlags(&p->st_d2h, cudaStreamNonBlocking));
    for (int i = 0; i < kSlots; i++) {
        SD_CUDA(h, cudaMalloc(&p->din_l[i], inb));
        SD_CUDA(h, cudaMalloc(&p->din_r[i], inb));
        SD_CUDA(h, cudaMalloc((void **)&p->dout[i], outb));
        SD_CUDA(h, cudaEventCreateWithFlags(&p->ev_h2d[i], cudaEventDisableTiming));
        SD_CUDA(h, cudaEventCreateWithFlags(&p->ev_comp[i], cudaEventDisableTiming));
        SD_CUDA(h, cudaEventCreateWithFlags(&p->ev_d2h[i], cudaEventDisableTiming));
    }
    p->dtype = dtype;
    h->host = std::move(p);
    return SD_OK;
}

}  // namespace

extern "C" {

int sd_set_compat(sd_handle *h, int on);

int sd_abi_version(void) { return SD_ABI_VERSION; }

int sd_config_default(sd_config *cfg) {
    if (!cfg) return SD_ERR_BAD_ARG;
    const sd_config d = {1080, 1920, 2, 75, 262, 1, 5, 5, 1, 4, 10};
    *cfg = d;
    return SD_OK;
}

int sd_dims(const sd_config *c, int32_t *Hd, int32_t *Wd, int32_t *L) {
    if (!c || validate(c)) return SD_ERR_BAD_ARG;
    const int K = c->downscale_factor;
    if (Hd) *Hd = (c->height + K - 1) / K;
    if (Wd) *Wd = (c->width + K - 1) / K;
    if (L) *L = c->max_disparity / K - c->min_disparity / K + 1;
    return SD_OK;
}

int sd_create(const sd_config *cfg, int device, int frames_per_launch, sd_handle **out) {
    if (!cfg || !out) return SD_ERR_BAD_ARG;
    *out = nullptr;
    sd_handle *h = new (std::nothrow) sd_handle();
    if (!h) return SD_ERR_NOMEM;
    *out = h;  // returned even on failure so the caller can read sd_last_error, then sd_destroy
    {
        const char *e = getenv("SD_DEBUG_GUARDS");
        h->allocs.guards = e && atoi(e) != 0;
    }
    h->cfg = *cfg;
    h->device = device;
    if (const char *why = validate(cfg)) return fail(h, SD_ERR_BAD_ARG, why);
    Geom &g = h->g;
    g.H = cfg->height;
    g.W = cfg->width;
    g.K = cfg->downscale_factor;
    sd_dims(cfg, &g.Hd, &g.Wd, &g.L);
    g.min_ds = cfg->min_disparity / g.K;
    g.r_cost = cfg->ncc_patch_radius;
    g.r_sad = cfg->sad_patch_radius;
    g.rs = cfg->small_mbm_radius;
    g.rm = cfg->mid_mbm_radius;
    g.rl = cfg->large_mbm_radius;
    g.threshold = (float)cfg->threshold;
    g.band_x_off = 0;
    g.Hd_glob = g.Hd;
    g.H_glob = g.H;
    int ndev = 0;
    SD_CUDA(h, cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(h, SD_ERR_BAD_ARG, "no such CUDA device");
    // Cost model of the fused kernel, in SM-time per frame: a launch of F frames runs ceil(tiles*F / slots) waves;
    // a wave costs (tiles per SM) * (tile pixels) / (measured efficiency of the variant on a full wave).
    //   specialised kernel : 32x64 tiles, 2 per SM, 0.86     warp-specialised kernel: 64x64 tiles, 1 per SM, 0.895
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    const PadGeom pgq = make_pad_geom(g.Hd, g.Wd, g.L, g.min_ds);
    const size_t smem_b = (size_t)(kTileH + 20) * 42 * 16 + (size_t)kBandRows * (kBandLW + pgq.rw) * 4;
    const int per_sm_fast = (2 * (smem_b + 1024) <= 227 * 1024) ? 2 : 1;
    h->sms = sms;
    h->per_sm_fast = per_sm_fast;
    const long long tiles_x = (g.Wd + kTileW - 1) / kTileW;
    const long long tiles_fast = tiles_x * ((g.Hd + 31) / 32), tiles_ws = tiles_x * ((g.Hd + 63) / 64);
    // scratch bytes per frame of a chunk (gray, pooled, records, padded planes; + the aggregated volume in reference-compat mode)
    const size_t per_frame = (size_t)g.H * g.W * 4 * 2 + (size_t)g.Hd * g.Wd * 60 + (g.min_ds != 0 ? (size_t)g.Hd * g.Wd * g.L * 4 : 0);
    auto cost = [&](bool ws, int f) {
        const long long slots = (long long)sms * (ws ? 1 : per_sm_fast);
        const long long waves = ((ws ? tiles_ws : tiles_fast) * f + slots - 1) / slots;
        const double wave = ws ? 4096.0 / 0.895 : per_sm_fast * 2048.0 / (per_sm_fast == 2 ? 0.86 : 0.80);
        return (double)waves * wave / f;
    };
    const bool ws_ok = mbm_wta_fast_supported(g) && mbm_wta_ws_supported(g);
    double best_cost = 1e300;
    int best_f = 1;
    bool best_ws = false;
    for (int v = 0; v < (ws_ok ? 2 : 1); v++)
        for (int f = 1; f <= 32; f++) {   // (larger launches amortise the tail of the screened kernels: 5 560 -> 5 700 frames/s at C3 from 15 to 32)
            if (frames_per_launch > 0 && f != frames_per_launch) continue;
            if (frames_per_launch <= 0 && f > 1 && (size_t)f * per_frame > ((size_t)4 << 30)) break;
            const double c = cost(v == 1, f);
            if (c < best_cost * 0.995 || (c <= best_cost * 1.0001 && (v == 1) == best_ws)) {  // near-ties: larger chunk
                if (c < best_cost) best_cost = c;
                best_f = f;
                best_ws = (v == 1);
            }
        }
    if (frames_per_launch <= 0) frames_per_launch = best_f;
    h->auto_ws = best_ws;
    h->chunk = frames_per_launch;

    DeviceGuard dg(device);
    if (!dg.ok) return fail(h, SD_ERR_CUDA, "cudaSetDevice failed");
    SD_CUDA(h, cudaEventCreateWithFlags(&h->ev_last, cudaEventDisableTiming));
    const size_t F = h->chunk, n = (size_t)g.H * g.W, nd = (size_t)g.Hd * g.Wd;
    SD_CUDA(h, h->allocs.alloc(&h->s.gray, F * 2 * n * sizeof(float)));
    SD_CUDA(h, h->allocs.alloc(&h->s.pool, F * 2 * nd * sizeof(float)));
    SD_CUDA(h, h->allocs.alloc(&h->s.wta4, F * nd * sizeof(float4)));
    SD_CUDA(h, h->allocs.alloc(&h->s.edge2, F * nd * sizeof(float2)));
    SD_CUDA(h, h->allocs.alloc(&h->s.refined, F * nd * sizeof(float)));
    if (mbm_wta_fast_supported(g)) {
        const PadGeom pg = make_pad_geom(g.Hd, g.Wd, g.L, g.min_ds);
        SD_CUDA(h, h->allocs.alloc(&h->s.padl, F * (size_t)pg.rows * pg.pwl * sizeof(float)));
        SD_CUDA(h, h->allocs.alloc(&h->s.padr, F * (size_t)pg.rows * pg.pwr * sizeof(float)));
        SD_CUDA(h, h->allocs.alloc(&h->s.range_flag, sizeof(int)));
        SD_CUDA(h, cudaMemset(h->s.range_flag, 0, sizeof(int)));
        {   // part slots for level-split launches: sized for the largest split any launch size of this handle would pick
            // (unscreened: plan_split; behind the screen: up to 8 parts while the launch has fewer than four waves of tiles)
            const long long slots = (long long)h->sms * h->per_sm_fast;
            const long long tiles1 = (long long)pg.tiles_x * pg.tiles_y;
            size_t need = 0;
            int max_split = 1;
            for (int f = 1; f <= h->chunk; f++) {
                int S = plan_split(h, f, false, nullptr);
                if (mbm_screen_supported(g) && tiles1 * f < 4 * slots) {
                    int Ss = (int)((4 * slots + tiles1 * f - 1) / (tiles1 * f));
                    Ss = Ss > 8 ? 8 : Ss;
                    if (Ss > S) S = Ss;
                }
                if (S > max_split) max_split = S;
                if (S > 1 && (size_t)S * f * nd > need) need = (size_t)S * f * nd;
            }
            if (need > 0 && need * (sizeof(float4) + sizeof(float2)) <= ((size_t)1 << 30)) {
                SD_CUDA(h, h->allocs.alloc(&h->s.wta4_parts, need * sizeof(float4)));
                SD_CUDA(h, h->allocs.alloc(&h->s.edge2_parts, need * sizeof(float2)));
                SD_CUDA(h, h->allocs.alloc(&h->s.part_range, (size_t)kMaxSplit * F * tiles1 * sizeof(int2)));
                h->parts_capacity = need;
            }
        }
        if (mbm_screen_supported(g)) {
            SD_CUDA(h, h->allocs.alloc(&h->s.pass_mask, F * (size_t)pg.tiles_x * pg.tiles_y * 4 * sizeof(unsigned)));
            SD_CUDA(h, h->allocs.alloc(&h->s.gather_mask, F * (size_t)pg.tiles_x * pg.tiles_y * 4 * sizeof(unsigned)));
            SD_CUDA(h, h->allocs.alloc(&h->s.tile_order, F * (size_t)pg.tiles_x * pg.tiles_y * kScreenBuckets * sizeof(int)));
            SD_CUDA(h, h->allocs.alloc(&h->s.bucket_count, kScreenCtrlInts * sizeof(int)));
            SD_CUDA(h, h->allocs.alloc(&h->s.screen_stats, 2 * sizeof(unsigned long long)));
            SD_CUDA(h, cudaMemset(h->s.screen_stats, 0, 2 * sizeof(unsigned long long)));
            SD_CUDA(h, h->stats.alloc());
            h->s.screen_host_word = h->stats.dev;
            h->screen = true;
        }
    }
    // The reference indexes the aggregated volume with the absolute disparity (secondary_matching.cu:28-31);
    // with min_disparity/K != 0 that differs from the relative index, so reproduce it by default.
    if (g.min_ds != 0) return sd_set_compat(h, 1);
    return SD_OK;
}

int sd_set_compat(sd_handle *h, int on) {
    if (!h) return SD_ERR_BAD_ARG;
    DeviceGuard dg(h->device);
    if (!dg.ok) return fail(h, SD_ERR_CUDA, "cudaSetDevice failed");
    if (on && !h->s.agg_vol) {
        // sized for both layouts: the whole volume [L][Hd*Wd] and the compact per-tile one of the gather pass
        size_t per_frame = (size_t)h->g.Hd * h->g.Wd * h->g.L;
        if (h->s.gather_mask && compact_volume_floats(h->g) > per_frame) per_frame = compact_volume_floats(h->g);
        SD_CUDA(h, h->allocs.alloc(&h->s.agg_vol, (size_t)h->chunk * per_frame * sizeof(float)));
    } else if (!on) {
        h->allocs.release(h->s.agg_vol);
    }
    h->g.abs_index = on ? 1 : 0;
    return SD_OK;
}

int sd_check_guards(sd_handle *h, long long *corrupted_bytes);

int sd_destroy(sd_handle *h) {
    if (!h) return SD_OK;
    if (h->allocs.guards && !h->allocs.live.empty()) {
        // debug handles (SD_DEBUG_GUARDS=1) check their guard bands one last time: a whole test run can be soaked this way
        long long bad = 0;
        if (sd_check_guards(h, &bad) == SD_OK && bad != 0)
            fprintf(stderr, "libstereo_b200: GUARD BANDS CORRUPTED: %lld bytes around the scratch of a %dx%d handle\n", bad, h->g.H, h->g.W);
    }
    DeviceGuard dg(h->device);
    delete h;
    return SD_OK;
}

int sd_compute(sd_handle *h, const void *left, const void *right, int dtype, int n_frames, float *out, void *stream) {
    if (!h) return SD_ERR_BAD_ARG;
    if (!left || !right || !out) return fail(h, SD_ERR_BAD_ARG, "null image pointer");
    if (dtype != SD_U8 && dtype != SD_F32) return fail(h, SD_ERR_SHAPE, "dtype must be SD_U8 or SD_F32");
    if (n_frames <= 0) return fail(h, SD_ERR_SHAPE, "n_frames must be positive");
    DeviceGuard dg(h->device);
    if (!dg.ok) return fail(h, SD_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t st = (cudaStream_t)stream;
    int rc = order_after_previous(h, st);
    if (rc != SD_OK) return rc;
    const size_t inb = in_bytes_per_frame(h, dtype), outn = (size_t)h->g.H * h->g.W;
    // Launches of (nearly) equal size rather than full chunks plus a short remainder: behind the level screen a short
    // launch is dominated by its heaviest tiles.  (With the left-right check a chunk holds chunk/2 pairs.)
    const int per = h->lr ? lr_pairs(h) : h->chunk;
    const int nchunks = (n_frames + per - 1) / per, base = n_frames / nchunks, extra = n_frames % nchunks;
    for (int c = 0, f0 = 0; c < nchunks; c++) {
        const int nf = base + (c < extra ? 1 : 0);
        rc = run_chunk(h, (const char *)left + inb * f0, (const char *)right + inb * f0, dtype, nf, out + outn * f0, st);
        if (rc != SD_OK) return rc;
        f0 += nf;
    }
    return mark_last_use(h, st);
}

int sd_compute_range(sd_handle *h, const void *left, const void *right, int dtype, int n_frames, float *out,
                     void *stream, int first_kernel, int last_kernel) {
    if (!h) return SD_ERR_BAD_ARG;
    if (first_kernel < 0 || last_kernel > 3 || first_kernel > last_kernel) return fail(h, SD_ERR_BAD_ARG, "kernel range must be within [0,3]");
    if (first_kernel == 0 && (!left || !right)) return fail(h, SD_ERR_BAD_ARG, "null image pointer");
    if (last_kernel == 3 && !out) return fail(h, SD_ERR_BAD_ARG, "null output pointer");
    if (dtype != SD_U8 && dtype != SD_F32) return fail(h, SD_ERR_SHAPE, "dtype must be SD_U8 or SD_F32");
    if (n_frames <= 0 || n_frames > h->chunk) return fail(h, SD_ERR_SHAPE, "sd_compute_range handles at most frames_per_launch frames");
    if (h->lr) return fail(h, SD_ERR_UNSUPPORTED, "sd_compute_range (row-band mode) does not support the left-right check");
    if (h->rect_maps) return fail(h, SD_ERR_UNSUPPORTED, "sd_compute_range (row-band mode) does not support rectification");
    DeviceGuard dg(h->device);
    if (!dg.ok) return fail(h, SD_ERR_CUDA, "cudaSetDevice failed");
    int rc = order_after_previous(h, (cudaStream_t)stream);
    if (rc != SD_OK) return rc;
    rc = run_chunk(h, left, right, dtype, n_frames, out, (cudaStream_t)stream, first_kernel, last_kernel);
    if (rc != SD_OK) return rc;
    return mark_last_use(h, (cudaStream_t)stream);
}

int sd_set_band(sd_handle *h, int pooled_row_offset, int global_height, const float *global_left_gray) {
    if (!h) return SD_ERR_BAD_ARG;
    const int K = h->g.K;
    if (global_height <= 0) {  // back to normal mode
        h->g.band_x_off = 0;
        h->g.Hd_glob = h->g.Hd;
        h->g.H_glob = h->g.H;
        memset(&h->gv, 0, sizeof(h->gv));
        return SD_OK;
    }
    if (h->lr) return fail(h, SD_ERR_UNSUPPORTED, "row-band mode does not support the left-right check (sd_set_lr_check(h, 0, ...) first)");
    if (h->rect_maps) return fail(h, SD_ERR_UNSUPPORTED, "row-band mode does not support rectification (sd_set_rectification(h, NULL, ...) first)");
    if (global_height % K != 0 || h->g.H % K != 0) return fail(h, SD_ERR_UNSUPPORTED, "band mode needs heights divisible by downscale_factor");
    if (!global_left_gray) return fail(h, SD_ERR_BAD_ARG, "band mode needs the global left gray image");
    h->g.band_x_off = pooled_row_offset;
    h->g.H_glob = global_height;
    h->g.Hd_glob = global_height / K;
    memset(&h->gv, 0, sizeof(h->gv));
    h->gv.flat = global_left_gray;
    return SD_OK;
}

// ---- row bands over peer memory ------------------------------------------------------------------------------------
namespace {
constexpr size_t kP2PFlagBytes = 4096;
enum { kFlagFromPrev = 0, kFlagFromNext = 1, kFlagGray = 8, kFlagFill = 16, kCtrScatter = 32, kCtrPublish = 33, kCtrFill = 34 };
inline char *p2p_window(const sd_handle *h, int q, int view) { return h->p2p.peer[q] + (size_t)view * h->p2p.win_bytes; }
inline float *p2p_gray(const sd_handle *h, int q, int parity, int plane = 0) {
    return (float *)(h->p2p.peer[q] + 2 * h->p2p.win_bytes + (size_t)parity * h->p2p.gray_bytes +
                     (size_t)plane * h->p2p.gray_plane_bytes);
}
inline unsigned *p2p_flags(const sd_handle *h, int q) { return (unsigned *)(h->p2p.peer[q] + 2 * h->p2p.win_bytes + 2 * h->p2p.gray_bytes); }
inline float *p2p_fill(const sd_handle *h, int q, int parity) {
    return (float *)((char *)p2p_flags(h, q) + kP2PFlagBytes + (size_t)parity * h->p2p.fill_bytes);
}
}  // namespace

int sd_band_p2p_init(sd_handle *h, int world, int rank, const int32_t *band_row0, int halo_rows, int dtype, void *ipc_handle_out) {
    if (!h || !band_row0 || !ipc_handle_out) return SD_ERR_BAD_ARG;
    if (world < 1 || world > 8 || rank < 0 || rank >= world) return fail(h, SD_ERR_BAD_ARG, "peer-memory band mode supports 1..8 ranks");
    if (dtype != SD_U8 && dtype != SD_F32) return fail(h, SD_ERR_SHAPE, "dtype must be SD_U8 or SD_F32");
    if (h->p2p.on) return fail(h, SD_ERR_BAD_ARG, "sd_band_p2p_init was already called on this handle");
    if (h->rect_maps) return fail(h, SD_ERR_UNSUPPORTED, "row-band mode does not support rectification (sd_set_rectification(h, NULL, ...) first)");
    const Geom &g = h->g;
    const int esize = dtype == SD_U8 ? 1 : 4, K = g.K;
    if ((g.W * esize) % 16 != 0 || g.W % 4 != 0) return fail(h, SD_ERR_UNSUPPORTED, "peer-memory band mode needs 16-byte image rows");
    int tallest = 0;
    for (int q = 0; q < world; q++) {
        const int rows = band_row0[q + 1] - band_row0[q];
        if (rows < halo_rows || rows % K != 0 || band_row0[q] % K != 0) return fail(h, SD_ERR_SHAPE, "bands must be multiples of downscale_factor and at least as tall as the halo");
        if (rows > tallest) tallest = rows;
    }
    if (halo_rows % K != 0 || band_row0[0] != 0) return fail(h, SD_ERR_SHAPE, "halo must be a multiple of downscale_factor; bands start at row 0");
    {   // the halo must cover aggregation + cost + 1 pooled rows and the secondary matching window of those rows
        const int need_a = g.rl + g.r_cost + 1, need_s = (K + g.r_sad + K - 1) / K;
        if (halo_rows / K < (need_a > need_s ? need_a : need_s))
            return fail(h, SD_ERR_UNSUPPORTED, "halo too small for this configuration: needs max(large_mbm_radius + ncc_patch_radius + 1, ceil((K + sad_patch_radius) / K)) pooled rows");
    }
    if (g.H != band_row0[rank + 1] - band_row0[rank] + 2 * halo_rows) return fail(h, SD_ERR_SHAPE, "the handle's height must be band rows + 2 * halo rows");
    DeviceGuard dg(h->device);
    if (!dg.ok) return fail(h, SD_ERR_CUDA, "cudaSetDevice failed");
    sd_handle::P2P &p = h->p2p;   // (as created: an init that failed has closed it again)
    p.world = world;
    p.rank = rank;
    p.dtype = dtype;
    p.halo_rows = halo_rows;
    for (int q = 0; q <= world; q++) p.row0[q] = band_row0[q];
    p.win_bytes = (((size_t)3 * (tallest + 2 * halo_rows) * g.W * esize) + 255) & ~(size_t)255;
    // (the left-right check adds the mirrored frame's gray plane, its background fill the two fill areas)
    p.gray_plane_bytes = (((size_t)tallest * g.W * sizeof(float)) + 255) & ~(size_t)255;
    p.gray_bytes = (h->lr ? 2 : 1) * p.gray_plane_bytes;
    p.fill_bytes = h->lr_fill ? fill_area_bytes(g.W) : 0;
    const size_t total = 2 * p.win_bytes + 2 * p.gray_bytes + kP2PFlagBytes + 2 * p.fill_bytes;
    SD_CUDA(h, cudaMalloc((void **)&p.base, total));
    cudaIpcMemHandle_t ipc;
    cudaError_t e = cudaMemset(p.base, 0, total);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&ipc, p.base);
    if (e != cudaSuccess) {
        p.close();
        return fail_cuda(h, e, "sd_band_p2p_init (memset / cudaIpcGetMemHandle)");
    }
    p.peer[rank] = p.base;
    p.timeout.alloc();   // optional: without it a peer that never shows up is not reported
    static_assert(sizeof(ipc) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(ipc_handle_out, &ipc, sizeof(ipc));
    p.on = true;
    p.connected = (world == 1);
    return SD_OK;
}

int sd_band_p2p_connect(sd_handle *h, const void *ipc_handles) {
    if (!h || !ipc_handles) return SD_ERR_BAD_ARG;
    if (!h->p2p.on) return fail(h, SD_ERR_BAD_ARG, "call sd_band_p2p_init first");
    DeviceGuard dg(h->device);
    if (!dg.ok) return fail(h, SD_ERR_CUDA, "cudaSetDevice failed");
    sd_handle::P2P &p = h->p2p;
    for (int q = 0; q < p.world; q++) {
        if (q == p.rank || p.peer[q]) continue;
        cudaIpcMemHandle_t ipc;
        memcpy(&ipc, (const char *)ipc_handles + (size_t)q * sizeof(ipc), sizeof(ipc));
        SD_CUDA(h, cudaIpcOpenMemHandle((void **)&p.peer[q], ipc, cudaIpcMemLazyEnablePeerAccess));
    }
    p.connected = true;
    return SD_OK;
}

int sd_band_p2p_compute(sd_handle *h, const void *left_band, const void *right_band, float *out, void *stream) {
    if (!h) return SD_ERR_BAD_ARG;
    if (!left_band || !right_band || !out) return fail(h, SD_ERR_BAD_ARG, "null image pointer");
    sd_handle::P2P &p = h->p2p;
    if (!p.on || !p.connected) return fail(h, SD_ERR_BAD_ARG, "peer-memory band mode is not connected (sd_band_p2p_init / _connect)");
    if (h->chunk < 1) return fail(h, SD_ERR_SHAPE, "handle has no scratch");
    if (p.timeout.host && *(volatile unsigned long long *)p.timeout.host != 0) {
        const unsigned long long w = *(volatile unsigned long long *)p.timeout.host;
        snprintf(h->err, sizeof(h->err), "row-band exchange timed out: frame %llu never received flag %llu from a peer rank "
                 "(a rank failed or made fewer sd_band_p2p_compute calls); results since then are invalid", w >> 32, (w & 0xffffffffull) - 1);
        return SD_ERR_CUDA;
    }
    DeviceGuard dg(h->device);
    if (!dg.ok) return fail(h, SD_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t st = (cudaStream_t)stream;
    int rc = order_after_previous(h, st);
    if (rc != SD_OK) return rc;
    const Geom &g = h->g;
    const int W = g.W, esize = p.dtype == SD_U8 ? 1 : 4, r = p.rank, n = p.world;
    const int prev = (r + n - 1) % n, next = (r + 1) % n;
    auto rows_of = [&](int q) { return p.row0[q + 1] - p.row0[q]; };
    const int band_rows = rows_of(r), halo = p.halo_rows;
    const unsigned epoch = ++p.epoch;
    unsigned *myflags = p2p_flags(h, r);
    // exchange step 1, fused with the copy into my own window: halos go straight into the neighbours' HBM
    SD_CUDA(h, launch_band_scatter(left_band, right_band, p2p_window(h, r, 0), p2p_window(h, r, 1), p2p_window(h, prev, 0),
                                   p2p_window(h, prev, 1), p2p_window(h, next, 0), p2p_window(h, next, 1), W * esize, band_rows,
                                   halo, band_rows + 2 * halo, rows_of(prev) + 2 * halo, rows_of(next) + 2 * halo,
                                   myflags + kCtrScatter, p2p_flags(h, prev) + kFlagFromNext, p2p_flags(h, next) + kFlagFromPrev,
                                   epoch, st));
    SD_CUDA(h, launch_wait_flags(myflags, kFlagFromPrev, 2, epoch, p.timeout.dev, st));
    // gray + pool on the local window [top halo | band | bottom halo] (with the left-right check: frame 0 and the mirrored
    // frame 1 of the pair, read from the same window -- mirroring reverses columns only)
    // (h->g is the handle's own geometry and is rewritten for the two halves of every frame: a handle is not
    //  thread-safe -- include/stereo_b200.h -- and the kernels receive Geom by value, so launches already in flight keep
    //  the values they were given)
    h->g.band_x_off = 0;
    h->g.Hd_glob = g.Hd;
    h->g.H_glob = g.H;
    memset(&h->gv, 0, sizeof(h->gv));
    rc = run_chunk(h, p2p_window(h, r, 0), p2p_window(h, r, 1), p.dtype, 1, out, st, 0, 0);
    if (rc != SD_OK) return rc;
    // exchange step 2: publish my left gray band (with the check also the mirrored frame's), tell every rank (myself
    // included)
    const int parity = (int)(epoch & 1u);
    unsigned *peer_flags[8];
    for (int q = 0; q < n; q++) peer_flags[q] = p2p_flags(h, q) + kFlagGray + r;
    if (h->lr)
        SD_CUDA(h, launch_publish_gray(h->s.gray + (size_t)halo * W, p2p_gray(h, r, parity), (size_t)band_rows * W,
                                       myflags + kCtrPublish, peer_flags, n, epoch, st, 2, (size_t)2 * g.H * W,
                                       p.gray_plane_bytes / sizeof(float)));
    else
        SD_CUDA(h, launch_publish_gray(h->s.gray + (size_t)halo * W, p2p_gray(h, r, parity), (size_t)band_rows * W,
                                       myflags + kCtrPublish, peer_flags, n, epoch, st));
    SD_CUDA(h, launch_wait_flags(myflags, kFlagGray, n, epoch, p.timeout.dev, st));
    // matching + secondary + fill on the window; the fill reads its colour row from whichever rank owns it
    h->g.band_x_off = (p.row0[r] - halo) / g.K;
    h->g.H_glob = p.row0[n];
    h->g.Hd_glob = p.row0[n] / g.K;
    h->gv.n = n;
    for (int q = 0; q < n; q++) {
        h->gv.band[q] = p2p_gray(h, q, parity);
        h->gv.row0[q] = p.row0[q];
    }
    h->gv.row0[n] = p.row0[n];
    h->gv_mir = h->gv;
    for (int q = 0; q < n; q++) h->gv_mir.band[q] = p2p_gray(h, q, parity, 1);
    rc = run_chunk(h, nullptr, nullptr, p.dtype, 1, out, st, 1, 3);
    if (rc != SD_OK) return rc;
    if (h->lr_fill) {
        // exchange step 3: the column pass of the background fill needs the frame's first / last row that kept a pixel,
        // which can lie on any rank.  Publish my band's bounds and rows, wait for every rank's, fill my band rows.
        unsigned *fill_flags[8];
        for (int q = 0; q < n; q++) fill_flags[q] = p2p_flags(h, q) + kFlagFill + r;
        SD_CUDA(h, launch_publish_fill_bounds(h->lr_rows + halo, out + (size_t)halo * W, band_rows, p.row0[r], W,
                                              p2p_fill(h, r, parity), myflags + kCtrFill, fill_flags, n, epoch, st));
        SD_CUDA(h, launch_wait_flags(myflags, kFlagFill, n, epoch, p.timeout.dev, st));
        FillAreas areas = {};
        areas.n = n;
        for (int q = 0; q < n; q++) areas.area[q] = p2p_fill(h, q, parity);
        SD_CUDA(h, launch_lr_fill_cols_band(out, h->lr_rows, halo, band_rows, p.row0[r], W, areas, st));
    }
    return mark_last_use(h, st);
}

int sd_compute_host(sd_handle *h, const void *left, const void *right, int dtype, int n_frames, float *out) {
    if (!h) return SD_ERR_BAD_ARG;
    if (!left || !right || !out) return fail(h, SD_ERR_BAD_ARG, "null image pointer");
    if (dtype != SD_U8 && dtype != SD_F32) return fail(h, SD_ERR_SHAPE, "dtype must be SD_U8 or SD_F32");
    if (n_frames <= 0) return fail(h, SD_ERR_SHAPE, "n_frames must be positive");
    DeviceGuard dg(h->device);
    if (!dg.ok) return fail(h, SD_ERR_CUDA, "cudaSetDevice failed");
    int rc = ensure_host_pipeline(h, dtype);
    if (rc != SD_OK) return rc;
    const HostPipeline &hp = *h->host;
    rc = order_after_previous(h, hp.st_comp);
    if (rc != SD_OK) return rc;
    const size_t inb = in_bytes_per_frame(h, dtype), outn = (size_t)h->g.H * h->g.W;
    // Chunk schedule: a short first chunk (its H2D copy cannot overlap anything) and a short last chunk (neither
    // can its D2H copy); full chunks in between keep the fused kernel's wave quantisation efficient.
    // Copies of a chunk cannot overlap its own kernels, so the host path uses chunks of at most kHostChunk frames (the
    // device path's larger default only matters for the fused kernel's wave quantisation).
    const int hc = host_chunk_frames(h);
    const int edge = (hc >= 4 && n_frames >= 3 * hc) ? 2 : hc;
    int it = 0;
    // On any failure below, copies to / from the caller's host buffers may still be in flight: drain before returning.
    struct Drain {
        const HostPipeline &hp;
        bool armed;
        ~Drain() {
            if (!armed) return;
            cudaStreamSynchronize(hp.st_h2d);
            cudaStreamSynchronize(hp.st_comp);
            cudaStreamSynchronize(hp.st_d2h);
        }
    } drain{hp, true};
    for (int f0 = 0; f0 < n_frames; it++) {
        int nf = hc;
        const int left_over = n_frames - f0;
        if (f0 == 0) nf = edge;
        else if (left_over <= edge) nf = left_over;
        else if (left_over - edge < hc) nf = left_over - edge;
        if (nf > left_over) nf = left_over;
        const int sl = it % kSlots;
        // inputs of slot sl may be overwritten once the kernels of its previous use are done
        if (it >= kSlots) SD_CUDA(h, cudaStreamWaitEvent(hp.st_h2d, hp.ev_comp[sl], 0));
        SD_CUDA(h, cudaMemcpyAsync(hp.din_l[sl], (const char *)left + inb * f0, inb * nf, cudaMemcpyHostToDevice, hp.st_h2d));
        SD_CUDA(h, cudaMemcpyAsync(hp.din_r[sl], (const char *)right + inb * f0, inb * nf, cudaMemcpyHostToDevice, hp.st_h2d));
        SD_CUDA(h, cudaEventRecord(hp.ev_h2d[sl], hp.st_h2d));
        SD_CUDA(h, cudaStreamWaitEvent(hp.st_comp, hp.ev_h2d[sl], 0));
        // the output of slot sl may be overwritten once its previous D2H is done
        if (it >= kSlots) SD_CUDA(h, cudaStreamWaitEvent(hp.st_comp, hp.ev_d2h[sl], 0));
        rc = run_chunk(h, hp.din_l[sl], hp.din_r[sl], dtype, nf, hp.dout[sl], hp.st_comp);
        if (rc != SD_OK) return rc;
        SD_CUDA(h, cudaEventRecord(hp.ev_comp[sl], hp.st_comp));
        SD_CUDA(h, cudaStreamWaitEvent(hp.st_d2h, hp.ev_comp[sl], 0));
        SD_CUDA(h, cudaMemcpyAsync(out + outn * f0, hp.dout[sl], outn * nf * sizeof(float), cudaMemcpyDeviceToHost, hp.st_d2h));
        SD_CUDA(h, cudaEventRecord(hp.ev_d2h[sl], hp.st_d2h));
        f0 += nf;
    }
    SD_CUDA(h, cudaStreamSynchronize(hp.st_d2h));
    SD_CUDA(h, cudaStreamSynchronize(hp.st_comp));
    drain.armed = false;
    h->ev_last_valid = false;  // everything on this handle has completed
    return SD_OK;
}

int sd_get_stage(sd_handle *h, int stage, int frame, float *dst, void *stream) {
    if (!h) return SD_ERR_BAD_ARG;
    if (!dst) return fail(h, SD_ERR_BAD_ARG, "null destination");
    if (frame < 0 || frame >= h->chunk) return fail(h, SD_ERR_SHAPE, "frame index outside the chunk");
    if (stage == SD_STAGE_RIGHT && !h->lr) return fail(h, SD_ERR_UNSUPPORTED, "the right view's map exists only with the left-right check on");
    if (stage == SD_STAGE_RIGHT && frame >= lr_pairs(h)) return fail(h, SD_ERR_SHAPE, "frame index outside the chunk (frames_per_launch / 2 pairs)");
    DeviceGuard dg(h->device);
    if (!dg.ok) return fail(h, SD_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t st = (cudaStream_t)stream;
    {
        const int rc = order_after_previous(h, st);
        if (rc != SD_OK) return rc;
    }
    const Geom &g = h->g;
    const size_t n = (size_t)g.H * g.W, nd = (size_t)g.Hd * g.Wd;
    const int threads = 256, blocks = (int)((nd + threads - 1) / threads);
    switch (stage) {
        case SD_STAGE_GRAY_L:
        case SD_STAGE_GRAY_R:
            SD_CUDA(h, cudaMemcpyAsync(dst, h->s.gray + ((size_t)frame * 2 + (stage - SD_STAGE_GRAY_L)) * n, n * 4,
                                       cudaMemcpyDeviceToDevice, st));
            break;
        case SD_STAGE_POOL_L:
        case SD_STAGE_POOL_R:
            SD_CUDA(h, cudaMemcpyAsync(dst, h->s.pool + ((size_t)frame * 2 + (stage - SD_STAGE_POOL_L)) * nd, nd * 4,
                                       cudaMemcpyDeviceToDevice, st));
            break;
        case SD_STAGE_WTA:
            extract_wta<<<blocks, threads, 0, st>>>(h->s.wta4 + frame * nd, dst, (int)nd, (float)g.min_ds);
            SD_CUDA(h, cudaGetLastError());
            break;
        case SD_STAGE_AGG3:
            extract_agg3<<<blocks, threads, 0, st>>>(h->s.wta4 + frame * nd, h->s.edge2 + frame * nd, dst, (int)nd, g.L);
            SD_CUDA(h, cudaGetLastError());
            break;
        case SD_STAGE_REFINED:
            SD_CUDA(h, cudaMemcpyAsync(dst, h->s.refined + frame * nd, nd * 4, cudaMemcpyDeviceToDevice, st));
            break;
        case SD_STAGE_RIGHT:
            unmirror_rows<<<dim3((g.W + 255) / 256, g.H), 256, 0, st>>>(h->rmap + (size_t)frame * n, dst, g.H, g.W);
            SD_CUDA(h, cudaGetLastError());
            break;
        default:
            return fail(h, SD_ERR_SHAPE, "unknown stage");
    }
    return mark_last_use(h, st);   // the copy reads scratch: a following call on another stream must wait for it
}

int sd_stage_pointer(sd_handle *h, int stage, int frame, const float **ptr) {
    if (!h || !ptr) return SD_ERR_BAD_ARG;
    *ptr = nullptr;
    if (frame < 0 || frame >= h->chunk) return fail(h, SD_ERR_SHAPE, "frame index outside the chunk");
    const Geom &g = h->g;
    const size_t n = (size_t)g.H * g.W, nd = (size_t)g.Hd * g.Wd;
    switch (stage) {
        case SD_STAGE_GRAY_L:
        case SD_STAGE_GRAY_R: *ptr = h->s.gray + ((size_t)frame * 2 + (stage - SD_STAGE_GRAY_L)) * n; break;
        case SD_STAGE_POOL_L:
        case SD_STAGE_POOL_R: *ptr = h->s.pool + ((size_t)frame * 2 + (stage - SD_STAGE_POOL_L)) * nd; break;
        case SD_STAGE_REFINED: *ptr = h->s.refined + frame * nd; break;
        case SD_STAGE_RIGHT: return fail(h, SD_ERR_UNSUPPORTED, "the right view's map is stored mirrored (use sd_get_stage)");
        default: return fail(h, SD_ERR_UNSUPPORTED, "this stage is not stored as a plain float plane (use sd_get_stage)");
    }
    return SD_OK;
}

int sd_set_debug_screen(sd_handle *h, float *approx_volume) {
    if (!h) return SD_ERR_BAD_ARG;
    if (approx_volume && !h->s.pass_mask) return fail(h, SD_ERR_UNSUPPORTED, "this configuration has no level screen");
    h->s.dbg_screen = approx_volume;
    return SD_OK;
}

int sd_set_debug_volumes(sd_handle *h, float *cost_volume, float *aggregated_volume) {
    if (!h) return SD_ERR_BAD_ARG;
    h->dbg_cost = cost_volume;
    h->dbg_agg = aggregated_volume;
    return SD_OK;
}

int sd_set_variant(sd_handle *h, int variant) {
    if (!h) return SD_ERR_BAD_ARG;
    if (variant < 0 || variant > 3) return fail(h, SD_ERR_BAD_ARG, "variant must be 0..3");
    if (variant == 3 && !mbm_wta_ws_supported(h->g))
        return fail(h, SD_ERR_UNSUPPORTED, "warp-specialised fused kernel needs radii 1/4/10, cost radius 1 and L <= ~150");
    if (variant == 2 && !mbm_wta_fast_supported(h->g))
        return fail(h, SD_ERR_UNSUPPORTED, "specialised fused kernel needs radii 1/4/10, cost radius 1");
    h->variant = variant;
    return SD_OK;
}

int sd_launches_per_call(sd_handle *h, int n_frames) {
    if (!h || n_frames <= 0) return 0;
    // gray+pool, [pad planes for the TMA-staged specialised kernels], [level screen], cost+agg+WTA, secondary, fill
    // (left-right check: chunks of chunk/2 pairs, kernels A..C over both frames of a pair, + the checked fill;
    //  + its row and column passes with the background fill; + the remap with rectification)
    int total = 0;
    const int per = h->lr ? lr_pairs(h) : h->chunk;
    const int nchunks = (n_frames + per - 1) / per, base = n_frames / nchunks, extra = n_frames % nchunks;
    for (int c = 0; c < nchunks; c++) {   // the same split as sd_compute
        const int nf = (base + (c < extra ? 1 : 0)) * (h->lr ? 2 : 1);
        total += h->lr ? (h->lr_fill ? 3 : 1) : 0;
        total += h->rect_maps ? 1 : 0;
        const bool scr = active_variant(h, nf) == 2 && screen_active(h, nf);
        // (+2 behind the screen in reference-compat mode: absolute-index targets + gather pass)
        total += 4 + (active_variant(h, nf) >= 2 ? 1 : 0) + (scr ? 1 : 0) + (scr && h->s.agg_vol ? 2 : 0) +
                 (active_split(h, nf) > 1 ? 1 : 0);   // + merge of the part slots
    }
    return total;
}

int sd_frames_per_launch(sd_handle *h) { return h ? h->chunk : 0; }

int sd_set_lr_check(sd_handle *h, int on, float tolerance, float invalid_disparity) {
    if (!h) return SD_ERR_BAD_ARG;
    // (every rank must run the same exchange steps on every frame, and the exported buffer is sized for the mode)
    if (h->p2p.on)
        return fail(h, SD_ERR_UNSUPPORTED, "the left-right check of a peer-memory band handle is fixed at sd_band_p2p_init: "
                                           "set it before sd_band_p2p_init");
    if (!on) {
        if (h->rmap) {
            DeviceGuard dg(h->device);
            if (!dg.ok) return fail(h, SD_ERR_CUDA, "cudaSetDevice failed");
            h->allocs.release(h->rmap);
            h->allocs.release(h->lr_rows);
        }
        h->lr = false;
        h->lr_fill = false;
        return SD_OK;
    }
    if (!(tolerance >= 0.0f && tolerance <= 3.402823466e38f)) return fail(h, SD_ERR_BAD_ARG, "tolerance must be finite and >= 0");
    if (h->chunk < 2)
        return fail(h, SD_ERR_SHAPE, "the left-right check runs each frame together with its mirrored pair: create the handle "
                                     "with frames_per_launch >= 2");
    if (h->gv.flat) return fail(h, SD_ERR_UNSUPPORTED, "row-band mode does not support the left-right check");
    if (!h->rmap) {
        DeviceGuard dg(h->device);
        if (!dg.ok) return fail(h, SD_ERR_CUDA, "cudaSetDevice failed");
        SD_CUDA(h, h->allocs.alloc(&h->rmap, (size_t)lr_pairs(h) * h->g.H * h->g.W * sizeof(float)));
    }
    h->lr = true;
    h->lr_tol = tolerance;
    h->lr_invalid = invalid_disparity;
    return SD_OK;
}

int sd_set_lr_fill(sd_handle *h, int on) {
    if (!h) return SD_ERR_BAD_ARG;
    if (h->p2p.on)
        return fail(h, SD_ERR_UNSUPPORTED, "the background fill of a peer-memory band handle is fixed at sd_band_p2p_init: "
                                           "set it before sd_band_p2p_init");
    if (!h->lr) return fail(h, SD_ERR_UNSUPPORTED, "the background fill needs the left-right check (sd_set_lr_check(h, 1, ...) first)");
    if (on && !h->lr_rows) {
        DeviceGuard dg(h->device);
        if (!dg.ok) return fail(h, SD_ERR_CUDA, "cudaSetDevice failed");
        SD_CUDA(h, h->allocs.alloc(&h->lr_rows, (size_t)lr_pairs(h) * h->g.H));
    }
    h->lr_fill = on != 0;
    return SD_OK;
}

int sd_lr_fill(const float *left_map, const float *right_map, int n, int H, int W, float tolerance, float invalid_disparity,
               float *out, void *cuda_stream) {
    if (!left_map || !right_map || !out || n <= 0 || H <= 0 || W <= 0) return SD_ERR_BAD_ARG;
    if (!(tolerance >= 0.0f && tolerance <= 3.402823466e38f)) return SD_ERR_BAD_ARG;
    if ((long long)n * H > 0x7fffffffLL) return SD_ERR_BAD_ARG;   // one block per row
    if (out == right_map) return SD_ERR_BAD_ARG;                   // the row pass reads the right map while it writes
    cudaStream_t st = (cudaStream_t)cuda_stream;
    unsigned char *rows = nullptr;
    if (cudaMallocAsync((void **)&rows, (size_t)n * H, st) != cudaSuccess) return SD_ERR_CUDA;
    const cudaError_t e = launch_lr_background_fill(left_map, right_map, false, n, H, W, tolerance, invalid_disparity, out,
                                                    rows, st);
    if (cudaFreeAsync(rows, st) != cudaSuccess || e != cudaSuccess) return SD_ERR_CUDA;
    return SD_OK;
}

int sd_set_rectification(sd_handle *h, const float *left_map_x, const float *left_map_y, const float *right_map_x,
                         const float *right_map_y, void *cuda_stream) {
    if (!h) return SD_ERR_BAD_ARG;
    const int given = !!left_map_x + !!left_map_y + !!right_map_x + !!right_map_y;
    if (given != 0 && given != 4) return fail(h, SD_ERR_BAD_ARG, "pass all four maps, or all four NULL to switch rectification off");
    DeviceGuard dg(h->device);
    if (!dg.ok) return fail(h, SD_ERR_CUDA, "cudaSetDevice failed");
    if (given == 0) {   // (cudaFree waits for the chunks still reading the buffers)
        h->allocs.release(h->rect_maps);
        h->allocs.release(h->rect_frames);
        return SD_OK;
    }
    if (h->gv.flat || h->p2p.on) return fail(h, SD_ERR_UNSUPPORTED, "row-band mode does not support rectification");
    if (h->g.H >= 32768 || h->g.W >= 32768) return fail(h, SD_ERR_UNSUPPORTED, "rectification needs H, W < 32768 (as cv2.remap)");
    const size_t n = (size_t)h->g.H * h->g.W;
    if (!h->rect_maps) {
        SD_CUDA(h, h->allocs.alloc(&h->rect_maps, 4 * n * sizeof(float)));
        const cudaError_t e = h->allocs.alloc(&h->rect_frames, (size_t)h->chunk * 2 * 3 * n * sizeof(float));
        if (e != cudaSuccess) {
            h->allocs.release(h->rect_maps);
            return fail_cuda(h, e, "sd_set_rectification (rectified frames)");
        }
    }
    // the previous call's chunks may still read the old maps: the copies follow them on cuda_stream
    cudaStream_t st = (cudaStream_t)cuda_stream;
    int rc = order_after_previous(h, st);
    if (rc != SD_OK) return rc;
    const float *src[4] = {left_map_x, left_map_y, right_map_x, right_map_y};
    for (int i = 0; i < 4; i++)
        SD_CUDA(h, cudaMemcpyAsync(h->rect_maps + i * n, src[i], n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return mark_last_use(h, st);
}

int sd_rectify(const float *map_x, const float *map_y, const void *src, void *dst, int dtype, int n_planes, int H, int W,
               void *cuda_stream) {
    if (!map_x || !map_y || !src || !dst || n_planes <= 0 || H <= 0 || W <= 0) return SD_ERR_BAD_ARG;
    if (dtype != SD_U8 && dtype != SD_F32) return SD_ERR_BAD_ARG;
    if (H >= 32768 || W >= 32768) return SD_ERR_BAD_ARG;
    if (dst == src) return SD_ERR_BAD_ARG;   // a gather cannot run in place
    RectifyViews v = {};
    v.view[0] = RectifyView{map_x, map_y, src, dst};
    return launch_rectify(v, 1, dtype, n_planes, H, W, (cudaStream_t)cuda_stream) == cudaSuccess ? SD_OK : SD_ERR_CUDA;
}

int sd_reproject(const float *disparity, int n, int H, int W, const double *Q, int handle_missing_values, float *xyz,
                 void *cuda_stream) {
    if (!disparity || !Q || !xyz || n <= 0 || H <= 0 || W <= 0) return SD_ERR_BAD_ARG;
    const unsigned long long hw = (unsigned long long)H * W;
    if ((unsigned long long)n > (1ull << 58) / hw) return SD_ERR_BAD_ARG;   // larger than any buffer: 12 * px must not wrap
    const unsigned long long px = n * hw;
    const uintptr_t d0 = (uintptr_t)disparity, d1 = d0 + 4 * px, x0 = (uintptr_t)xyz, x1 = x0 + 12 * px;
    if (x0 < d1 && d0 < x1) return SD_ERR_BAD_ARG;                 // the points would overwrite maps still to be read
    ReprojectQ q;
    memcpy(q.q, Q, sizeof(q.q));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    unsigned *mins = nullptr;
    if (handle_missing_values && cudaMallocAsync((void **)&mins, (size_t)n * sizeof(unsigned), st) != cudaSuccess)
        return SD_ERR_CUDA;
    const cudaError_t e = launch_reproject(disparity, n, H, W, q, mins, xyz, st);
    if ((mins && cudaFreeAsync(mins, st) != cudaSuccess) || e != cudaSuccess) return SD_ERR_CUDA;
    return SD_OK;
}

int sd_set_level_split(sd_handle *h, int on) {
    if (!h) return SD_ERR_BAD_ARG;
    h->split_off = (on == 0);
    return SD_OK;
}

int sd_level_split(sd_handle *h, int n_frames) {
    if (!h || n_frames <= 0) return 0;
    return active_split(h, n_frames > h->chunk ? h->chunk : n_frames);
}

int sd_active_variant(sd_handle *h) { return h ? active_variant(h, h->chunk) : 0; }

int sd_set_screen(sd_handle *h, int on) {
    if (!h) return SD_ERR_BAD_ARG;
    if (on && !h->s.pass_mask)
        return fail(h, SD_ERR_UNSUPPORTED, "the level screen needs the specialised fused kernel (radii 1/4/10, cost radius 1) and 3 <= L <= 128");
    h->screen = on != 0;
    h->screen_pause = 0;
    return SD_OK;
}

int sd_screen_paused(sd_handle *h) { return h ? h->screen_pause : 0; }

int sd_screen_active(sd_handle *h) { return (h && active_variant(h, h->chunk) == 2 && screen_active(h, h->chunk)) ? 1 : 0; }

int sd_screen_stats(sd_handle *h, double *evaluated_fraction, int reset) {
    if (!h || !evaluated_fraction) return SD_ERR_BAD_ARG;
    *evaluated_fraction = 1.0;
    if (!h->s.screen_stats) return SD_OK;
    DeviceGuard dg(h->device);
    if (!dg.ok) return fail(h, SD_ERR_CUDA, "cudaSetDevice failed");
    unsigned long long st[2] = {0, 0};
    if (h->ev_last_valid) SD_CUDA(h, cudaEventSynchronize(h->ev_last));
    SD_CUDA(h, cudaMemcpy(st, h->s.screen_stats, sizeof(st), cudaMemcpyDeviceToHost));
    if (st[1] > 0) *evaluated_fraction = (double)st[0] / (double)st[1];
    if (reset) SD_CUDA(h, cudaMemset(h->s.screen_stats, 0, sizeof(st)));
    return SD_OK;
}

int sd_profile_enable(sd_handle *h, int on) {
    if (!h) return SD_ERR_BAD_ARG;
    h->prof = on != 0;
    return SD_OK;
}

static int profile_collect(sd_handle *h, double *ms6, int *n6) {
    DeviceGuard dg(h->device);
    std::vector<cudaEvent_t> &ev = h->prof_events;
    for (int k = 0; k < kProfMarks - 1; k++) {
        ms6[k] = 0.0;
        n6[k] = 0;
    }
    if (!ev.empty()) SD_CUDA(h, cudaEventSynchronize(ev.back()));
    for (size_t i = 0; i + kProfMarks <= ev.size(); i += kProfMarks) {
        for (int k = 0; k < kProfMarks - 1; k++) {
            float t = 0.f;
            SD_CUDA(h, cudaEventElapsedTime(&t, ev[i + k], ev[i + k + 1]));
            ms6[k] += t;
            n6[k] += 1;
        }
    }
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
    ev.clear();
    return SD_OK;
}

int sd_profile_read(sd_handle *h, double *ms, int *launches) {
    if (!h || !ms || !launches) return SD_ERR_BAD_ARG;
    double m6[kProfMarks - 1];
    int n6[kProfMarks - 1];
    const int rc = profile_collect(h, m6, n6);
    if (rc != SD_OK) return rc;
    ms[0] = m6[0]; ms[1] = m6[1] + m6[2] + m6[3]; ms[2] = m6[4]; ms[3] = m6[5];
    launches[0] = n6[0]; launches[1] = n6[3]; launches[2] = n6[4]; launches[3] = n6[5];
    return SD_OK;
}

int sd_profile_read_detail(sd_handle *h, double *ms, int *launches) {
    if (!h || !ms || !launches) return SD_ERR_BAD_ARG;
    return profile_collect(h, ms, launches);
}

int sd_check_guards(sd_handle *h, long long *corrupted_bytes) {
    if (!h || !corrupted_bytes) return SD_ERR_BAD_ARG;
    *corrupted_bytes = 0;
    if (!h->allocs.guards) return fail(h, SD_ERR_UNSUPPORTED, "guard bands are off: create the handle with SD_DEBUG_GUARDS=1 in the environment");
    DeviceGuard dg(h->device);
    if (!dg.ok) return fail(h, SD_ERR_CUDA, "cudaSetDevice failed");
    SD_CUDA(h, cudaDeviceSynchronize());
    std::vector<unsigned char> host(kGuardBytes + 256);
    long long bad = 0;
    for (const auto &a : h->allocs.live) {
        const size_t padded = (a.second + 255) & ~(size_t)255;
        // front band; then [payload end, padded end) + back band
        SD_CUDA(h, cudaMemcpy(host.data(), a.first, kGuardBytes, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < kGuardBytes; i++) bad += host[i] != kGuardPattern;
        const size_t tail = padded - a.second + kGuardBytes;
        SD_CUDA(h, cudaMemcpy(host.data(), a.first + kGuardBytes + a.second, tail, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < tail; i++) bad += host[i] != kGuardPattern;
    }
    *corrupted_bytes = bad;
    return SD_OK;
}

const char *sd_last_error(sd_handle *h) { return h ? h->err : "null handle"; }

int sd_last_cuda_error(sd_handle *h) { return h ? h->last_cuda : 0; }

}  // extern "C"
