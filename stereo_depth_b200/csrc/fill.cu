// Kernel D+E: disparity upscale + vertical bilateral fill + horizontal bilateral fill, fused.
//
// Reference: upscale_disparity_vertical_fill.cu:20-51 then horizontal_disparity_fill.cu:19-40
// (two kernels, the second in place).  The horizontal pass only ever reads columns that are
// multiples of K, and those hold exactly what the vertical pass wrote, so every output pixel is a
// pure function of the refined disparity and the left gray image:
//   vf(r, c)  for c % K == 0:  x = r / K, i = r % K, p = K*disp[x][c/K]
//        i == 0            -> p
//        n = K*disp[x-1][c/K];  |p-n| <= thr -> p + (i*(n-p))/K
//        else  cur=GL[r][c]:  |cur-GL[Kx][c]| <= |cur-GL[(K+1)x][c]| ? p : n      (sic: (K+1)*x)
//   out(r, c): m = c % K, nk = c - m, p = vf(r,nk), n = vf(r,nk+K)
//        |p-n| <= thr -> p + (m*(n-p))/K   else colour pick between GL[r][nk], GL[r][nk+K]
// SAFE definitions where the reference is undefined (oracle/stereo_oracle.c so_vfill/so_hfill):
//   rows 1..K-1 of the image (never written by the reference) replicate p;
//   GL[(K+1)x] wraps modulo H;  column nk+K == W reads the next row's column 0 like the
//   reference's flat index does, and p on the last row / when W % K != 0.
// HBM-bound: reads disp [Hd,Wd] and (rarely) gray, writes [H,W]; 4 pixels per thread, STG.128.
#include "common.cuh"

namespace sd {
namespace {

// x / K for the compile-time factors the reference is used with (exact: K is a power of two), IEEE division otherwise.
template <int KT>
__device__ __forceinline__ float div_k(float x, float fk) {
    if (KT == 1) return x;
    if (KT == 2) return __fmul_rn(x, 0.5f);
    if (KT == 4) return __fmul_rn(x, 0.25f);
    return __fdiv_rn(x, fk);
}

// Row `row` of the GLOBAL left gray image (only the rare colour-pick branch gets here).
__device__ __forceinline__ const float *global_gray_row(const GrayView &gv, const float *gl, int row, int W) {
    if (gv.n == 0) return (gv.flat ? gv.flat : gl) + (size_t)row * W;
    // compile-time indices only: the view stays in the kernel's parameter space (no local copy)
    const float *p = gv.band[0];
    int first = gv.row0[0];
#pragma unroll
    for (int q = 1; q < 8; q++)
        if (q < gv.n && row >= gv.row0[q]) {
            p = gv.band[q];
            first = gv.row0[q];
        }
    return p + (size_t)(row - first) * W;
}

// gl = left gray of this handle's (local) image; glg = where the GLOBAL image lives (== gl outside band mode).
template <int KT>
__device__ __forceinline__ float vfill_value(const Geom &g, const float *__restrict__ gl, const GrayView &glg,
                                             const float *__restrict__ disp, int r, int c) {
    const int K = KT > 0 ? KT : g.K, x = r / K, i = r - x * K, yd = c / K;
    const float fk = (float)K;
    const float p = __fmul_rn(fk, __ldg(disp + (size_t)x * g.Wd + yd));
    const int xg = wrapm(x + g.band_x_off, g.Hd_glob);  // global pooled row (the reference's x)
    if (i == 0 || xg == 0 || x == 0) return p;
    const float n = __fmul_rn(fk, __ldg(disp + (size_t)(x - 1) * g.Wd + yd));
    if (fabsf(__fsub_rn(p, n)) <= g.threshold)
        return __fadd_rn(p, div_k<KT>(__fmul_rn((float)i, __fsub_rn(n, p)), fk));
    const float prev_color = __ldg(gl + (size_t)(K * x) * g.W + c);
    const float next_color = __ldg(global_gray_row(glg, gl, wrapm((K + 1) * xg, g.H_glob), g.W) + c);
    const float cur = __ldg(gl + (size_t)r * g.W + c);
    return (fabsf(__fsub_rn(cur, prev_color)) <= fabsf(__fsub_rn(cur, next_color))) ? p : n;
}

template <int KT>
__device__ __forceinline__ float hfill_value(const Geom &g, const float *__restrict__ gl, int r, int c, int nk,
                                             float p, float n) {
    const int m = c - nk, K = KT > 0 ? KT : g.K;
    if (fabsf(__fsub_rn(p, n)) <= g.threshold)
        return __fadd_rn(p, div_k<KT>(__fmul_rn((float)m, __fsub_rn(n, p)), (float)K));
    const size_t o = (size_t)r * g.W;
    const float pc = __ldg(gl + o + nk);
    const size_t cf = o + nk + K;
    const float nc = (cf < (size_t)g.H * g.W) ? __ldg(gl + cf) : pc;
    const float cur = __ldg(gl + o + c);
    return (fabsf(__fsub_rn(cur, pc)) <= fabsf(__fsub_rn(cur, nc))) ? p : n;
}

// value of the "next" mod-K sample to the right of nk on row r
template <int KT>
__device__ __forceinline__ float next_sample(const Geom &g, const float *__restrict__ gl, const GrayView &glg,
                                             const float *__restrict__ disp, int r, int nk, float p) {
    const int K = KT > 0 ? KT : g.K;
    if (nk + K < g.W) return vfill_value<KT>(g, gl, glg, disp, r, nk + K);
    // the reference's flat index lands on column 0 of the next row -- unless this is the GLOBAL last row
    const int rg = wrapm(r + g.band_x_off * K, g.H_glob);
    if (g.W % K == 0 && rg + 1 < g.H_glob && r + 1 < g.H) return vfill_value<KT>(g, gl, glg, disp, r + 1, 0);
    return p;
}

// Left-right consistency check of the left value d at (r, c) of frame `frame` (LrCheck in common.cuh).  The partner is
// read from the MIRRORED right map at column W-1-yr: for the small disparity changes within a warp the reads stay
// contiguous.  (c - W < rint(d) <= c  <=>  0 <= yr < W, without converting a huge d to int.)
// Column of the partner in the mirrored right map (W-1-yr), or -1 when there is none.
__device__ __forceinline__ int lr_partner(int W, int c, float d) {
    if (!(fabsf(d) <= 3.402823466e38f)) return -1;   // NaN, +-inf
    const float rd = rintf(d);
    if (!(rd <= (float)c) || !(rd > (float)(c - W))) return -1;
    return W - 1 - (c - (int)rd);
}

__device__ __forceinline__ float lr_checked(const Geom &g, const LrCheck &lr, int frame, int r, int c, float d) {
    const int m = lr_partner(g.W, c, d);
    if (m < 0) return lr.invalid;
    const float dr = __ldg(lr.right_mirrored + ((size_t)frame * g.H + r) * g.W + m);
    return (fabsf(__fsub_rn(d, dr)) <= lr.tolerance) ? d : lr.invalid;
}

template <int KT, bool LR>
__global__ void __launch_bounds__(256) fill_kernel(Geom g, const float *__restrict__ gray, const GrayView glg,
                                                   const float *__restrict__ refined, float *__restrict__ out, bool vec_ok,
                                                   const LrCheck lr) {
    const int c4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const int r = blockIdx.y * blockDim.y + threadIdx.y;
    const int frame = blockIdx.z;
    if (r >= g.H || c4 >= g.W) return;
    const size_t plane = (size_t)g.H * g.W;
    const float *gl = gray + (size_t)frame * 2 * plane;
    const float *disp = refined + (size_t)frame * g.Hd * g.Wd;
    float *o = out + (size_t)frame * plane + (size_t)r * g.W + c4;
    float v[4];
    int nk_cached = -1;
    float p = 0.0f, n = 0.0f;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int c = c4 + k;
        if (c >= g.W) break;
        const int K = KT > 0 ? KT : g.K;
        const int nk = c - c % K;
        if (nk != nk_cached) {
            p = (nk_cached >= 0 && nk == nk_cached + K) ? n : vfill_value<KT>(g, gl, glg, disp, r, nk);
            n = next_sample<KT>(g, gl, glg, disp, r, nk, p);
            nk_cached = nk;
        }
        v[k] = hfill_value<KT>(g, gl, r, c, nk, p, n);
        if (LR) v[k] = lr_checked(g, lr, frame, r, c, v[k]);
    }
    if (vec_ok && c4 + 3 < g.W) {
        *reinterpret_cast<float4 *>(o) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
        for (int k = 0; k < 4 && c4 + k < g.W; k++) o[k] = v[k];
    }
}

// K = 2 fast path: a thread produces a 2-row x 4-column output block (rows 2x, 2x+1) from 3 + 3 refined
// disparities; the rare colour-pick branches fall back to the generic helpers above, so semantics are identical.
template <bool LR>
__global__ void __launch_bounds__(256) fill_k2_kernel(Geom g, const float *__restrict__ gray, const GrayView glg,
                                                      const float *__restrict__ refined, float *__restrict__ out,
                                                      const LrCheck lr) {
    const int c4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const int x = blockIdx.y * blockDim.y + threadIdx.y;
    const int frame = blockIdx.z;
    if (x >= g.Hd || c4 >= g.W) return;
    const size_t plane = (size_t)g.H * g.W;
    const float *gl = gray + (size_t)frame * 2 * plane;
    const float *disp = refined + (size_t)frame * g.Hd * g.Wd;
    const int y0 = c4 >> 1;
    const bool has3 = c4 + 4 < g.W;
    const float *da = disp + (size_t)x * g.Wd + y0;
    const float a0 = __ldg(da), a1 = __ldg(da + 1), a2 = has3 ? __ldg(da + 2) : 0.0f;
    const int xg = wrapm(x + g.band_x_off, g.Hd_glob);
    const bool first = (xg == 0) || (x == 0);  // the reference returns before the vertical fill for x == 0
    float b0 = 0.0f, b1 = 0.0f, b2 = 0.0f;
    if (!first) {
        b0 = __ldg(da - g.Wd);
        b1 = __ldg(da - g.Wd + 1);
        b2 = has3 ? __ldg(da - g.Wd + 2) : 0.0f;
    }
    const float thr = g.threshold;
    float4 res[2] = {};   // (LR: both rows first, so that the 8 partner loads of the check are in flight together)
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const int r = 2 * x + i;
        if (r >= g.H) break;
        auto vf = [&](float d, float dprev, int c) {
            const float p = __fmul_rn(2.0f, d);
            if (i == 0 || first) return p;
            const float n = __fmul_rn(2.0f, dprev);
            if (fabsf(__fsub_rn(p, n)) <= thr) return __fadd_rn(p, __fmul_rn(__fsub_rn(n, p), 0.5f));
            return vfill_value<2>(g, gl, glg, disp, r, c);
        };
        auto hf = [&](float p, float n, int c) {
            if (fabsf(__fsub_rn(p, n)) <= thr) return __fadd_rn(p, __fmul_rn(__fsub_rn(n, p), 0.5f));
            return hfill_value<2>(g, gl, r, c, c - 1, p, n);
        };
        const float v0 = vf(a0, b0, c4), v1 = vf(a1, b1, c4 + 2);
        const float v2 = has3 ? vf(a2, b2, c4 + 4) : next_sample<2>(g, gl, glg, disp, r, c4 + 2, v1);
        res[i] = make_float4(v0, hf(v0, v1, c4 + 1), v1, hf(v1, v2, c4 + 3));
        if (!LR) *reinterpret_cast<float4 *>(out + (size_t)frame * plane + (size_t)r * g.W + c4) = res[i];
    }
    if (LR) {
        const int rows = g.H - 2 * x < 2 ? g.H - 2 * x : 2;
        float d[2][4], dr[2][4];
        int m[2][4];
#pragma unroll
        for (int i = 0; i < 2; i++) {
            d[i][0] = res[i].x, d[i][1] = res[i].y, d[i][2] = res[i].z, d[i][3] = res[i].w;
#pragma unroll
            for (int k = 0; k < 4; k++) m[i][k] = i < rows ? lr_partner(g.W, c4 + k, d[i][k]) : -1;
        }
#pragma unroll
        for (int i = 0; i < 2; i++) {
            const float *rrow = lr.right_mirrored + ((size_t)frame * g.H + 2 * x + i) * g.W;
#pragma unroll
            for (int k = 0; k < 4; k++) dr[i][k] = m[i][k] >= 0 ? __ldg(rrow + m[i][k]) : 0.0f;
        }
#pragma unroll
        for (int i = 0; i < 2; i++) {
            if (i >= rows) break;
            float o[4];
#pragma unroll
            for (int k = 0; k < 4; k++)
                o[k] = (m[i][k] >= 0 && fabsf(__fsub_rn(d[i][k], dr[i][k])) <= lr.tolerance) ? d[i][k] : lr.invalid;
            *reinterpret_cast<float4 *>(out + (size_t)frame * plane + (size_t)(2 * x + i) * g.W + c4) =
                make_float4(o[0], o[1], o[2], o[3]);
        }
    }
}

// ---- background fill of the pixels the left-right check rejects (DESIGN.md §13) ------------------------------------
// Row pass: one block per row, tiles of kBgTile columns, kBgItems consecutive columns per thread.  A hole's left bound
// is the last kept column before it (block-wide exclusive max scan + the carry of earlier tiles), its right bound the
// first kept column after it (exclusive min scan from the right).  Holes whose right bound lies beyond the tile -- the
// row's trailing run so far -- stay pending and are written as one constant run once the bound is known (or with the
// left bound / `invalid` after the last tile).  Holes are only written after every read of their tile, and bounds are
// kept pixels, which the fill never changes: so `out` may alias `left`.
constexpr int kBgThreads = 256, kBgItems = 8, kBgTile = kBgThreads * kBgItems, kBgWarps = kBgThreads / 32;
constexpr int kNone = 0x7fffffff;

// fill value of a hole bounded by the kept values da (left) and db (right): the smaller, the left one on ties
__device__ __forceinline__ float bg_min(float da, float db) { return db < da ? db : da; }

template <bool MIRRORED>
__global__ void __launch_bounds__(kBgThreads) lr_fill_rows_kernel(const float *left, const float *__restrict__ right,
                                                                  float *out, unsigned char *__restrict__ row_kept, int W,
                                                                  float tolerance, float invalid) {
    __shared__ int warp_last[kBgWarps], warp_first[kBgWarps];
    const size_t row = blockIdx.x;
    const float *dl = left + row * W;
    const float *dr = right + row * W;
    float *o = out + row * W;
    const bool copy_kept = out != left;
    const bool vec = W % 4 == 0 && (reinterpret_cast<uintptr_t>(left) & 15u) == 0;   // float4 loads of the row
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int carry = -1;    // last kept column of the tiles before this one
    int pend = -1;     // first column of the pending trailing hole run
    for (int t0 = 0; t0 < W; t0 += kBgTile) {
        const int c0 = t0 + threadIdx.x * kBgItems;
        float d[kBgItems];
        if (vec && c0 + kBgItems <= W) {
#pragma unroll
            for (int k = 0; k < kBgItems; k += 4) {
                const float4 v = *reinterpret_cast<const float4 *>(dl + c0 + k);
                d[k] = v.x, d[k + 1] = v.y, d[k + 2] = v.z, d[k + 3] = v.w;
            }
        } else {
#pragma unroll
            for (int k = 0; k < kBgItems; k++) d[k] = c0 + k < W ? dl[c0 + k] : 0.0f;
        }
        int m[kBgItems];
        float pr[kBgItems];   // (all partner loads first, so that they are in flight together)
#pragma unroll
        for (int k = 0; k < kBgItems; k++) m[k] = c0 + k < W ? lr_partner(W, c0 + k, d[k]) : -1;
#pragma unroll
        for (int k = 0; k < kBgItems; k++) pr[k] = m[k] >= 0 ? __ldg(dr + (MIRRORED ? m[k] : W - 1 - m[k])) : 0.0f;
        unsigned keep = 0;
        int last = -1, first = kNone;
#pragma unroll
        for (int k = 0; k < kBgItems; k++) {
            const int c = c0 + k;
            if (m[k] >= 0 && fabsf(__fsub_rn(d[k], pr[k])) <= tolerance) {
                keep |= 1u << k;
                last = c;
                first = first == kNone ? c : first;
            }
        }
        // exclusive scans over the threads: last kept column to the left, first kept column to the right
        int incl_last = last, incl_first = first;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            const int a = __shfl_up_sync(0xffffffffu, incl_last, s);
            const int b = __shfl_down_sync(0xffffffffu, incl_first, s);
            if (lane >= s) incl_last = max(incl_last, a);
            if (lane + s < 32) incl_first = min(incl_first, b);
        }
        int before = __shfl_up_sync(0xffffffffu, incl_last, 1);
        int after = __shfl_down_sync(0xffffffffu, incl_first, 1);
        if (lane == 0) before = -1;
        if (lane == 31) after = kNone;
        if (lane == 31) warp_last[warp] = incl_last;
        if (lane == 0) warp_first[warp] = incl_first;
        __syncthreads();
        int tile_last = -1, tile_first = kNone;
#pragma unroll
        for (int w = 0; w < kBgWarps; w++) {
            if (w < warp) before = max(before, warp_last[w]);
            if (w > warp) after = min(after, warp_first[w]);
            tile_last = max(tile_last, warp_last[w]);
            tile_first = min(tile_first, warp_first[w]);
        }
        before = max(before, carry);
        if (pend >= 0 && tile_first != kNone) {   // the pending run ends at this tile's first kept column
            const float db = dl[tile_first];
            const float v = carry >= 0 ? bg_min(dl[carry], db) : db;
            for (int c = pend + threadIdx.x; c < t0; c += kBgThreads) o[c] = v;
            pend = -1;
        }
        int next[kBgItems];
        int b = after;
#pragma unroll
        for (int k = kBgItems - 1; k >= 0; k--) {
            next[k] = b;
            if (keep >> k & 1u) b = c0 + k;
        }
        int a = before;
#pragma unroll
        for (int k = 0; k < kBgItems; k++) {
            const int c = c0 + k;
            if (c >= W) break;
            if (keep >> k & 1u) {
                a = c;
                if (copy_kept) o[c] = d[k];
            } else if (next[k] != kNone) {
                const float db = dl[next[k]];
                o[c] = a >= 0 ? bg_min(dl[a], db) : db;
            }   // else: part of the pending trailing run
        }
        if (tile_first == kNone) {
            if (pend < 0) pend = t0;
        } else {
            carry = tile_last;
            pend = tile_last + 1 < W ? tile_last + 1 : -1;
        }
        __syncthreads();   // warp_last / warp_first are rewritten by the next tile
    }
    if (pend >= 0) {   // a run that touches the right border: its one kept neighbour, or `invalid` in an empty row
        const float v = carry >= 0 ? dl[carry] : invalid;
        for (int c = pend + threadIdx.x; c < W; c += kBgThreads) o[c] = v;
    }
    if (threadIdx.x == 0) row_kept[row] = carry >= 0 ? 1 : 0;
}

// Column pass: a row without kept pixels copies the first non-empty row of its frame when it lies above it, the last
// one when it lies below it; rows between non-empty rows stay `invalid`.  Blocks of non-empty rows return at once.
__global__ void __launch_bounds__(256) lr_fill_cols_kernel(float *out, const unsigned char *__restrict__ row_kept, int H,
                                                           int W) {
    __shared__ int sh_first[8], sh_last[8];
    const size_t row = blockIdx.x;
    if (row_kept[row]) return;
    const size_t frame = row / H;
    const int r = (int)(row - frame * H);
    const unsigned char *fk = row_kept + frame * H;
    int first = kNone, last = -1;
    for (int i = threadIdx.x; i < H; i += 256)
        if (fk[i]) {
            first = min(first, i);
            last = max(last, i);
        }
    first = __reduce_min_sync(0xffffffffu, first);
    last = __reduce_max_sync(0xffffffffu, last);
    if ((threadIdx.x & 31) == 0) {
        sh_first[threadIdx.x >> 5] = first;
        sh_last[threadIdx.x >> 5] = last;
    }
    __syncthreads();
#pragma unroll
    for (int w = 0; w < 8; w++) {
        first = min(first, sh_first[w]);
        last = max(last, sh_last[w]);
    }
    if (last < 0) return;   // no kept pixel in the frame: all `invalid`
    const int src = r < first ? first : (r > last ? last : -1);
    if (src < 0) return;
    const float *s = out + (frame * H + src) * W;
    float *o = out + row * W;
    for (int c = threadIdx.x; c < W; c += 256) o[c] = s[c];
}

// Column pass of one row band (peer-memory row-band mode, DESIGN.md §8): the same rule with the frame's GLOBAL first /
// last non-empty row, taken from every rank's published fill bounds in rank order, and the row to copy read from the
// published copy of the rank that owns it.  One block per band row; blocks of non-empty rows return at once.
__global__ void __launch_bounds__(256) lr_fill_cols_band_kernel(float *out, const unsigned char *__restrict__ row_kept,
                                                                int row_first, int glob_row0, int W, const FillAreas areas) {
    const int r = row_first + blockIdx.x;
    if (row_kept[r]) return;
    int first = -1, last = -1;
    const float *src_first = nullptr, *src_last = nullptr;
    // compile-time indices only: the areas stay in the kernel's parameter space (no local copy)
#pragma unroll
    for (int q = 0; q < 8; q++)
        if (q < areas.n) {
            const float *a = areas.area[q];
            const int f = reinterpret_cast<const int *>(a)[0];
            if (f >= 0) {
                if (first < 0) {
                    first = f;
                    src_first = a + kFillAreaHeaderFloats;
                }
                last = reinterpret_cast<const int *>(a)[1];
                src_last = a + kFillAreaHeaderFloats + W;
            }
        }
    if (last < 0) return;   // no kept pixel in the frame: all `invalid`
    const int rg = glob_row0 + (int)blockIdx.x;
    const float *s = rg < first ? src_first : (rg > last ? src_last : nullptr);
    if (!s) return;
    float *o = out + (size_t)r * W;
    for (int c = threadIdx.x; c < W; c += 256) o[c] = s[c];
}

template <bool LR>
cudaError_t fill(const Geom &g, int frames, const Scratch &s, const GrayView &gl_glob, float *out, const LrCheck &lr,
                 cudaStream_t st) {
    dim3 block(32, 8), grid(((g.W + 3) / 4 + 31) / 32, (g.H + 7) / 8, frames);
    const bool vec_ok = (g.W % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15u) == 0);
    if (g.K == 2 && vec_ok) {
        dim3 grid2((g.W / 4 + 31) / 32, (g.Hd + 7) / 8, frames);
        fill_k2_kernel<LR><<<grid2, block, 0, st>>>(g, s.gray, gl_glob, s.refined, out, lr);
        return cudaGetLastError();
    }
    switch (g.K) {
        case 1: fill_kernel<1, LR><<<grid, block, 0, st>>>(g, s.gray, gl_glob, s.refined, out, vec_ok, lr); break;
        case 2: fill_kernel<2, LR><<<grid, block, 0, st>>>(g, s.gray, gl_glob, s.refined, out, vec_ok, lr); break;
        case 4: fill_kernel<4, LR><<<grid, block, 0, st>>>(g, s.gray, gl_glob, s.refined, out, vec_ok, lr); break;
        default: fill_kernel<0, LR><<<grid, block, 0, st>>>(g, s.gray, gl_glob, s.refined, out, vec_ok, lr); break;
    }
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_fill(const Geom &g, int frames, const Scratch &s, const GrayView &gl_glob, float *out, cudaStream_t st) {
    return fill<false>(g, frames, s, gl_glob, out, LrCheck{nullptr, 0.0f, 0.0f}, st);
}

cudaError_t launch_fill_lr(const Geom &g, int frames, const Scratch &s, const GrayView &gl_glob, float *out, const LrCheck &lr,
                           cudaStream_t st) {
    return fill<true>(g, frames, s, gl_glob, out, lr, st);
}

cudaError_t launch_lr_fill_rows(const float *left, const float *right_mirrored, int frames, int H, int W, float tolerance,
                                float invalid, float *out, unsigned char *row_kept, cudaStream_t st) {
    lr_fill_rows_kernel<true><<<(unsigned)frames * (unsigned)H, kBgThreads, 0, st>>>(left, right_mirrored, out, row_kept, W,
                                                                                    tolerance, invalid);
    return cudaGetLastError();
}

cudaError_t launch_lr_fill_cols_band(float *out, const unsigned char *row_kept, int row_first, int band_rows, int glob_row0,
                                     int W, const FillAreas &areas, cudaStream_t st) {
    lr_fill_cols_band_kernel<<<band_rows, 256, 0, st>>>(out, row_kept, row_first, glob_row0, W, areas);
    return cudaGetLastError();
}

cudaError_t launch_lr_background_fill(const float *left, const float *right, bool right_mirrored, int frames, int H, int W,
                                      float tolerance, float invalid, float *out, unsigned char *row_kept,
                                      cudaStream_t st) {
    const unsigned rows = (unsigned)frames * (unsigned)H;
    if (right_mirrored)
        lr_fill_rows_kernel<true><<<rows, kBgThreads, 0, st>>>(left, right, out, row_kept, W, tolerance, invalid);
    else
        lr_fill_rows_kernel<false><<<rows, kBgThreads, 0, st>>>(left, right, out, row_kept, W, tolerance, invalid);
    lr_fill_cols_kernel<<<rows, 256, 0, st>>>(out, row_kept, H, W);
    return cudaGetLastError();
}

}  // namespace sd
