// Kernel A: fused RGB->gray (both views) + KxK mean pool.  HBM-bound streaming kernel.
//
// Reference semantics reproduced bit for bit:
//   gray  = fma(B, 0.1140f, fma(R, 0.2989f, G * 0.5870f))       rgb_to_grayscale.cu:24-28 as compiled
//           (nvcc contracts R+G+B of the source into FMUL, FFMA, FFMA -- oracle/_ref/reference_sass.txt)
//   pool  = (((0 + g00) + g01) + g10 ...) / float(K*K)           mean_pool.cu:25-35 (row-major taps, IEEE divide)
// One launch handles every frame of the chunk and both views (blockIdx.z = frame*2 + side).
// Input is the CHW uint8 image a camera delivers, or the float32 CHW tensor the reference's
// `.float()` produces (cuda_stereo_matching_backend.py:14-15); uint8 -> float is exact.
#include "common.cuh"

namespace sd {
namespace {

__device__ __forceinline__ float gray_px(float r, float g, float b) {
    float t = __fmul_rn(g, 0.5870f);
    t = __fmaf_rn(r, 0.2989f, t);
    return __fmaf_rn(b, 0.1140f, t);
}

template <typename T>
__device__ __forceinline__ float ld_px(const T *p) {
    return (float)__ldg(p);
}

// MIRRORED frames (left-right check, api.cu): frames >= nfwd are the pair (flip R, flip L) of caller frame
// frame - nfwd, read straight from the caller's input -- views swapped, columns reversed.  Everything is then computed
// in the mirrored image's own coordinates, so gray, pooled sums (tap order included) and the SAFE clamp are those of the
// flipped image.  frames < nfwd are the ordinary forward frames.  With the check off the kernels are instantiated with
// MIRROR = false: the code of the forward-only path is unchanged.
template <bool MIRROR, typename T>
__device__ __forceinline__ const T *frame_view(const T *left, const T *right, int frame, int side, int nfwd,
                                               size_t plane, bool &mir) {
    mir = MIRROR && frame >= nfwd;
    return ((side != 0) != mir ? right : left) + (size_t)(mir ? frame - nfwd : frame) * 3 * plane;
}

// ---- generic path: any K, any size; one thread per pooled pixel ---------------------------------
template <typename T, bool MIRROR>
__global__ void __launch_bounds__(256) gray_pool_generic(const T *__restrict__ left, const T *__restrict__ right,
                                                         float *__restrict__ gray, float *__restrict__ pool,
                                                         int H, int W, int K, int Hd, int Wd, int nfwd) {
    const int y = blockIdx.x * blockDim.x + threadIdx.x;
    const int x = blockIdx.y * blockDim.y + threadIdx.y;
    const int frame = blockIdx.z >> 1, side = blockIdx.z & 1;
    if (x >= Hd || y >= Wd) return;
    const size_t plane = (size_t)H * W;
    bool mir;
    const T *img = frame_view<MIRROR>(left, right, frame, side, nfwd, plane, mir);
    float *g = gray + ((size_t)frame * 2 + side) * plane;
    float s = 0.0f;
    for (int i = 0; i < K; i++) {
        for (int j = 0; j < K; j++) {
            int r = x * K + i, c = y * K + j;
            const bool inside = (r < H) && (c < W);
            r = min(r, H - 1);  // SAFE definition where the reference reads past the image (H % K != 0)
            c = min(c, W - 1);
            const size_t o = (size_t)r * W + c;
            const size_t oi = mir ? (size_t)r * W + (W - 1 - c) : o;   // (the clamp above is in mirrored coordinates)
            const float v = gray_px(ld_px(img + oi), ld_px(img + plane + oi), ld_px(img + 2 * plane + oi));
            if (inside) g[o] = v;
            s = __fadd_rn(s, v);
        }
    }
    pool[((size_t)frame * 2 + side) * Hd * Wd + (size_t)x * Wd + y] = __fdiv_rn(s, (float)(K * K));
}

// ---- K = 2 fast paths: 128-bit loads and stores ------------------------------------------------
// uint8: a thread owns 2 rows x 16 columns: 6 x LDG.128 in, 8 x STG.128 gray + 2 x STG.128 pooled out.
// A mirrored frame's group [16cx, 16cx+16) is the input's [W-16cx-16, W-16cx) (16-byte aligned since W % 16 == 0),
// byte-reversed in registers.
template <bool MIRROR>
__global__ void __launch_bounds__(256) gray_pool_k2_u8(const uint8_t *__restrict__ left, const uint8_t *__restrict__ right,
                                                       float *__restrict__ gray, float *__restrict__ pool,
                                                       int H, int W, int Hd, int Wd, int nfwd) {
    const int cx = blockIdx.x * blockDim.x + threadIdx.x;  // 16-column group
    const int x = blockIdx.y * blockDim.y + threadIdx.y;   // pooled row
    const int frame = blockIdx.z >> 1, side = blockIdx.z & 1;
    if (x >= Hd || cx * 16 >= W) return;
    const size_t plane = (size_t)H * W;
    bool mir;
    const uint8_t *img = frame_view<MIRROR>(left, right, frame, side, nfwd, plane, mir);
    float *g = gray + ((size_t)frame * 2 + side) * plane;
    const size_t o0 = (size_t)(2 * x) * W + cx * 16;
    const size_t i0 = mir ? (size_t)(2 * x) * W + (W - 16 * cx - 16) : o0;
    uint4 v[2][3];
#pragma unroll
    for (int i = 0; i < 2; i++)
#pragma unroll
        for (int c = 0; c < 3; c++) v[i][c] = __ldg(reinterpret_cast<const uint4 *>(img + c * plane + i0 + (size_t)i * W));
    if (mir) {
#pragma unroll
        for (int i = 0; i < 2; i++)
#pragma unroll
            for (int c = 0; c < 3; c++) {
                const uint4 t = v[i][c];
                v[i][c] = make_uint4(__byte_perm(t.w, 0, 0x0123), __byte_perm(t.z, 0, 0x0123), __byte_perm(t.y, 0, 0x0123),
                                     __byte_perm(t.x, 0, 0x0123));
            }
    }
    float gr[2][16];
#pragma unroll
    for (int i = 0; i < 2; i++) {
        const uint32_t *rw = &v[i][0].x, *gw = &v[i][1].x, *bw = &v[i][2].x;
#pragma unroll
        for (int k = 0; k < 16; k++) {
            const float r = (float)((rw[k >> 2] >> (8 * (k & 3))) & 0xffu);
            const float gg = (float)((gw[k >> 2] >> (8 * (k & 3))) & 0xffu);
            const float b = (float)((bw[k >> 2] >> (8 * (k & 3))) & 0xffu);
            gr[i][k] = gray_px(r, gg, b);
        }
        float4 *dst = reinterpret_cast<float4 *>(g + o0 + (size_t)i * W);
#pragma unroll
        for (int q = 0; q < 4; q++) dst[q] = make_float4(gr[i][4 * q], gr[i][4 * q + 1], gr[i][4 * q + 2], gr[i][4 * q + 3]);
    }
    float p[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
        float s = __fadd_rn(0.0f, gr[0][2 * k]);
        s = __fadd_rn(s, gr[0][2 * k + 1]);
        s = __fadd_rn(s, gr[1][2 * k]);
        s = __fadd_rn(s, gr[1][2 * k + 1]);
        p[k] = __fmul_rn(s, 0.25f);  // == s / 4.0f exactly
    }
    float4 *pd = reinterpret_cast<float4 *>(pool + ((size_t)frame * 2 + side) * Hd * Wd + (size_t)x * Wd + cx * 8);
    pd[0] = make_float4(p[0], p[1], p[2], p[3]);
    pd[1] = make_float4(p[4], p[5], p[6], p[7]);
}

// float32: a thread owns 2 rows x 8 columns: 12 x LDG.128 in, 4 x STG.128 gray + 1 x STG.128 pooled out.
// Mirrored frames as in the uint8 path: input columns [W-8cx-8, W-8cx) (W % 8 == 0), reversed in registers.
template <bool MIRROR>
__global__ void __launch_bounds__(256) gray_pool_k2_f32(const float *__restrict__ left, const float *__restrict__ right,
                                                        float *__restrict__ gray, float *__restrict__ pool,
                                                        int H, int W, int Hd, int Wd, int nfwd) {
    const int cx = blockIdx.x * blockDim.x + threadIdx.x;  // 8-column group
    const int x = blockIdx.y * blockDim.y + threadIdx.y;
    const int frame = blockIdx.z >> 1, side = blockIdx.z & 1;
    if (x >= Hd || cx * 8 >= W) return;
    const size_t plane = (size_t)H * W;
    bool mir;
    const float *img = frame_view<MIRROR>(left, right, frame, side, nfwd, plane, mir);
    float *g = gray + ((size_t)frame * 2 + side) * plane;
    const size_t o0 = (size_t)(2 * x) * W + cx * 8;
    const size_t i0 = mir ? (size_t)(2 * x) * W + (W - 8 * cx - 8) : o0;
    float4 v[2][3][2];
#pragma unroll
    for (int i = 0; i < 2; i++)
#pragma unroll
        for (int c = 0; c < 3; c++)
#pragma unroll
            for (int q = 0; q < 2; q++)
                v[i][c][q] = __ldg(reinterpret_cast<const float4 *>(img + c * plane + i0 + (size_t)i * W) + q);
    float gr[2][8];
#pragma unroll
    for (int i = 0; i < 2; i++) {
#pragma unroll
        for (int q = 0; q < 2; q++) {
            gr[i][4 * q + 0] = gray_px(v[i][0][q].x, v[i][1][q].x, v[i][2][q].x);
            gr[i][4 * q + 1] = gray_px(v[i][0][q].y, v[i][1][q].y, v[i][2][q].y);
            gr[i][4 * q + 2] = gray_px(v[i][0][q].z, v[i][1][q].z, v[i][2][q].z);
            gr[i][4 * q + 3] = gray_px(v[i][0][q].w, v[i][1][q].w, v[i][2][q].w);
        }
        if (mir) {   // (gray is per pixel: reversing the gray values == reversing the input)
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const float t = gr[i][k];
                gr[i][k] = gr[i][7 - k];
                gr[i][7 - k] = t;
            }
        }
        float4 *dst = reinterpret_cast<float4 *>(g + o0 + (size_t)i * W);
        dst[0] = make_float4(gr[i][0], gr[i][1], gr[i][2], gr[i][3]);
        dst[1] = make_float4(gr[i][4], gr[i][5], gr[i][6], gr[i][7]);
    }
    float p[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        float s = __fadd_rn(0.0f, gr[0][2 * k]);
        s = __fadd_rn(s, gr[0][2 * k + 1]);
        s = __fadd_rn(s, gr[1][2 * k]);
        s = __fadd_rn(s, gr[1][2 * k + 1]);
        p[k] = __fmul_rn(s, 0.25f);
    }
    *reinterpret_cast<float4 *>(pool + ((size_t)frame * 2 + side) * Hd * Wd + (size_t)x * Wd + cx * 4) =
        make_float4(p[0], p[1], p[2], p[3]);
}

// Wrap-padded copies of the pooled planes (PadGeom in common.cuh).  A thread writes 4 consecutive padded
// columns (STG.128) of one row of one view; the wrap is one conditional add/sub in the common case.
__device__ __forceinline__ int wrap_near(int i, int n) {
    if (i < 0) i += n;
    else if (i >= n) i -= n;
    return ((unsigned)i < (unsigned)n) ? i : wrapm(i, n);  // images narrower than the padding: true modulo
}

__global__ void __launch_bounds__(256) pad_pooled_kernel(const float *__restrict__ pool, float *__restrict__ padl,
                                                         float *__restrict__ padr, int Hd, int Wd, PadGeom pg,
                                                         int *__restrict__ range_flag, int range_epoch) {
    const int c4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const int r = blockIdx.y;
    const int frame = blockIdx.z >> 1, side = blockIdx.z & 1;
    const int pw = side ? pg.pwr : pg.pwl;   // multiples of 4
    if (c4 >= pw) return;
    const float *src = pool + ((size_t)frame * 2 + side) * Hd * Wd + (size_t)wrap_near(r - 11, Hd) * Wd;
    const int vc = c4 - (side ? pg.shift_r : 15);
    float4 v;
    v.x = __ldg(src + wrap_near(vc, Wd));
    v.y = __ldg(src + wrap_near(vc + 1, Wd));
    v.z = __ldg(src + wrap_near(vc + 2, Wd));
    v.w = __ldg(src + wrap_near(vc + 3, Wd));
    *reinterpret_cast<float4 *>((side ? padr : padl) + ((size_t)frame * pg.rows + r) * pw + c4) = v;
    // The level screen's error bound needs every similarity tap 255-|l-r| to be >= 0: flag pooled values outside
    // [0,255] (NaN fails the comparison too).  Cannot happen with uint8 images.
    if (range_flag) {
        const float mn = fminf(fminf(v.x, v.y), fminf(v.z, v.w)), mx = fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w));
        const bool nan = (v.x != v.x) || (v.y != v.y) || (v.z != v.z) || (v.w != v.w);
        if (nan || !(mn >= 0.0f) || !(mx <= 255.0f)) *range_flag = range_epoch;
    }
}

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }


template <bool MIRROR>
cudaError_t gray_pool(const Geom &g, const void *left, const void *right, int dtype, int frames, const Scratch &s,
                      cudaStream_t st, int nfwd) {
    const bool even = (g.K == 2) && (g.H % 2 == 0) && aligned16(left) && aligned16(right) &&
                      aligned16(s.gray) && aligned16(s.pool);
    if (even && dtype == SD_U8 && g.W % 16 == 0) {
        dim3 block(32, 8), grid((g.W / 16 + 31) / 32, (g.Hd + 7) / 8, frames * 2);
        gray_pool_k2_u8<MIRROR><<<grid, block, 0, st>>>((const uint8_t *)left, (const uint8_t *)right, s.gray, s.pool,
                                                        g.H, g.W, g.Hd, g.Wd, nfwd);
    } else if (even && dtype == SD_F32 && g.W % 8 == 0) {
        dim3 block(32, 8), grid((g.W / 8 + 31) / 32, (g.Hd + 7) / 8, frames * 2);
        gray_pool_k2_f32<MIRROR><<<grid, block, 0, st>>>((const float *)left, (const float *)right, s.gray, s.pool,
                                                         g.H, g.W, g.Hd, g.Wd, nfwd);
    } else {
        dim3 block(32, 8), grid((g.Wd + 31) / 32, (g.Hd + 7) / 8, frames * 2);
        if (dtype == SD_U8)
            gray_pool_generic<uint8_t, MIRROR><<<grid, block, 0, st>>>((const uint8_t *)left, (const uint8_t *)right,
                                                                       s.gray, s.pool, g.H, g.W, g.K, g.Hd, g.Wd, nfwd);
        else
            gray_pool_generic<float, MIRROR><<<grid, block, 0, st>>>((const float *)left, (const float *)right, s.gray,
                                                                     s.pool, g.H, g.W, g.K, g.Hd, g.Wd, nfwd);
    }
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_gray_pool(const Geom &g, const void *left, const void *right, int dtype, int frames,
                             const Scratch &s, cudaStream_t st, int mirrored) {
    return mirrored > 0 ? gray_pool<true>(g, left, right, dtype, frames, s, st, frames - mirrored)
                        : gray_pool<false>(g, left, right, dtype, frames, s, st, frames);
}

cudaError_t launch_pad_pooled(const Geom &g, int frames, const Scratch &s, cudaStream_t st) {
    const PadGeom pg = make_pad_geom(g.Hd, g.Wd, g.L, g.min_ds);
    const int pw = pg.pwl > pg.pwr ? pg.pwl : pg.pwr;
    dim3 grid((pw / 4 + 255) / 256, pg.rows, frames * 2);
    pad_pooled_kernel<<<grid, 256, 0, st>>>(s.pool, s.padl, s.padr, g.Hd, g.Wd, pg, s.range_flag, s.range_epoch);
    return cudaGetLastError();
}

}  // namespace sd
