// Rectification remap (DESIGN.md §14): exactly cv2.remap(src, map_x, map_y, INTER_LINEAR, BORDER_CONSTANT, 0) with
// CV_32FC1 maps, for uint8 and float32 planes.  Output pixel (r, c) samples the source at (map_x[r,c], map_y[r,c]):
//   ix = rint(x * 32) (half to even), x0 = ix >> 5, fx = ix & 31; the same for y.  A NaN coordinate samples nothing.
//   taps (y0,x0) (y0,x0+1) (y0+1,x0) (y0+1,x0+1) with weights (1-ay)(1-ax), (1-ay)ax, ay(1-ax), ay ax, a = f/32;
//   a tap outside [0,W) x [0,H) reads 0 and keeps its weight.
//   uint8: fixed-point weights rint(c * 32768), out = (sum w_k p_k + 2^14) >> 15.  The products of two multiples of 1/32
//          are exact in fp32, so rint(c * 32768) = 32 (32-fy)(32-fx) etc. and the four always sum to 32768: OpenCV's
//          correction of the largest weight never applies and the weights are computed in integers here.
//   float32: ((c0 p00 + c1 p01) + c2 p10) + c3 p11, every operation rounded (OpenCV's order; no FMA).
// __float2int_rn saturates where OpenCV saturates the tap to a short: for H, W < 32768 (sd_set_rectification and
// sd_rectify refuse larger images) both put every tap of a huge or infinite coordinate outside the image.
//
// One thread owns kPx adjacent output pixels (linear index within the [H][W] plane) of one view: it converts its map
// entries to a tap offset, an in-image mask and the weights once, then loops over all planes of the launch (the frames
// of a chunk times their 3 channels), gathering 4 taps per pixel.  So the maps are read once per launch, and adjacent
// threads gather adjacent source columns (L1 / L2 hits).
#include "common.cuh"

namespace sd {

namespace {

constexpr int kPx = 4;          // output pixels per thread
constexpr int kThreads = 256;

struct Taps {
    int off;        // y0 * W + x0 (the first tap; may lie outside the plane)
    unsigned mask;  // bit k: tap k (00, 01, 10, 11) lies inside the image
    int fx, fy;
};

__device__ __forceinline__ Taps make_taps(float x, float y, int H, int W) {
    Taps t;
    const int ix = __float2int_rn(__fmul_rn(x, 32.f)), iy = __float2int_rn(__fmul_rn(y, 32.f));
    const int x0 = ix >> 5, y0 = iy >> 5;
    t.fx = ix & 31;
    t.fy = iy & 31;
    const bool in_x0 = (unsigned)x0 < (unsigned)W, in_x1 = (unsigned)(x0 + 1) < (unsigned)W;
    const bool in_y0 = (unsigned)y0 < (unsigned)H, in_y1 = (unsigned)(y0 + 1) < (unsigned)H;
    const bool nan = (x != x) || (y != y);
    t.mask = nan ? 0u : ((in_y0 && in_x0) | ((in_y0 && in_x1) << 1) | ((in_y1 && in_x0) << 2) | ((in_y1 && in_x1) << 3));
    t.off = t.mask ? y0 * W + x0 : 0;   // (only formed for a tap inside: then |y0|, |x0| < 32768)
    return t;
}

template <typename T>
__device__ __forceinline__ float tap(const T *__restrict__ p, const Taps &t, int k, int d) {
    return (t.mask >> k & 1u) ? (float)__ldg(p + t.off + d) : 0.f;
}

template <typename T> struct Weights;

template <> struct Weights<unsigned char> {
    int w[4];
    __device__ __forceinline__ explicit Weights(const Taps &t) {
        w[0] = 32 * (32 - t.fy) * (32 - t.fx);
        w[1] = 32 * (32 - t.fy) * t.fx;
        w[2] = 32 * t.fy * (32 - t.fx);
        w[3] = 32 * t.fy * t.fx;
    }
    __device__ __forceinline__ unsigned char apply(const unsigned char *__restrict__ p, const Taps &t, int W) const {
        auto tp = [&](int k, int d) { return (t.mask >> k & 1u) ? (int)__ldg(p + t.off + d) : 0; };
        const int acc = w[0] * tp(0, 0) + w[1] * tp(1, 1) + w[2] * tp(2, W) + w[3] * tp(3, W + 1);
        return (unsigned char)((acc + (1 << 14)) >> 15);   // (0 <= acc <= 255 * 32768: no clamp needed)
    }
};

template <> struct Weights<float> {
    float c[4];
    __device__ __forceinline__ explicit Weights(const Taps &t) {
        const float ax = t.fx * (1.f / 32.f), ay = t.fy * (1.f / 32.f);
        c[0] = __fmul_rn(1.f - ay, 1.f - ax);
        c[1] = __fmul_rn(1.f - ay, ax);
        c[2] = __fmul_rn(ay, 1.f - ax);
        c[3] = __fmul_rn(ay, ax);
    }
    __device__ __forceinline__ float apply(const float *__restrict__ p, const Taps &t, int W) const {
        const float s = __fadd_rn(__fmul_rn(c[0], tap(p, t, 0, 0)), __fmul_rn(c[1], tap(p, t, 1, 1)));
        return __fadd_rn(__fadd_rn(s, __fmul_rn(c[2], tap(p, t, 2, W))), __fmul_rn(c[3], tap(p, t, 3, W + 1)));
    }
};

template <typename T> struct Vec4;
template <> struct Vec4<unsigned char> { using type = uchar4; };
template <> struct Vec4<float> { using type = float4; };

// grid.y = view; `vec`: the maps and every output plane of every view start kPx-element aligned, so loads of the maps
// and stores of the output go kPx at a time (the gathers are scalar)
template <typename T>
__global__ void __launch_bounds__(kThreads) rectify_kernel(RectifyViews v, int planes, int H, int W, bool vec) {
    const RectifyView rv = blockIdx.y ? v.view[1] : v.view[0];   // (not view[blockIdx.y]: that copies the parameters to the stack)
    const long long n = (long long)H * W;
    const long long i0 = ((long long)blockIdx.x * kThreads + threadIdx.x) * kPx;
    if (i0 >= n) return;
    const int m = n - i0 < kPx ? (int)(n - i0) : kPx;
    const bool full = vec && m == kPx;
    float mx[kPx], my[kPx];
    if (full) {
        const float4 a = __ldg((const float4 *)(rv.map_x + i0)), b = __ldg((const float4 *)(rv.map_y + i0));
        mx[0] = a.x; mx[1] = a.y; mx[2] = a.z; mx[3] = a.w;
        my[0] = b.x; my[1] = b.y; my[2] = b.z; my[3] = b.w;
    } else {
#pragma unroll
        for (int k = 0; k < kPx; k++) {
            mx[k] = k < m ? __ldg(rv.map_x + i0 + k) : __int_as_float(0x7fc00000);
            my[k] = k < m ? __ldg(rv.map_y + i0 + k) : 0.f;
        }
    }
    Taps t[kPx];
#pragma unroll
    for (int k = 0; k < kPx; k++) t[k] = make_taps(mx[k], my[k], H, W);
    Weights<T> w[kPx] = {Weights<T>(t[0]), Weights<T>(t[1]), Weights<T>(t[2]), Weights<T>(t[3])};
    const T *src = (const T *)rv.src;
    T *dst = (T *)rv.dst + i0;
    for (int p = 0; p < planes; p++, src += n, dst += n) {
        T o[kPx];
#pragma unroll
        for (int k = 0; k < kPx; k++) o[k] = w[k].apply(src, t[k], W);
        if (full) {
            typename Vec4<T>::type q;
            q.x = o[0]; q.y = o[1]; q.z = o[2]; q.w = o[3];
            *(typename Vec4<T>::type *)dst = q;
        } else {
#pragma unroll
            for (int k = 0; k < kPx; k++)
                if (k < m) dst[k] = o[k];
        }
    }
}

bool aligned(const void *p, size_t a) { return ((uintptr_t)p & (a - 1)) == 0; }

}  // namespace

cudaError_t launch_rectify(const RectifyViews &v, int n_views, int dtype, int planes, int H, int W, cudaStream_t st) {
    const long long n = (long long)H * W;
    const size_t esize = dtype == SD_U8 ? 1 : 4;
    bool vec = n % kPx == 0;
    for (int i = 0; i < n_views; i++)
        vec = vec && aligned(v.view[i].map_x, 16) && aligned(v.view[i].map_y, 16) && aligned(v.view[i].dst, kPx * esize);
    const dim3 grid((unsigned)((n + (long long)kThreads * kPx - 1) / ((long long)kThreads * kPx)), n_views);
    if (dtype == SD_U8) rectify_kernel<unsigned char><<<grid, kThreads, 0, st>>>(v, planes, H, W, vec);
    else rectify_kernel<float><<<grid, kThreads, 0, st>>>(v, planes, H, W, vec);
    return cudaGetLastError();
}

}  // namespace sd
