// Reprojection to 3-D (DESIGN.md §15): exactly cv2.reprojectImageTo3D(disparity, Q, xyz, handleMissingValues) for
// float32 maps and a float64 Q, output CV_32FC3 ([n][H][W][3] floats).  Output pixel (x = column, y = row), disparity d:
//   h_k = (((0 + q_k0 x) + q_k1 y) + q_k2 d) + q_k3         k = 0..3, each operation a float64 round-to-nearest, no FMA
//   ia = 1 / h_3                                             (IEEE float64, so h_3 = 0 gives +-inf)
//   (X, Y, Z) = float32(float64(float32(h_k)) * ia)          k = 0, 1, 2 (OpenCV: Vec3f p = Vec3d(h); p /= h[3])
// The leading `0 +` is OpenCV's Matx product: it turns a -0 sum into +0.  Then every pixel with
// |float64(d) - m| <= FLT_EPSILON gets Z = 10000, where m = FLT_MAX (OpenCV's initial minimum, so this marks d = FLT_MAX
// even without handleMissingValues) or, with handleMissingValues, the frame's minimum over its non-NaN disparities (a
// frame that is all NaN keeps FLT_MAX).  Denormal float32 outputs are kept: the library builds without --ftz.
//
// One thread owns kPx adjacent pixels of one row: it forms the frame-independent prefix s_k = (0 + q_k0 x) + q_k1 y of
// its pixels once (the first two steps of the sequential order) and then loops over the frames, one float4 load of d
// and three float4 stores (48 bytes) per frame when aligned.  The minimum is a separate reduction (frame_min_kernel):
// an order-preserving uint32 key of each float and one atomicMin per block and frame.
#include <cfloat>

#include "common.cuh"

namespace sd {

namespace {

constexpr int kPx = 4;          // pixels per thread
constexpr int kThreads = 256;
constexpr int kLoads = 4;        // loads in flight per thread in frame_min_kernel
constexpr unsigned kNoMin = 0xffffffffu;   // key of a frame without a non-NaN value (the key of no float but NaN)

// monotone: a < b (non-NaN floats, -0 < +0) <=> key(a) < key(b)
__device__ __forceinline__ unsigned order_key(float v) {
    const unsigned b = __float_as_uint(v);
    return v != v ? kNoMin : (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__device__ __forceinline__ float key_value(unsigned k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// grid.y runs over the frames (strided past 65535); min_key[f] must start at kNoMin
__global__ void __launch_bounds__(kThreads) frame_min_kernel(const float *__restrict__ d, int n, long long hw, bool vec,
                                                             unsigned *__restrict__ min_key) {
    const long long stride = (long long)gridDim.x * kThreads, i0 = (long long)blockIdx.x * kThreads + threadIdx.x;
    for (int f = blockIdx.y; f < n; f += gridDim.y) {
        const float *p = d + (long long)f * hw;
        unsigned k = kNoMin;
        // kLoads independent loads per thread and pass, all in flight before the first is used
        if (vec) {
            const long long q = hw >> 2;
#pragma unroll 1
            for (long long base = i0; base < q; base += kLoads * stride) {
                float4 v[kLoads];
#pragma unroll
                for (int l = 0; l < kLoads; l++)
                    v[l] = base + l * stride < q ? __ldg((const float4 *)p + base + l * stride)
                                                 : make_float4(NAN, NAN, NAN, NAN);
#pragma unroll
                for (int l = 0; l < kLoads; l++)
                    k = min(min(k, order_key(v[l].x)), min(order_key(v[l].y), min(order_key(v[l].z), order_key(v[l].w))));
            }
        } else {
#pragma unroll 1
            for (long long base = i0; base < hw; base += kLoads * stride) {
                float v[kLoads];
#pragma unroll
                for (int l = 0; l < kLoads; l++) v[l] = base + l * stride < hw ? __ldg(p + base + l * stride) : NAN;
#pragma unroll
                for (int l = 0; l < kLoads; l++) k = min(k, order_key(v[l]));
            }
        }
        // one atomic per block: same-address atomics serialise in L2, one per warp cost ~3 us per 1080p frame
        __shared__ unsigned warp_min[kThreads / 32];
        k = __reduce_min_sync(0xffffffffu, k);
        if ((threadIdx.x & 31) == 0) warp_min[threadIdx.x >> 5] = k;
        __syncthreads();
        if (threadIdx.x < 32) {
            k = __reduce_min_sync(0xffffffffu, threadIdx.x < kThreads / 32 ? warp_min[threadIdx.x] : kNoMin);
            if (threadIdx.x == 0 && k != kNoMin) atomicMin(min_key + f, k);
        }
        __syncthreads();   // warp_min is reused by the next frame
    }
}

// (X, Y, Z) of one pixel from its prefixes s[0..3] and disparity d
__device__ __forceinline__ void point(const ReprojectQ &Q, const double *s, float d, float *o) {
    const double dd = (double)d;
    double h[4];
#pragma unroll
    for (int k = 0; k < 4; k++) h[k] = __dadd_rn(__dadd_rn(s[k], __dmul_rn(Q.q[4 * k + 2], dd)), Q.q[4 * k + 3]);
    const double ia = __drcp_rn(h[3]);   // the correctly rounded 1 / h_3, as the division
#pragma unroll
    for (int k = 0; k < 3; k++) o[k] = __double2float_rn(__dmul_rn((double)__double2float_rn(h[k]), ia));
}

// vec: W % kPx == 0 and both buffers 16-byte aligned, so every thread's kPx pixels load as one float4 and store as
// three; min_key: [n] keys of frame_min_kernel, or NULL without handleMissingValues
__global__ void __launch_bounds__(kThreads) reproject_kernel(const float *__restrict__ disp, float *__restrict__ xyz, int n,
                                                             int H, int W, ReprojectQ Q,
                                                             const unsigned *__restrict__ min_key, bool vec) {
    const int wq = (W + kPx - 1) / kPx;
    const long long t = (long long)blockIdx.x * kThreads + threadIdx.x;
    if (t >= (long long)H * wq) return;
    const int y = (int)(t / wq), c0 = (int)(t % wq) * kPx;
    const int m = W - c0 < kPx ? W - c0 : kPx;
    double s[kPx][4];
#pragma unroll
    for (int j = 0; j < kPx; j++)
#pragma unroll
        for (int k = 0; k < 4; k++)
            s[j][k] = __dadd_rn(__dadd_rn(0.0, __dmul_rn(Q.q[4 * k], (double)(c0 + j))), __dmul_rn(Q.q[4 * k + 1], (double)y));
    const long long hw = (long long)H * W, i0 = (long long)y * W + c0;
    const float *dp = disp + i0;
    float *op = xyz + 3 * i0;
    for (int f = 0; f < n; f++, dp += hw, op += 3 * hw) {
        float d[kPx];
        if (vec) {
            const float4 v = __ldg((const float4 *)dp);
            d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
        } else {
#pragma unroll
            for (int j = 0; j < kPx; j++) d[j] = j < m ? __ldg(dp + j) : 0.f;
        }
        float o[3 * kPx];
#pragma unroll
        for (int j = 0; j < kPx; j++) point(Q, s[j], d[j], o + 3 * j);
        if (min_key) {
            const unsigned k = __ldg(min_key + f);
            const float mf = k == kNoMin ? FLT_MAX : key_value(k);
            // every non-NaN d of the frame is >= m, and a d that passes the float64 test lies below m + FLT_EPSILON *
            // (1 + 2^-53) < m + 1, so d <= float32(m + 1) is a float pre-test and the float64 one runs on its few hits
            const float hi = mf + 1.f;
            const double mn = (double)mf;
#pragma unroll
            for (int j = 0; j < kPx; j++)
                if (d[j] <= hi && fabs(__dsub_rn((double)d[j], mn)) <= (double)FLT_EPSILON) o[3 * j + 2] = 10000.f;
        } else {   // m = FLT_MAX: the float32 values next to it lie 2^104 away, so the test is d == FLT_MAX
#pragma unroll
            for (int j = 0; j < kPx; j++)
                if (d[j] == FLT_MAX) o[3 * j + 2] = 10000.f;
        }
        if (vec) {
            float4 *q = (float4 *)op;
            q[0] = make_float4(o[0], o[1], o[2], o[3]);
            q[1] = make_float4(o[4], o[5], o[6], o[7]);
            q[2] = make_float4(o[8], o[9], o[10], o[11]);
        } else {
#pragma unroll
            for (int j = 0; j < 3 * kPx; j++)
                if (j < 3 * m) op[j] = o[j];
        }
    }
}

bool aligned16(const void *p) { return ((uintptr_t)p & 15) == 0; }

}  // namespace

cudaError_t launch_reproject(const float *disp, int n, int H, int W, const ReprojectQ &Q, unsigned *min_key, float *xyz,
                             cudaStream_t st) {
    const long long hw = (long long)H * W;
    if (min_key) {
        cudaError_t e = cudaMemsetAsync(min_key, 0xff, (size_t)n * sizeof(unsigned), st);
        if (e != cudaSuccess) return e;
        const bool vec = hw % 4 == 0 && aligned16(disp);
        const long long per = (long long)kThreads * kLoads * (vec ? 4 : 1);   // one pass of kLoads loads per thread
        const unsigned bx = (unsigned)(hw + per - 1 < (long long)65535 * per ? (hw + per - 1) / per : 65535);
        frame_min_kernel<<<dim3(bx, n < 65535 ? n : 65535), kThreads, 0, st>>>(disp, n, hw, vec, min_key);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    const long long threads = (long long)H * ((W + kPx - 1) / kPx);
    const bool vec = W % kPx == 0 && aligned16(disp) && aligned16(xyz);
    reproject_kernel<<<(unsigned)((threads + kThreads - 1) / kThreads), kThreads, 0, st>>>(disp, xyz, n, H, W, Q, min_key,
                                                                                          vec);
    return cudaGetLastError();
}

}  // namespace sd
