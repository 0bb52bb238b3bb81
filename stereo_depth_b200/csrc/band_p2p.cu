// Row-band mode over peer memory (NVLink / NVSwitch): the two exchange steps of a banded frame as kernels that store
// straight into the neighbours' HBM and signal with system-scope flags -- no NCCL call, no staging copy, no host sync.
//
//   band_scatter_kernel   my raw band rows -> my own window, and my first / last `halo` rows -> the bottom / top halo
//                         of the previous / next rank's window (the ring is closed: the reference's row padding is
//                         circular, device_functions.cuh:13-14).  The last block to finish releases the two flags.
//   publish_gray_kernel   my left gray band -> my published buffer (double buffered by frame parity); the last block
//                         releases one flag at every peer.  The fill kernel then reads the one row it needs,
//                         GL[(K+1)x] (upscale_disparity_vertical_fill.cu:31), from whichever rank owns it.  With the
//                         left-right check it publishes the mirrored frame's left gray band too (second plane).
//   publish_fill_bounds_kernel  (background fill of the check only) my band's first / last row that kept a pixel and
//                         copies of those two rows -> my fill area (double buffered by frame parity); the last block
//                         releases one flag at every peer.  The column pass then applies the frame's global rule.
//   wait_flags_kernel     one warp spins (ld.acquire.sys) until the flags it is given reach the frame's epoch.
//
// Ordering argument (why single windows, two gray buffers and two fill areas suffice) is in DESIGN.md section 8.
#include "common.cuh"

namespace sd {
namespace {

__device__ __forceinline__ void st_release_sys(unsigned *p, unsigned v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Block-wide "I am the last block of this launch": every block fences its peer stores first.
__device__ __forceinline__ bool last_block_done(unsigned *counter, unsigned nblocks) {
    __shared__ unsigned s_last;
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0 && threadIdx.y == 0) {
        const unsigned old = atomicAdd(counter, 1u);
        s_last = (old == nblocks - 1) ? 1u : 0u;
        if (s_last) {
            __threadfence_system();   // acquire side: everything the other blocks fenced before their increment
            *counter = 0u;            // ready for the next launch (stream ordered)
        }
    }
    __syncthreads();
    return s_last != 0u;
}

// One thread moves 16 bytes.  Rows are [view][channel][row] of `row_bytes` bytes (a multiple of 16).
__global__ void __launch_bounds__(256) band_scatter_kernel(const uint4 *__restrict__ left, const uint4 *__restrict__ right,
                                                           uint4 *own_l, uint4 *own_r, uint4 *prev_l, uint4 *prev_r,
                                                           uint4 *next_l, uint4 *next_r, int row_vec, int band_rows, int halo,
                                                           int own_rows, int prev_rows, int next_rows, unsigned *counter,
                                                           unsigned *flag_at_prev, unsigned *flag_at_next, unsigned epoch) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;   // 16-byte column
    const int r = blockIdx.y;                              // band row
    const int vc = blockIdx.z;                             // view * 3 + channel
    if (v < row_vec) {
        const int view = vc / 3, ch = vc % 3;
        const uint4 val = __ldg((view ? right : left) + ((size_t)ch * band_rows + r) * row_vec + v);
        uint4 *own = view ? own_r : own_l, *prv = view ? prev_r : prev_l, *nxt = view ? next_r : next_l;
        own[((size_t)ch * own_rows + halo + r) * row_vec + v] = val;
        // my first rows are the previous rank's bottom halo, my last rows the next rank's top halo
        if (r < halo) prv[((size_t)ch * prev_rows + (prev_rows - halo) + r) * row_vec + v] = val;
        if (r >= band_rows - halo) nxt[((size_t)ch * next_rows + (r - (band_rows - halo))) * row_vec + v] = val;
    }
    if (last_block_done(counter, gridDim.x * gridDim.y * gridDim.z) && threadIdx.x == 0) {
        st_release_sys(flag_at_prev, epoch);
        st_release_sys(flag_at_next, epoch);
    }
}

struct PeerFlags {
    unsigned *p[8];
    int n;
};

// (planes > 1 with the left-right check: the forward and the mirrored frame's left gray band, strides in float4)
__global__ void __launch_bounds__(256) publish_gray_kernel(const float4 *__restrict__ src, float4 *__restrict__ dst, size_t n4,
                                                           unsigned *counter, PeerFlags peers, unsigned epoch, int planes,
                                                           size_t src_plane4, size_t dst_plane4) {
    for (int pl = 0; pl < planes; pl++)
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x)
            dst[pl * dst_plane4 + i] = __ldg(src + pl * src_plane4 + i);
    if (last_block_done(counter, gridDim.x) && threadIdx.x < peers.n) st_release_sys(peers.p[threadIdx.x], epoch);
}

// Fill-bounds exchange (background fill of the left-right check, DESIGN.md §13): block (x, y) copies segment x of the
// band's first (y = 0) or last (y = 1) row that kept a pixel; every block finds the two rows itself from the band's row
// flags (a few hundred bytes).  Block (0, 0) writes their global rows; the last block releases one flag at every peer.
__global__ void __launch_bounds__(256) publish_fill_bounds_kernel(const unsigned char *__restrict__ row_kept,
                                                                  const float *__restrict__ rows, int band_rows, int glob_row0,
                                                                  int W, float *area, unsigned *counter, PeerFlags peers,
                                                                  unsigned epoch) {
    __shared__ int sh_first[8], sh_last[8];
    int first = 0x7fffffff, last = -1;
    for (int i = threadIdx.x; i < band_rows; i += 256)
        if (row_kept[i]) {
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
    if (last >= 0) {
        const float *s = rows + (size_t)(blockIdx.y ? last : first) * W;
        float *d = area + kFillAreaHeaderFloats + (size_t)blockIdx.y * W;
        for (int c = blockIdx.x * 256 + threadIdx.x; c < W; c += gridDim.x * 256) d[c] = s[c];
    }
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {
        reinterpret_cast<int *>(area)[0] = last >= 0 ? glob_row0 + first : -1;
        reinterpret_cast<int *>(area)[1] = last >= 0 ? glob_row0 + last : -1;
    }
    if (last_block_done(counter, gridDim.x * gridDim.y) && threadIdx.x < peers.n) st_release_sys(peers.p[threadIdx.x], epoch);
}

// A missing peer must neither hang the GPU nor poison the CUDA context: after ~10 s the waiting lane posts
// {epoch, flag index + 1} to a mapped host word and gives up (the frame's result is then garbage); the host reports it as
// an error on the next sd_band_p2p_compute / sd_band_p2p_status call.
__global__ void wait_flags_kernel(const unsigned *flags, int first, int count, unsigned epoch, unsigned long long *timeout_word) {
    const int i = threadIdx.x;
    if (i < count) {
        const long long t0 = clock64();
        // epochs wrap after 2^32 frames; the signed difference keeps the comparison valid across the wrap
        while ((int)(ld_acquire_sys(flags + first + i) - epoch) < 0) {
            __nanosleep(200);
            if (clock64() - t0 > (20ll << 30)) {
                if (timeout_word) *reinterpret_cast<volatile unsigned long long *>(timeout_word) =
                    ((unsigned long long)epoch << 32) | (unsigned)(first + i + 1);
                else __trap();
                break;
            }
        }
    }
}

}  // namespace

cudaError_t launch_band_scatter(const void *left, const void *right, void *own_l, void *own_r, void *prev_l, void *prev_r,
                                void *next_l, void *next_r, int row_bytes, int band_rows, int halo, int own_rows, int prev_rows,
                                int next_rows, unsigned *counter, unsigned *flag_at_prev, unsigned *flag_at_next, unsigned epoch,
                                cudaStream_t st) {
    const int row_vec = row_bytes / 16;
    dim3 grid((row_vec + 255) / 256, band_rows, 6);
    band_scatter_kernel<<<grid, 256, 0, st>>>((const uint4 *)left, (const uint4 *)right, (uint4 *)own_l, (uint4 *)own_r,
                                              (uint4 *)prev_l, (uint4 *)prev_r, (uint4 *)next_l, (uint4 *)next_r, row_vec,
                                              band_rows, halo, own_rows, prev_rows, next_rows, counter, flag_at_prev,
                                              flag_at_next, epoch);
    return cudaGetLastError();
}

namespace {
PeerFlags peer_flags_of(unsigned *const *peer_flags, int n_peers) {
    PeerFlags pf;
    pf.n = n_peers;
    for (int i = 0; i < 8; i++) pf.p[i] = i < n_peers ? peer_flags[i] : nullptr;
    return pf;
}
}  // namespace

cudaError_t launch_publish_gray(const float *src, float *dst, size_t n_floats, unsigned *counter, unsigned *const *peer_flags,
                                int n_peers, unsigned epoch, cudaStream_t st, int planes, size_t src_plane, size_t dst_plane) {
    const PeerFlags pf = peer_flags_of(peer_flags, n_peers);
    const size_t n4 = n_floats / 4;
    int blocks = (int)((n4 + 255) / 256);
    if (blocks > 592) blocks = 592;
    if (blocks < 1) blocks = 1;
    publish_gray_kernel<<<blocks, 256, 0, st>>>((const float4 *)src, (float4 *)dst, n4, counter, pf, epoch, planes,
                                                src_plane / 4, dst_plane / 4);
    return cudaGetLastError();
}

cudaError_t launch_publish_fill_bounds(const unsigned char *row_kept, const float *rows, int band_rows, int glob_row0, int W,
                                       float *area, unsigned *counter, unsigned *const *peer_flags, int n_peers,
                                       unsigned epoch, cudaStream_t st) {
    const PeerFlags pf = peer_flags_of(peer_flags, n_peers);
    int seg = (W + 1023) / 1024;   // (about 4 columns per thread)
    if (seg > 16) seg = 16;
    publish_fill_bounds_kernel<<<dim3(seg, 2), 256, 0, st>>>(row_kept, rows, band_rows, glob_row0, W, area, counter, pf, epoch);
    return cudaGetLastError();
}

cudaError_t launch_wait_flags(const unsigned *flags, int first, int count, unsigned epoch, unsigned long long *timeout_word,
                              cudaStream_t st) {
    wait_flags_kernel<<<1, 32, 0, st>>>(flags, first, count, epoch, timeout_word);
    return cudaGetLastError();
}

}  // namespace sd
