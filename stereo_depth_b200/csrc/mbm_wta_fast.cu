// Kernel B, specialised variant: fused similarity cost + multi-block aggregation + winner-take-all
// for the reference's default radii (cost 3x3, windows 3x21 / 21x3 / 9x9).  CUDA-core (fp32 add)
// bound: 237 lane-ops per (pixel, disparity) cell, ~0.4 B of HBM traffic per cell -- no tensor cores.
//
// Bit-exactness rules out box filters / sliding windows: every window sum must be the reference's
// sequential fp32 chain (rows outer, columns inner, from 0.0f).  The kernel therefore spends its time
// on 204 dependent-order adds per cell and is organised to issue them at full rate:
//   * two disparity levels per pass, interleaved as float2 -> every add is one packed FADD2
//     (add.rn.f32x2, IEEE-exact per lane) and LDS.128 fetches two cells x two levels;
//   * a thread owns 4x4 pixels x 2 levels: one LDS.128 feeds ~14 packed adds (each cost cell is loaded
//     once per window per thread and reused by every pixel of the 4x4 block whose window covers it);
//   * the cost plane lives in shared memory with its 16-byte chunks split by parity (even chunks first,
//     odd chunks second) so the 32-byte lane stride of the 4-pixel ownership is bank-conflict free;
//   * the pooled left/right row bands are staged in shared memory once per tile by TMA bulk copies
//     (cp.async.bulk + mbarrier) from wrap-padded planes that already hold the reference's circular padding,
//     and reused by all L/2 passes;
//   * the 3x3 cost is computed by row-streaming 4-column strips: every |L-R| tap is evaluated once and
//     reused by the 3 cost rows and up to 3 cost columns that contain it;
//   * WTA keeps only (best, previous level, one pending A[d-1]) in registers and writes a pixel's 16-byte record
//     (d*, A[d*-1], A[d*], A[d*+1]) once it is complete and still standing; the [Hd,Wd,L] volume never exists.
//
// Semantics: identical to mbm_wta_generic.cu / oracle so_cost + so_aggregate + so_wta (SAFE padding).
// References: device_functions.cuh:53-73, ncc_matching_cost_volume_construction.cu:67-76,
// multi_block_matching_cost_aggregation.cu:56-87, wta_disparity_selection.cu:22-30.
#include <type_traits>

#include "common.cuh"
#include "mbm_helpers.cuh"

namespace sd {
namespace {

using namespace mbm;

constexpr int SEG = 9;            // cost-plane rows per cost-phase work item

template <int BH>
struct Cfg {
    static constexpr int NT = (BH / 4) * 16;
    static constexpr int PRW = BH + 20;                        // cost-plane rows
    static constexpr int NSEG = (PRW + SEG - 1) / SEG;
    static constexpr int BR = SEG * NSEG + 2;                  // band rows (incl. rows only dead items touch)
    static_assert(BH != kTileH || BR == kBandRows, "band geometry must match PadGeom");
    static constexpr int ITEMS = NSTRIP * NSEG;
};

template <int BH>
__host__ __device__ inline size_t smem_bytes(int L, int min_ds) {
    return (size_t)Cfg<BH>::PRW * NCHUNK * 16 + (size_t)Cfg<BH>::BR * (LW + make_pad_geom(64, 64, L, min_ds).rw) * 4;
}

// STORE: 0 nothing, 1 the whole aggregated volume (plane-major), 2 GATHER: no WTA at all, the flagged pairs' values go
// to the compact per-tile volume (Geom::abs_index == 2) and wta4 / edge2 are left untouched.
// SPLIT: level split (n_split_arg > 1 parts per tile); false compiles the part logic away (n_split == 1).
template <int BH, bool DBG, int STORE, bool SPLIT>
__global__ void __launch_bounds__(Cfg<BH>::NT, (BH <= 32) ? 2 : 1)
mbm_wta_fast_kernel(Geom g, PadGeom pg, const float *__restrict__ padl, const float *__restrict__ padr,
                    float4 *__restrict__ wta4, float2 *__restrict__ edge2, float *__restrict__ dbg_cost,
                    float *__restrict__ dbg_agg, float *__restrict__ agg_planes, const unsigned *__restrict__ pass_mask,
                    const int *__restrict__ range_flag, int range_epoch, const int *__restrict__ tile_order,
                    const int *__restrict__ bucket_count, int n_split_arg, int2 *__restrict__ part_range, int store_from) {
    using C = Cfg<BH>;
    const int n_split = SPLIT ? n_split_arg : 1;
    extern __shared__ float4 smem4[];
    float4 *plane = smem4;                                              // [PRW][42] chunks of (cell,level) pairs
    float *bandL = reinterpret_cast<float *>(plane + C::PRW * NCHUNK);  // [BR][LW]
    float *bandR = bandL + C::BR * LW;                                  // [BR][RW]

    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    // Which tile: by default the blocks in launch order.  Behind the level screen the tiles differ widely in cost
    // (3 .. M level pairs), so the screen sorts them into 8 buckets by pair count and blocks take them heaviest first
    // (longest-processing-time order: no long tile is left to start last).
    // LEVEL SPLIT (launches too small to fill the GPU: single frames, thin row bands): gridDim.z = frames * n_split and
    // consecutive blocks are the parts of one tile.  Part p evaluates the p-th share of the tile's flagged level pairs
    // (by rank, ascending) into the p-th slot of the part arrays (wta4 / edge2 then point at [n_split][frames][Hd*Wd]) and
    // notes the first / last level it evaluated in part_range; merge_parts_kernel combines the slots.
    // n_split == 1: every flagged pair, final arrays.
    const int lin = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
    const int part = lin % n_split;
    const int n_tiles = gridDim.x * gridDim.y * (gridDim.z / n_split);   // tiles of the launch (all frames)
    int tile = lin / n_split;
    if (tile_order) {
        int cnt[kScreenBuckets];
#pragma unroll
        for (int b = 0; b < kScreenBuckets; b++) cnt[b] = __ldg(bucket_count + b);   // independent loads, one round trip
        int rem = tile, slot = 0;
        bool found = false;
#pragma unroll
        for (int b = kScreenBuckets - 1; b >= 0; b--) {
            if (!found && rem < cnt[b]) {
                slot = b * n_tiles + rem;
                found = true;
            }
            if (!found) rem -= cnt[b];
        }
        if (found) tile = tile_order[slot];
    }
    const int tile_x = tile % gridDim.x, tile_y = (tile / gridDim.x) % gridDim.y;
    const int frame = tile / (gridDim.x * gridDim.y), r0 = tile_y * BH, c0 = tile_x * BW;
    const int Hd = g.Hd, Wd = g.Wd, L = g.L;
    const int Lp = (L + 1) & ~1, M = Lp >> 1;
    const size_t np = (size_t)Hd * Wd;
    const int RW = pg.rw;

    // ---- stage the pooled row bands once per tile with TMA bulk copies ---------------------------------
    // The wrap-padded planes (pad_pooled_kernel) make every band row one contiguous 16-byte aligned segment:
    // one cp.async.bulk per row and view, completion counted in bytes on an mbarrier.
    __shared__ __align__(8) uint64_t band_bar;
    // Level pairs this tile has to evaluate (certified screen, mbm_screen.cu); all of them without a screen or
    // when the screen's precondition (pooled values in [0,255]) does not hold for this chunk.
    __shared__ unsigned s_pass[4];
    if (tid == 0) mbar_init(&band_bar, 1);
    if (tid < 4) {
        unsigned w = 0xffffffffu;
        // (gather pass: the masks are exact requests, not a screen result -- they hold whatever the range flag says)
        if (pass_mask && (STORE == 2 || *range_flag != range_epoch))
            w = pass_mask[(size_t)tile * 4 + tid];
        const int valid_bits = M - 32 * tid;   // only pairs 0 .. M-1 exist
        s_pass[tid] = valid_bits >= 32 ? w : (valid_bits > 0 ? (w & ((1u << valid_bits) - 1u)) : 0u);
    }
    __syncthreads();
    // this part's share of the flagged pairs, by rank
    const int n_flag = __popc(s_pass[0]) + __popc(s_pass[1]) + __popc(s_pass[2]) + __popc(s_pass[3]);
    const int r_begin = (part * n_flag) / n_split, r_end = ((part + 1) * n_flag) / n_split;
    const int px0 = r0 + 4 * ty, py0 = c0 + 4 * tx;  // first owned pixel
    const size_t o00 = ((size_t)part * (gridDim.z / n_split) + frame) * np + (size_t)px0 * Wd + py0;
    if (n_split > 1 && r_begin == r_end) {
        // nothing to do for this part (fewer flagged pairs than parts): "no maximum here" records, empty range
#pragma unroll
        for (int k = 0; k < 16; k++)
            if (px0 + (k >> 2) < Hd && py0 + (k & 3) < Wd) wta4[o00 + (size_t)(k >> 2) * Wd + (k & 3)] = make_float4(-1.0f, 0.0f, 0.0f, 0.0f);
        if (tid == 0) part_range[(size_t)part * n_tiles + tile] = make_int2(-1, -1);
        return;
    }
    if (tid < 32) {
        if (tid == 0) mbar_expect_tx(&band_bar, (unsigned)(C::BR * (LW + RW) * 4));
        __syncwarp();
        const float *sl = padl + ((size_t)frame * pg.rows + r0) * pg.pwl + c0;
        const float *sr = padr + ((size_t)frame * pg.rows + r0) * pg.pwr + c0;
        for (int rr = tid; rr < C::BR; rr += 32) {
            tma_bulk_g2s(bandL + rr * LW, sl + (size_t)rr * pg.pwl, LW * 4, &band_bar);
            tma_bulk_g2s(bandR + rr * RW, sr + (size_t)rr * pg.pwr, (unsigned)(RW * 4), &band_bar);
        }
    }

    // ---- per-pixel WTA state (16 pixels, index k = a*4 + b) ---------------------------------------
    // Only the running maximum, the previous level and one pending A[d-1] stay in registers.  A pixel's record
    // (d*, A[d*-1], A[d*], A[d*+1]) goes to HBM/L2 once it is complete and still standing (see the WTA update
    // below) -- at most about ln(L) times per pixel -- which keeps ~50 registers free for the adder chains.
    // Pixels outside the image start at +inf and therefore never store.
    float best[16], prev[16], pam[16];
    unsigned pend = 0;  // bit k: pixel k's maximum sits at the odd level of the last evaluated pair; its record (with
                        // pam[k] = A[d*-1]) is written when the next pair delivers A[d*+1], or at the end
#pragma unroll
    for (int k = 0; k < 16; k++) {
        const bool valid = (px0 + (k >> 2) < Hd) && (py0 + (k & 3) < Wd);
        best[k] = valid ? kFltMin : __int_as_float(0x7f800000);
        prev[k] = 0.0f;
    }

    // cost-phase work item of this thread
    const bool has_item = tid < C::ITEMS;
    const int strip = tid % NSTRIP, seg = tid / NSTRIP;

    {
        int spins = 0;
        while (!mbar_try_wait(&band_bar, 0))
            if (++spins > (1 << 24)) __trap();  // a lost transaction must not hang the GPU
    }

    int rank = 0, m_first = -1, m_last = -1;
    for (int m = 0; m < M; m++) {
        // Skipped level pairs leave prev[] / pend stale.  That only ever reaches records that a later level
        // overwrites: the reference's arg-max d* is always evaluated together with d*-1 and d*+1 (circular), and
        // adjacent flagged pairs that fall into different parts are joined by merge_parts_kernel.
        if (!((s_pass[(m >> 5) & 3] >> (m & 31)) & 1u)) continue;
        if (SPLIT || STORE == 2) {
            if (rank++ < r_begin) continue;
            if (rank > r_end) break;
        }
        const bool first_pass = (m_first < 0);
        if (first_pass) m_first = m;
        const int m_prev = m_last;   // the pair evaluated before this one
        m_last = m;
        const int d0 = 2 * m;
        // ================= cost phase: plane[R][s] = (cost(d0), cost(d0+1)) ==========================
        // The right band is read at column offset e = Lp-2-d0 (even): 16-byte aligned on every other
        // pass.  Two straight-line variants keep every load at its widest conflict-free form.
        auto cost_phase = [&](auto aligned_tag) {
            constexpr bool ALIGNED = decltype(aligned_tag)::value;
            const int R0 = seg * SEG;
            const float *bl = bandL + R0 * LW + strip * 4 + 4;
            const float *br = bandR + R0 * RW + strip * 4 + (Lp - 2 - d0);
            float2 T[3][6];
            // Band loads are issued one full row ahead of their use through volatile asm (kept in program
            // order by the compiler): the LDS latency then overlaps the previous row's taps and chains.
            struct Raw {
                float4 l4;
                float2 l2;
                float r[8];
            };
            auto load_raw = [&](int brow) {
                Raw w;
                w.l4 = lds128(bl + brow * LW);
                w.l2 = lds64(bl + brow * LW + 4);
                if (ALIGNED) {
                    const float4 q0 = lds128(br + brow * RW), q1 = lds128(br + brow * RW + 4);
                    w.r[0] = q0.x; w.r[1] = q0.y; w.r[2] = q0.z; w.r[3] = q0.w;
                    w.r[4] = q1.x; w.r[5] = q1.y; w.r[6] = q1.z; w.r[7] = q1.w;
                } else {
                    const float2 ra = lds64(br + brow * RW);
                    const float4 q = lds128(br + brow * RW + 2);
                    const float2 rd = lds64(br + brow * RW + 6);
                    w.r[0] = ra.x; w.r[1] = ra.y; w.r[2] = q.x; w.r[3] = q.y;
                    w.r[4] = q.z; w.r[5] = q.w; w.r[6] = rd.x; w.r[7] = rd.y;
                }
                return w;
            };
            auto taps = [&](const Raw &w, float2(&t)[6]) {
                const float lv[6] = {w.l4.x, w.l4.y, w.l4.z, w.l4.w, w.l2.x, w.l2.y};
#pragma unroll
                for (int j = 0; j < 6; j++) t[j] = make_float2(tap(lv[j], w.r[j + 1]), tap(lv[j], w.r[j]));
            };
            Raw raw[2];
            raw[0] = load_raw(0);
            raw[1] = load_raw(1);
            taps(raw[0], T[0]);
            raw[0] = load_raw(2);
            taps(raw[1], T[1]);
#pragma unroll
            for (int rr = 0; rr < SEG; rr++) {
                float2(&top)[6] = T[rr % 3];
                float2(&mid)[6] = T[(rr + 1) % 3];
                float2(&bot)[6] = T[(rr + 2) % 3];
                if (rr + 1 < SEG) raw[(rr + 1) & 1] = load_raw(rr + 3);  // next row's band values
                taps(raw[rr & 1], bot);                                  // band row rr + 2
                // four independent 9-tap chains, interleaved; (0.0f + x) + y == x + y exactly
                float2 c[4];
#pragma unroll
                for (int i = 0; i < 4; i++) c[i] = __fadd2_rn(top[i], top[i + 1]);
#pragma unroll
                for (int i = 0; i < 4; i++) c[i] = __fadd2_rn(c[i], top[i + 2]);
#pragma unroll
                for (int q = 0; q < 3; q++)
#pragma unroll
                    for (int i = 0; i < 4; i++) c[i] = __fadd2_rn(c[i], mid[i + q]);
#pragma unroll
                for (int q = 0; q < 3; q++)
#pragma unroll
                    for (int i = 0; i < 4; i++) c[i] = __fadd2_rn(c[i], bot[i + q]);
                const int R = R0 + rr;
                if (R < C::PRW) {
                    plane[R * NCHUNK + strip] = make_float4(c[0].x, c[0].y, c[1].x, c[1].y);
                    plane[R * NCHUNK + HALF + strip] = make_float4(c[2].x, c[2].y, c[3].x, c[3].y);
                }
            }
        };
        if (has_item) {
            if (((Lp - 2 - d0) & 3) == 0) cost_phase(std::true_type{});
            else cost_phase(std::false_type{});
        }
        __syncthreads();

        // ================= aggregation phase ==========================================================
        // Loop nests put the tap index outermost and the 16 pixels innermost: consecutive instructions
        // belong to independent chains, while each chain still adds its taps in (row, col) order.
        float2 hv[16], acc[16];
        // ---- H: 3 rows x 21 cols.  plane rows 4ty+9 .. 4ty+14, cells 4tx .. 4tx+23 -----------------------
        {
            const float4 *hp = plane + (4 * ty + 9) * NCHUNK + tx;
#pragma unroll
            for (int t = 0; t < 6; t++) {
                float2 v[24];
#pragma unroll
                for (int j = 0; j < 12; j++) {
                    const float4 q = hp[t * NCHUNK + chunk_pos(j)];
                    v[2 * j] = lo2(q);
                    v[2 * j + 1] = hi2(q);
                }
#pragma unroll
                for (int j = 0; j < 21; j++) {
#pragma unroll
                    for (int a = 0; a < 4; a++) {
                        const int rel = t - 1 - a;  // window row offset of plane row t for pixel row a
                        if (rel < -1 || rel > 1) continue;
                        if (rel == -1 && j == 0) continue;  // folded into j == 1
#pragma unroll
                        for (int b = 0; b < 4; b++) {
                            if (rel == -1 && j == 1) hv[a * 4 + b] = __fadd2_rn(v[b], v[b + 1]);
                            else hv[a * 4 + b] = __fadd2_rn(hv[a * 4 + b], v[b + j]);
                        }
                    }
                }
            }
        }
        // ---- V: 21 rows x 3 cols.  plane rows 4ty .. 4ty+23, cells 4tx+8 .. 4tx+15 (uses +9..+14) -----
        {
            const float4 *vp = plane + (4 * ty) * NCHUNK + tx + 2;
            auto vrow = [&](const float4 *p, int amin, int amax, int first_a) {
                // first_a: pixel row whose window starts at this plane row (-1: none)
                const float4 q0 = p[0], q1 = p[HALF], q2 = p[1], q3 = p[HALF + 1];
                const float2 w[8] = {lo2(q0), hi2(q0), lo2(q1), hi2(q1), lo2(q2), hi2(q2), lo2(q3), hi2(q3)};
#pragma unroll
                for (int c3 = 0; c3 < 3; c3++) {
#pragma unroll
                    for (int a = 0; a < 4; a++) {
                        if (a < amin || a > amax) continue;
                        if (a == first_a && c3 == 0) continue;  // folded into c3 == 1
#pragma unroll
                        for (int b = 0; b < 4; b++) {
                            if (a == first_a && c3 == 1) acc[a * 4 + b] = __fadd2_rn(w[b + 1], w[b + 2]);
                            else acc[a * 4 + b] = __fadd2_rn(acc[a * 4 + b], w[b + 1 + c3]);
                        }
                    }
                }
            };
            vrow(vp + 0 * NCHUNK, 0, 0, 0);
            vrow(vp + 1 * NCHUNK, 0, 1, 1);
            vrow(vp + 2 * NCHUNK, 0, 2, 2);
            vrow(vp + 3 * NCHUNK, 0, 3, 3);
            // rows 4 .. 20, where every pixel row's window is open: a manual software pipeline issues the next row's
            // loads before this row's adds (measured faster than the rolled and the fully unrolled loop, DESIGN.md §4-B)
            auto vload = [&](const float4 *p, float4(&q)[4]) { q[0] = p[0]; q[1] = p[HALF]; q[2] = p[1]; q[3] = p[HALF + 1]; };
            auto vcomp = [&](const float4(&q)[4]) {
                const float2 w[8] = {lo2(q[0]), hi2(q[0]), lo2(q[1]), hi2(q[1]), lo2(q[2]), hi2(q[2]), lo2(q[3]), hi2(q[3])};
#pragma unroll
                for (int c3 = 0; c3 < 3; c3++)
#pragma unroll
                    for (int k = 0; k < 16; k++) acc[k] = __fadd2_rn(acc[k], w[(k & 3) + 1 + c3]);
            };
            float4 qa[4], qb[4];
            const float4 *p = vp + 4 * NCHUNK;
            vload(p, qa);
#pragma unroll 1
            for (int t = 4; t < 20; t += 2, p += 2 * NCHUNK) {
                vload(p + NCHUNK, qb);
                vcomp(qa);
                vload(p + 2 * NCHUNK, qa);
                vcomp(qb);
            }
            vcomp(qa);  // row 20
            vrow(vp + 21 * NCHUNK, 1, 3, -1);
            vrow(vp + 22 * NCHUNK, 2, 3, -1);
            vrow(vp + 23 * NCHUNK, 3, 3, -1);
#pragma unroll
            for (int k = 0; k < 16; k++) hv[k] = __fmul2_rn(hv[k], acc[k]);
        }
        // ---- C: 9 rows x 9 cols.  plane rows 4ty+6 .. 4ty+17, cells 4tx+6 .. 4tx+17 ----------------------
        {
            const float4 *cp = plane + (4 * ty + 6) * NCHUNK + tx;
            auto crow = [&](const float4 *p, int amin, int amax, int first_a) {
                // logical chunks 2tx+3 .. 2tx+8
                const float4 q0 = p[HALF + 1], q1 = p[2], q2 = p[HALF + 2], q3 = p[3], q4 = p[HALF + 3], q5 = p[4];
                const float2 u[12] = {lo2(q0), hi2(q0), lo2(q1), hi2(q1), lo2(q2), hi2(q2),
                                      lo2(q3), hi2(q3), lo2(q4), hi2(q4), lo2(q5), hi2(q5)};
#pragma unroll
                for (int j = 0; j < 9; j++) {
#pragma unroll
                    for (int a = 0; a < 4; a++) {
                        if (a < amin || a > amax) continue;
                        if (a == first_a && j == 0) continue;  // folded into j == 1
#pragma unroll
                        for (int b = 0; b < 4; b++) {
                            if (a == first_a && j == 1) acc[a * 4 + b] = __fadd2_rn(u[b], u[b + 1]);
                            else acc[a * 4 + b] = __fadd2_rn(acc[a * 4 + b], u[b + j]);
                        }
                    }
                }
            };
            crow(cp + 0 * NCHUNK, 0, 0, 0);
            crow(cp + 1 * NCHUNK, 0, 1, 1);
            crow(cp + 2 * NCHUNK, 0, 2, 2);
            crow(cp + 3 * NCHUNK, 0, 3, 3);
            const float4 *p = cp + 4 * NCHUNK;
#pragma unroll 1
            for (int t = 4; t <= 8; t++, p += NCHUNK) crow(p, 0, 3, -1);
            crow(cp + 9 * NCHUNK, 1, 3, -1);
            crow(cp + 10 * NCHUNK, 2, 3, -1);
            crow(cp + 11 * NCHUNK, 3, 3, -1);
#pragma unroll
            for (int k = 0; k < 16; k++) hv[k] = __fmul2_rn(hv[k], acc[k]);  // (H*V)*C
        }

        // ================= winner-take-all update (ascending d, strict >) =============================
        if (DBG && frame == 0) {  // debug volumes of frame 0 in the reference's [Hd][Wd][L] layout (parity tests)
#pragma unroll
            for (int k = 0; k < 16; k++) {
                const int x = px0 + (k >> 2), y = py0 + (k & 3);
                if (x < Hd && y < Wd) {
                    const int s = 4 * tx + (k & 3) + 10, R = 4 * ty + (k >> 2) + 10;
                    const float4 q = plane[R * NCHUNK + chunk_pos(s >> 1)];
                    const float2 cc = (s & 1) ? hi2(q) : lo2(q);
                    const size_t o = ((size_t)x * Wd + y) * L + d0;
                    if (dbg_cost) dbg_cost[o] = cc.x;
                    if (dbg_agg) dbg_agg[o] = hv[k].x;
                    if (d0 + 1 < L) {
                        if (dbg_cost) dbg_cost[o + 1] = cc.y;
                        if (dbg_agg) dbg_agg[o + 1] = hv[k].y;
                    }
                }
            }
        }
        if (STORE == 2) {
            // gather pass: pair m is the (rank-1)-th flagged pair of this tile; its two levels go to
            // agg_planes[tile][rank][level parity][32*64] -- one coalesced 16-byte store per thread row and level
            float *q0 = agg_planes + ((size_t)tile * M + (rank - 1)) * (2 * BH * BW) + (4 * ty) * BW + 4 * tx;
#pragma unroll
            for (int a = 0; a < 4; a++) {
                *reinterpret_cast<float4 *>(q0 + a * BW) = make_float4(hv[a * 4].x, hv[a * 4 + 1].x, hv[a * 4 + 2].x, hv[a * 4 + 3].x);
                *reinterpret_cast<float4 *>(q0 + a * BW + BH * BW) =
                    make_float4(hv[a * 4].y, hv[a * 4 + 1].y, hv[a * 4 + 2].y, hv[a * 4 + 3].y);
            }
            __syncthreads();  // everyone is done reading the plane before the next pass overwrites it
            continue;
        }
        if (STORE == 1 && agg_planes && (m == 0 || m >= store_from)) {
            // reference-compat mode: materialise the aggregated volume, plane-major [F][L][Hd*Wd] so that the 4
            // pixels of a thread row are one coalesced 16-byte store per level.  (store_from: the absolute-index reads
            // only ever touch level 0 and the levels from min(min_ds - 1, L - min_ds) on, see launch_t.)
            float *pl0 = agg_planes + ((size_t)frame * L + d0) * np + (size_t)px0 * Wd + py0;
            const bool vec = ((Wd & 3) == 0) && (py0 + 3 < Wd);
#pragma unroll
            for (int a = 0; a < 4; a++) {
                if (px0 + a >= Hd) break;
                float *q0 = pl0 + (size_t)a * Wd;
                if (vec) {
                    *reinterpret_cast<float4 *>(q0) = make_float4(hv[a * 4].x, hv[a * 4 + 1].x, hv[a * 4 + 2].x, hv[a * 4 + 3].x);
                    if (d0 + 1 < L)
                        *reinterpret_cast<float4 *>(q0 + np) =
                            make_float4(hv[a * 4].y, hv[a * 4 + 1].y, hv[a * 4 + 2].y, hv[a * 4 + 3].y);
                } else {
#pragma unroll
                    for (int b = 0; b < 4; b++)
                        if (py0 + b < Wd) {
                            q0[b] = hv[a * 4 + b].x;
                            if (d0 + 1 < L) q0[np + b] = hv[a * 4 + b].y;
                        }
                }
            }
        }
        // (unsplit: only pair 0 -- behind the screen A[0] and the fallback record matter only when level 0 is a candidate;
        //  a part slot always needs its "no maximum in this range" record and its first level's value)
        if (SPLIT ? first_pass : (m == 0)) {
#pragma unroll
            for (int k = 0; k < 16; k++) {
                const int x = px0 + (k >> 2), y = py0 + (k & 3);
                if (x < Hd && y < Wd) {
                    const size_t o = o00 + (size_t)(k >> 2) * Wd + (k & 3);
                    edge2[o].x = hv[k].x;                                    // A[first level this part evaluates] (A[0] unsplit)
                    // record if nothing ever beats FLT_MIN; in a part slot d = -1 says "no maximum in this range"
                    wta4[o] = make_float4(n_split > 1 ? -1.0f : 0.0f, 0.0f, hv[k].x, hv[k].y);
                }
            }
        }
        const bool has2 = (d0 + 1 < L);
        const float fd0 = (float)d0, fdp = (float)(2 * m_prev + 1);   // fdp: level of a pending maximum (odd level of the pair before)
        unsigned npend = 0;
        // A record is written once it is COMPLETE and still standing: a maximum at the even level of the pair has both
        // neighbours at hand; one at the odd level waits (pend, pam = its A[d-1]) for the next evaluated pair, whose
        // first level is its A[d+1] -- unless that level beats it, in which case nothing was ever stored for it.  On
        // cost curves that rise over many levels (natural scenes, out-of-range disparities) this saves a 16-byte store
        // per pixel and level.
#pragma unroll
        for (int k = 0; k < 16; k++) {
            const float a0 = hv[k].x, a1 = hv[k].y;
            float4 *rec = wta4 + o00 + (size_t)(k >> 2) * Wd + (k & 3);
            if ((pend & (1u << k)) && !(a0 > best[k])) *rec = make_float4(fdp, pam[k], best[k], a0);
            if (a0 > best[k]) {
                best[k] = a0;
                if (!(has2 && a1 > a0)) *rec = make_float4(fd0, prev[k], a0, a1);
            }
            if (has2 && a1 > best[k]) {
                best[k] = a1;
                pam[k] = a0;
                npend |= 1u << k;
            }
            prev[k] = has2 ? a1 : a0;
        }
        pend = npend;
        __syncthreads();  // everyone is done reading the plane before the next pass overwrites it
    }

    if (STORE == 2) return;
#pragma unroll
    for (int k = 0; k < 16; k++)   // maxima at the very last level evaluated: A[d*+1] lies beyond (circular wrap / next part)
        if (pend & (1u << k)) wta4[o00 + (size_t)(k >> 2) * Wd + (k & 3)] = make_float4((float)(2 * m_last + 1), pam[k], best[k], 0.0f);
#pragma unroll
    for (int k = 0; k < 16; k++) {
        const int x = px0 + (k >> 2), y = py0 + (k & 3);
        if (x < Hd && y < Wd) edge2[o00 + (size_t)(k >> 2) * Wd + (k & 3)].y = prev[k];  // A[last level evaluated] (A[L-1] unsplit)
    }
    if (n_split > 1 && tid == 0) part_range[(size_t)part * n_tiles + tile] = make_int2(2 * m_first, 2 * m_last + 1);
}

// Combines the part slots of a level-split launch into the final records: the maximum over the parts in ascending level
// order with strict '>' (the first maximum wins, wta_disparity_selection.cu:22-29).  Its neighbours A[d*-1] / A[d*+1] come
// from the adjacent part's edge values when d* is the first / last level its part evaluated: the pairs holding d*-1 and
// d*+1 are always flagged, so they are the last pair of the previous part / the first pair of the next one.
// (A[0], A[L-1]) for the circular wrap come from the outermost non-empty parts.
__global__ void merge_parts_kernel(const float4 *__restrict__ pw, const float2 *__restrict__ pe, const int2 *__restrict__ part_range,
                                   float4 *__restrict__ wta4, float2 *__restrict__ edge2, int Hd, int Wd, int frames, int S,
                                   int tiles_x, int tiles_y) {
    const size_t np = (size_t)Hd * Wd, n = np * frames;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int frame = (int)(i / np), x = (int)((i % np) / Wd), y = (int)(i % Wd);
    const size_t tile = ((size_t)frame * tiles_y + x / kTileH) * tiles_x + y / kTileW, n_tiles = (size_t)frames * tiles_x * tiles_y;
    float best = kFltMin;
    float4 out = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    int wp = -1, p_first = -1, p_last = -1;
    for (int p = 0; p < S; p++) {
        if (part_range[(size_t)p * n_tiles + tile].x < 0) continue;   // empty part
        if (p_first < 0) p_first = p;
        p_last = p;
        const float4 r = pw[(size_t)p * n + i];
        if (r.x >= 0.0f && r.z > best) {
            best = r.z;
            out = r;
            wp = p;
        }
    }
    if (wp < 0) {
        // nothing beats FLT_MIN: level 0 with (A[0], A[1]) like the unsplit kernel (the first part's first pair)
        const float4 r0 = pw[(size_t)(p_first < 0 ? 0 : p_first) * n + i];
        out = make_float4(0.0f, 0.0f, r0.z, r0.w);
    } else {
        const int2 rg = part_range[(size_t)wp * n_tiles + tile];
        const int d = (int)out.x;
        if (d == rg.x) {   // A[d*-1] is the previous non-empty part's last level
            for (int p = wp - 1; p >= 0; p--)
                if (part_range[(size_t)p * n_tiles + tile].x >= 0) {
                    out.y = pe[(size_t)p * n + i].y;
                    break;
                }
        }
        if (d == rg.y) {   // A[d*+1] is the next non-empty part's first level
            for (int p = wp + 1; p < S; p++)
                if (part_range[(size_t)p * n_tiles + tile].x >= 0) {
                    out.w = pe[(size_t)p * n + i].x;
                    break;
                }
        }
    }
    wta4[i] = out;
    if (p_first >= 0) edge2[i] = make_float2(pe[(size_t)p_first * n + i].x, pe[(size_t)p_last * n + i].y);
}

template <int BH, bool DBG, int STORE>
cudaError_t launch_t(const Geom &g, int frames, const Scratch &s, float *dbg_cost, float *dbg_agg, cudaStream_t st,
                     bool use_screen = false, int split = 1) {
    const size_t smem = smem_bytes<BH>(g.L, g.min_ds);
    const PadGeom pg = make_pad_geom(g.Hd, g.Wd, g.L, g.min_ds);
    // per-device attribute: set on every launch (cheap) so multi-GPU processes stay correct
    cudaError_t e = cudaFuncSetAttribute(mbm_wta_fast_kernel<BH, DBG, STORE, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    dim3 grid((g.Wd + BW - 1) / BW, (g.Hd + BH - 1) / BH, frames);
    // Whole-volume store (STORE == 1, reference-compat mode): which levels can secondary matching's absolute-index reads
    // agg[..][pad_index(q, L)], q = d* + min_ds + {-1, 0, 1} (secondary_matching.cu:28-31), ever touch?  q < L: level q >=
    // min_ds - 1;  q == L: level 0;  q > L: a negative pad_index, i.e. level 2L - q >= L - min_ds of an earlier pixel
    // (for min_ds <= L; beyond that several pixels back, any level).  Everything below is never read: not stored.
    int store_from = 0;
    if (STORE == 1 && !DBG && g.abs_index && g.min_ds >= 1 && g.min_ds <= g.L) {
        const int first_level = g.min_ds - 1 < g.L - g.min_ds ? g.min_ds - 1 : g.L - g.min_ds;
        store_from = first_level / 2;
    }
    if (STORE == 2) {
        mbm_wta_fast_kernel<BH, DBG, STORE, false><<<grid, Cfg<BH>::NT, smem, st>>>(
            g, pg, s.padl, s.padr, s.wta4, s.edge2, nullptr, nullptr, s.agg_vol, s.gather_mask, s.range_flag, s.range_epoch,
            nullptr, s.bucket_count, 1, nullptr, 0);
        return cudaGetLastError();
    }
    if (split > 1) {
        // level split: every tile's flagged level pairs are spread over `split` blocks writing part slots, then merged
        if (STORE != 0 || DBG || !s.wta4_parts || !s.edge2_parts || !s.part_range) return cudaErrorNotSupported;
        grid.z = frames * split;
        e = cudaFuncSetAttribute(mbm_wta_fast_kernel<BH, false, 0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        mbm_wta_fast_kernel<BH, false, 0, true><<<grid, Cfg<BH>::NT, smem, st>>>(
            g, pg, s.padl, s.padr, s.wta4_parts, s.edge2_parts, nullptr, nullptr, nullptr, use_screen ? s.pass_mask : nullptr,
            s.range_flag, s.range_epoch, use_screen ? s.tile_order : nullptr, s.bucket_count, split, s.part_range, 0);
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        const size_t n = (size_t)frames * g.Hd * g.Wd;
        merge_parts_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(s.wta4_parts, s.edge2_parts, s.part_range, s.wta4, s.edge2,
                                                                      g.Hd, g.Wd, frames, split, pg.tiles_x, pg.tiles_y);
        return cudaGetLastError();
    }
    mbm_wta_fast_kernel<BH, DBG, STORE, false><<<grid, Cfg<BH>::NT, smem, st>>>(
        g, pg, s.padl, s.padr, s.wta4, s.edge2, dbg_cost, dbg_agg, s.agg_vol, use_screen ? s.pass_mask : nullptr,
        s.range_flag, s.range_epoch, use_screen ? s.tile_order : nullptr, s.bucket_count, 1, nullptr, store_from);
    return cudaGetLastError();
}

}  // namespace

bool mbm_wta_fast_supported(const Geom &g) {
    return g.r_cost == 1 && g.rs == 1 && g.rm == 4 && g.rl == 10 && g.L >= 1 && smem_bytes<32>(g.L, g.min_ds) <= 227 * 1024;
}

// The wrap-padded planes (launch_pad_pooled) and, with use_screen, the pass masks of this chunk (launch_mbm_screen)
// must already be in flight on `st`.
cudaError_t launch_mbm_wta_fast(const Geom &g, int frames, const Scratch &s, float *dbg_cost, float *dbg_agg,
                                cudaStream_t st, bool use_screen, bool gather, int split) {
    if (!mbm_wta_fast_supported(g) || !s.padl || !s.padr) return cudaErrorNotSupported;
    if (gather) {
        if (!s.agg_vol || !s.gather_mask) return cudaErrorNotSupported;
        return launch_t<32, false, 2>(g, frames, s, nullptr, nullptr, st);
    }
    // the debug / whole-volume modes need every level: no screen there
    if (dbg_cost || dbg_agg) return launch_t<32, true, 1>(g, frames, s, dbg_cost, dbg_agg, st);
    if (s.agg_vol) return launch_t<32, false, 1>(g, frames, s, nullptr, nullptr, st);
    return launch_t<32, false, 0>(g, frames, s, nullptr, nullptr, st, use_screen, split);
}

}  // namespace sd
