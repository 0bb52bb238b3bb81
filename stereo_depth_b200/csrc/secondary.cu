// Kernel C: secondary matching on the full-resolution gray images + the two parabola fits.
//
// Reference: secondary_matching.cu:24-71 with device_functions.cuh:22-73.  Per downscaled pixel:
//   dm   = int(d_wta);  candidates s in [K(dm-1), K(dm+1)];
//   S(s) = chain from 0.0f over i,j in [-r,r] (rows outer) of 255 - |GL[xK+i][yK+j] - GR[xK+i][yK+j-s]|
//   ds   = first arg-max of S (strict >, init FLT_MIN, default K(dm-1));
//   only if K(dm-1) < ds < K(dm+1):
//     qm = peak(dm, A[dm], dm+1, A[dm+1], dm-1, A[dm-1])   (A = aggregated cost, circular in d)
//     qs = peak(ds, S(ds), ds+1, S(ds+1), ds-1, S(ds-1))   (both neighbours are candidates already)
//     dm' = qm - dm; ds' = qs - ds; t = (ds + ds') - K dm
//     out = dm' * t > 0 ? (ds + ds')/K : ((dm + dm') + (ds + ds')/K) / 2
// The parabola's FMA contraction pattern follows the reference's SASS (see oracle/stereo_oracle.c).
// The aggregated volume is never in HBM: kernel B left (d*, A[d*-1], max A, A[d*+1]) and (A[0], A[L-1]).
// With min_disparity/K != 0 the reference indexes the volume with the ABSOLUTE disparity (secondary_matching.cu:28-31,
// an upstream bug).  That is reproduced by default (Geom::abs_index, sd_set_compat): the three values are then read
// through the reference's own pad_index / flat-offset arithmetic; sd_set_compat(h, 0) selects the relative index.
#include "common.cuh"

namespace sd {
namespace {

__device__ __forceinline__ float quad_peak(float x1, float y1, float x2, float y2, float x3, float y3) {
    const float den = __fmul_rn(__fmul_rn(__fsub_rn(x1, x2), __fsub_rn(x2, x3)), __fsub_rn(x1, x3));
    float m;
    if (y1 > y2) m = (y1 > y3) ? x1 : x3;
    else m = (y2 > y3) ? x2 : x3;
    if (den != 0.0f) {
        const float a = __fmaf_rn(x1, __fsub_rn(y3, y2), __fmaf_rn(x3, __fsub_rn(y2, y1), __fmul_rn(x2, __fsub_rn(y1, y3))));
        const float b = __fmaf_rn(__fmul_rn(x2, x2), __fsub_rn(y3, y1),
                                  __fmaf_rn(__fmul_rn(x3, x3), __fsub_rn(y1, y2),
                                            __fmul_rn(__fmul_rn(x1, x1), __fsub_rn(y2, y3))));
        if (a < 0.0f) m = __fdiv_rn(-b, __fadd_rn(a, a));
    }
    return m;
}

// NC = number of candidates kept in registers (2K+1); NC == 0: runtime K, neighbours recomputed.
// 4 blocks per SM: other occupancy bounds were measured and gave no gain.
template <int KT>
__global__ void __launch_bounds__(128, 4) secondary_kernel(Geom g, const float *__restrict__ gray,
                                                        const float4 *__restrict__ wta4,
                                                        const float2 *__restrict__ edge2, const float *__restrict__ agg_vol,
                                                        const unsigned *__restrict__ gather_mask, PadGeom pg,
                                                        float *__restrict__ refined) {
    const int y = blockIdx.x * blockDim.x + threadIdx.x;
    const int x = blockIdx.y * blockDim.y + threadIdx.y;
    const int frame = blockIdx.z;
    if (x >= g.Hd || y >= g.Wd) return;
    const int K = KT > 0 ? KT : g.K;
    const int H = g.H, W = g.W, r = g.r_sad;
    const size_t plane = (size_t)H * W;
    const float *gl = gray + (size_t)frame * 2 * plane, *gr = gl + plane;
    const size_t o = (size_t)frame * g.Hd * g.Wd + (size_t)x * g.Wd + y;
    const float4 w = wta4[o];
    const int bd = (int)w.x;
    const float dispf = __fadd_rn(w.x, (float)g.min_ds);  // wta_disparity_selection.cu:30
    const int dm = (int)dispf;
    const int lo = K * (dm - 1), hi = K * (dm + 1);
    float result = dispf;

    constexpr int NC = KT > 0 ? 2 * KT + 1 : 1;
    float S[NC];
    float c_sad = kFltMin;
    int d_sad = lo;
    if (KT > 0) {
#pragma unroll
        for (int k = 0; k < NC; k++) S[k] = 0.0f;
        // Tap (j, k) reads GL[c+j] and GR[c+j-(lo+k)] = GR[base + (j-k+KT)] with base = c - KT*dm:
        // per image row only 2r+1 left and 2r+2KT+1 right values are distinct.  RS = sad radius when it
        // is the reference default (registers), otherwise fall through to the per-tap loads below.
        constexpr int RS = 5, NL = 2 * RS + 1, NR = 2 * RS + 2 * KT + 1;
        const int c = y * K;
        int base = c - K * dm;
        // Left image border: the whole right-view window [base-RS-KT-1, base+RS+KT] lies left of column 0 and wraps
        // (circular padding) to the same columns + W -- still one contiguous, equally aligned run when W is even.
        if (base + RS + KT < 0 && (W & 1) == 0 && base + W - RS - KT - 1 >= 0) base += W;
        const bool interior = (r == RS) && (x * K - RS >= 0) && (x * K + RS < H) && (c - RS >= 0) && (c + RS < W) &&
                              (base - RS - KT >= 0) && (base + RS + KT < W);
        if (KT == 2 && interior && (W & 1) == 0 && c - RS - 1 >= 0 && base - RS - KT - 1 >= 0) {
            // K = 2: the first needed column is odd for both views; start one earlier and use 8-byte loads
            // (adjacent lanes are 8 bytes apart: every LDG.64 is fully coalesced).
            const float2 *lp = reinterpret_cast<const float2 *>(gl + (size_t)(x * K - RS) * W + (c - RS - 1));
            const float2 *rp = reinterpret_cast<const float2 *>(gr + (size_t)(x * K - RS) * W + (base - RS - KT - 1));
            const int pitch2 = W >> 1;
            // Candidates are accumulated as packed pairs (S1,S0), (S3,S2) + scalar S4.  For even tap columns the two
            // right-view operands of a pair are an aligned register pair straight from an LDG.64, so the tap itself is
            // two packed ops (FADD2 with a broadcast left operand, FADD2 255-|.|); odd columns compute scalar taps
            // into a register pair.  Either way each chain adds its taps in (row, column) order: bit-identical.
            float2 s10 = make_float2(0.0f, 0.0f), s32 = make_float2(0.0f, 0.0f);
            float s4 = 0.0f;
            const float2 c255 = make_float2(255.0f, 255.0f);
            // Software pipeline with two register sets (no copies): while the 55 taps of one image row are evaluated
            // from set A, the 14 loads of the next row are in flight into set B, and vice versa.
            struct Row {
                float2 l[(NL + 1) / 2], r[(NR + 1) / 2];
            };
            auto load_row = [&](Row &w) {
#pragma unroll
                for (int j = 0; j < (NL + 1) / 2; j++) w.l[j] = __ldg(lp + j);
#pragma unroll
                for (int q = 0; q < (NR + 1) / 2; q++) w.r[q] = __ldg(rp + q);
                lp += pitch2;
                rp += pitch2;
            };
            auto eval_row = [&](const Row &w) {
                // lv(k) / rv(k): element k of the 12 left / 16 right values of this row
                auto lv = [&](int k) { return (k & 1) ? w.l[k >> 1].y : w.l[k >> 1].x; };
                auto rv = [&](int k) { return (k & 1) ? w.r[k >> 1].y : w.r[k >> 1].x; };
#pragma unroll
                for (int j = 0; j < NL; j++) {
                    const float l = lv(j + 1);
                    if ((j & 1) == 0) {
                        const float2 t10 = __fadd2_rn(make_float2(l, l), make_float2(-rv(j + 4), -rv(j + 5)));  // k = 1, 0
                        const float2 t32 = __fadd2_rn(make_float2(l, l), make_float2(-rv(j + 2), -rv(j + 3)));  // k = 3, 2
                        s10 = __fadd2_rn(s10, __fadd2_rn(c255, make_float2(-fabsf(t10.x), -fabsf(t10.y))));
                        s32 = __fadd2_rn(s32, __fadd2_rn(c255, make_float2(-fabsf(t32.x), -fabsf(t32.y))));
                    } else {
                        const float u1 = __fsub_rn(255.0f, fabsf(__fsub_rn(l, rv(j + 4))));
                        const float u0 = __fsub_rn(255.0f, fabsf(__fsub_rn(l, rv(j + 5))));
                        const float u3 = __fsub_rn(255.0f, fabsf(__fsub_rn(l, rv(j + 2))));
                        const float u2 = __fsub_rn(255.0f, fabsf(__fsub_rn(l, rv(j + 3))));
                        s10 = __fadd2_rn(s10, make_float2(u1, u0));
                        s32 = __fadd2_rn(s32, make_float2(u3, u2));
                    }
                    s4 = __fadd_rn(s4, __fsub_rn(255.0f, fabsf(__fsub_rn(l, rv(j + 1)))));
                }
            };
            static_assert(NL % 2 == 1, "row loop below assumes an odd number of rows");
            Row ra, rb;
            load_row(ra);
#pragma unroll 1
            for (int i = 0; i < NL / 2; i++) {
                load_row(rb);
                eval_row(ra);
                load_row(ra);
                eval_row(rb);
            }
            eval_row(ra);
            S[0] = s10.y;
            S[1 % NC] = s10.x;
            S[2 % NC] = s32.y;
            S[3 % NC] = s32.x;
            S[4 % NC] = s4;
        } else if (interior) {
            const float *lp = gl + (size_t)(x * K - RS) * W + (c - RS);
            const float *rp = gr + (size_t)(x * K - RS) * W + (base - RS - KT);
#pragma unroll 1
            for (int i = 0; i < NL; i++, lp += W, rp += W) {
                float lv[NL], rv[NR];
#pragma unroll
                for (int j = 0; j < NL; j++) lv[j] = __ldg(lp + j);
#pragma unroll
                for (int q = 0; q < NR; q++) rv[q] = __ldg(rp + q);
#pragma unroll
                for (int j = 0; j < NL; j++)
#pragma unroll
                    for (int k = 0; k < NC; k++)
                        S[k] = __fadd_rn(S[k], __fsub_rn(255.0f, fabsf(__fsub_rn(lv[j], rv[j - k + 2 * KT]))));
            }
        } else if (r == RS && W > K * (g.L + g.min_ds) + 4 * (RS + KT + 1) && H > 2 * RS) {
            // border pixels: same register-blocked structure; every index is within one period of the image, so the
            // circular padding is a single conditional add/subtract per load (no integer modulo)
            auto near = [](int i, int n) { return i < 0 ? i + n : (i >= n ? i - n : i); };
            const int cl = near(c - RS, W) , cr = near(near(base, W) - RS - KT, W);
#pragma unroll 1
            for (int i = 0; i < NL; i++) {
                const size_t ro = (size_t)near(x * K - RS + i, H) * W;
                float lv[NL], rv[NR];
#pragma unroll
                for (int j = 0; j < NL; j++) lv[j] = __ldg(gl + ro + (cl + j >= W ? cl + j - W : cl + j));
#pragma unroll
                for (int q = 0; q < NR; q++) rv[q] = __ldg(gr + ro + (cr + q >= W ? cr + q - W : cr + q));
#pragma unroll
                for (int j = 0; j < NL; j++)
#pragma unroll
                    for (int k = 0; k < NC; k++)
                        S[k] = __fadd_rn(S[k], __fsub_rn(255.0f, fabsf(__fsub_rn(lv[j], rv[j - k + 2 * KT]))));
            }
        } else if (r == RS) {
            // tiny images: true modulo on every index
#pragma unroll 1
            for (int i = 0; i < NL; i++) {
                const size_t ro = (size_t)wrapm(x * K - RS + i, H) * W;
                float lv[NL], rv[NR];
#pragma unroll
                for (int j = 0; j < NL; j++) lv[j] = __ldg(gl + ro + wrapm(c - RS + j, W));
#pragma unroll
                for (int q = 0; q < NR; q++) rv[q] = __ldg(gr + ro + wrapm(base - RS - KT + q, W));
#pragma unroll
                for (int j = 0; j < NL; j++)
#pragma unroll
                    for (int k = 0; k < NC; k++)
                        S[k] = __fadd_rn(S[k], __fsub_rn(255.0f, fabsf(__fsub_rn(lv[j], rv[j - k + 2 * KT]))));
            }
        } else {
            for (int i = -r; i <= r; i++) {
                const size_t ro = (size_t)wrapm(x * K + i, H) * W;
                for (int j = -r; j <= r; j++) {
                    const int cc = y * K + j;
                    const float l = __ldg(gl + ro + wrapm(cc, W));
#pragma unroll
                    for (int k = 0; k < NC; k++) {
                        const float rr = __ldg(gr + ro + wrapm(cc - (lo + k), W));
                        S[k] = __fadd_rn(S[k], __fsub_rn(255.0f, fabsf(__fsub_rn(l, rr))));
                    }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < NC; k++)
            if (S[k] > c_sad) {
                c_sad = S[k];
                d_sad = lo + k;
            }
    } else {
        for (int s = lo; s <= hi; s++) {
            float c = 0.0f;
            for (int i = -r; i <= r; i++) {
                const size_t ro = (size_t)wrapm(x * K + i, H) * W;
                for (int j = -r; j <= r; j++) {
                    const float l = __ldg(gl + ro + wrapm(y * K + j, W));
                    const float rr = __ldg(gr + ro + wrapm(y * K + j - s, W));
                    c = __fadd_rn(c, __fsub_rn(255.0f, fabsf(__fsub_rn(l, rr))));
                }
            }
            if (c > c_sad) {
                c_sad = c;
                d_sad = s;
            }
        }
    }

    if (d_sad > lo && d_sad < hi) {
        float sp = 0.0f, sm = 0.0f;
        if (KT > 0) {
#pragma unroll
            for (int k = 1; k < NC - 1; k++)
                if (lo + k == d_sad) {
                    sp = S[k + 1];
                    sm = S[k - 1];
                }
        } else {
            for (int i = -r; i <= r; i++) {
                const size_t ro = (size_t)wrapm(x * K + i, H) * W;
                for (int j = -r; j <= r; j++) {
                    const float l = __ldg(gl + ro + wrapm(y * K + j, W));
                    const float rp = __ldg(gr + ro + wrapm(y * K + j - (d_sad + 1), W));
                    const float rm = __ldg(gr + ro + wrapm(y * K + j - (d_sad - 1), W));
                    sp = __fadd_rn(sp, __fsub_rn(255.0f, fabsf(__fsub_rn(l, rp))));
                    sm = __fadd_rn(sm, __fsub_rn(255.0f, fabsf(__fsub_rn(l, rm))));
                }
            }
        }
        const float2 e = edge2[o];
        float a_d = (bd == 0) ? e.x : w.z;
        float a_m1 = (bd == 0) ? e.y : w.y;
        float a_p1 = (bd == g.L - 1) ? e.x : w.w;
        if (g.abs_index && agg_vol) {
            // reference-compat: the reference reads agg[x][y][pad_index(ABSOLUTE disparity, L)] with unchecked flat
            // addressing (secondary_matching.cu:28-31): a negative pad_index lands in the previous pixel's levels.
            const size_t npix = (size_t)g.Hd * g.Wd;
            const float *vol = agg_vol + (size_t)frame * g.L * npix;   // plane-major [L][Hd*Wd]
            const long long po = ((long long)x * g.Wd + y) * g.L;
            auto rd = [&](int q, float safe) {
                const long long flat = po + ref_pad_index(q, g.L);     // index into the reference's [Hd][Wd][L] tensor
                if (flat < 0) return safe;                             // before the tensor: SAFE (relative) value
                const int lv = (int)(flat % g.L);
                const long long sp = flat / g.L;                       // source pixel (this one, or an earlier one)
                if (g.abs_index == 2) {
                    // compact volume of the gather pass: [F*tiles][rank of the pair in the tile's mask][parity][32*64]
                    const int sx = (int)(sp / g.Wd), sy = (int)(sp % g.Wd), m = lv >> 1, M = (g.L + 1) >> 1;
                    const size_t tile = ((size_t)frame * pg.tiles_y + sx / kTileH) * pg.tiles_x + sy / kTileW;
                    const unsigned *mk = gather_mask + tile * 4;
                    int rank = __popc(__ldg(mk + (m >> 5)) & ((1u << (m & 31)) - 1u));
                    for (int w = 0; w < (m >> 5); w++) rank += __popc(__ldg(mk + w));
                    return __ldg(agg_vol + (tile * M + rank) * (size_t)(2 * kTileH * kTileW) + (size_t)(lv & 1) * (kTileH * kTileW) +
                                 (sx % kTileH) * kTileW + (sy % kTileW));
                }
                return __ldg(vol + (size_t)lv * npix + (size_t)sp);
            };
            a_d = rd(dm, a_d);
            a_p1 = rd(dm + 1, a_p1);
            a_m1 = rd(dm - 1, a_m1);
        }
        const float fdm = (float)dm, fds = (float)d_sad, fk = (float)K;
        const float qm = quad_peak(fdm, a_d, (float)(dm + 1), a_p1, (float)(dm - 1), a_m1);
        const float qs = quad_peak(fds, c_sad, (float)(d_sad + 1), sp, (float)(d_sad - 1), sm);
        const float delta_mbm = __fsub_rn(qm, fdm);
        const float delta_sad = __fsub_rn(qs, fds);
        const float pos = __fadd_rn(fds, delta_sad);
        const float t = __fsub_rn(pos, (float)(K * dm));
        if (__fmul_rn(delta_mbm, t) > 0.0f) result = __fdiv_rn(pos, fk);
        else result = __fmul_rn(__fadd_rn(__fadd_rn(fdm, delta_mbm), __fdiv_rn(pos, fk)), 0.5f);
    }
    refined[o] = result;
}

// Which aggregated values will secondary matching's absolute-index reads touch?  One thread per pooled pixel: the
// three reads agg[x][y][pad_index(dm + {0, +1, -1}, L)] of secondary_matching.cu:28-31 (flat addressing: a negative
// pad_index lands in an earlier pixel), each marked as a level pair in the mask of the 32x64 tile that holds the SOURCE
// pixel.  The gather pass of the fused kernel then evaluates exactly those pairs.  (Every pixel is marked: whether its
// refinement branch is taken is only known once secondary matching has run.)
__global__ void abs_targets_kernel(Geom g, PadGeom pg, const float4 *__restrict__ wta4, unsigned *__restrict__ gather_mask) {
    const int y = blockIdx.x * blockDim.x + threadIdx.x;
    const int x = blockIdx.y * blockDim.y + threadIdx.y;
    const int frame = blockIdx.z;
    if (x >= g.Hd || y >= g.Wd) return;
    const size_t o = (size_t)frame * g.Hd * g.Wd + (size_t)x * g.Wd + y;
    const int dm = (int)__fadd_rn(wta4[o].x, (float)g.min_ds);
    const long long po = ((long long)x * g.Wd + y) * g.L;
#pragma unroll
    for (int k = -1; k <= 1; k++) {
        const long long flat = po + ref_pad_index(dm + k, g.L);
        if (flat < 0) continue;
        const int lv = (int)(flat % g.L), m = lv >> 1;
        const long long sp = flat / g.L;
        const int sx = (int)(sp / g.Wd), sy = (int)(sp % g.Wd);
        unsigned *w = gather_mask + (((size_t)frame * pg.tiles_y + sx / kTileH) * pg.tiles_x + sy / kTileW) * 4 + (m >> 5);
        const unsigned bit = 1u << (m & 31);
        if (!(*reinterpret_cast<volatile unsigned *>(w) & bit)) atomicOr(w, bit);   // mostly already set by a neighbour
    }
}

}  // namespace

cudaError_t launch_abs_targets(const Geom &g, int frames, const Scratch &s, cudaStream_t st) {
    if (!s.gather_mask) return cudaErrorNotSupported;
    const PadGeom pg = make_pad_geom(g.Hd, g.Wd, g.L, g.min_ds);
    cudaError_t e = cudaMemsetAsync(s.gather_mask, 0, (size_t)frames * pg.tiles_x * pg.tiles_y * 4 * sizeof(unsigned), st);
    if (e != cudaSuccess) return e;
    dim3 block(32, 8), grid((g.Wd + 31) / 32, (g.Hd + 7) / 8, frames);
    abs_targets_kernel<<<grid, block, 0, st>>>(g, pg, s.wta4, s.gather_mask);
    return cudaGetLastError();
}

cudaError_t launch_secondary(const Geom &g, int frames, const Scratch &s, cudaStream_t st) {
    dim3 block(32, 4), grid((g.Wd + 31) / 32, (g.Hd + 3) / 4, frames);
    const PadGeom pg = make_pad_geom(g.Hd, g.Wd, g.L, g.min_ds);
    switch (g.K) {
        case 1: secondary_kernel<1><<<grid, block, 0, st>>>(g, s.gray, s.wta4, s.edge2, s.agg_vol, s.gather_mask, pg, s.refined); break;
        case 2: secondary_kernel<2><<<grid, block, 0, st>>>(g, s.gray, s.wta4, s.edge2, s.agg_vol, s.gather_mask, pg, s.refined); break;
        case 3: secondary_kernel<3><<<grid, block, 0, st>>>(g, s.gray, s.wta4, s.edge2, s.agg_vol, s.gather_mask, pg, s.refined); break;
        case 4: secondary_kernel<4><<<grid, block, 0, st>>>(g, s.gray, s.wta4, s.edge2, s.agg_vol, s.gather_mask, pg, s.refined); break;
        default: secondary_kernel<0><<<grid, block, 0, st>>>(g, s.gray, s.wta4, s.edge2, s.agg_vol, s.gather_mask, pg, s.refined); break;
    }
    return cudaGetLastError();
}

}  // namespace sd
