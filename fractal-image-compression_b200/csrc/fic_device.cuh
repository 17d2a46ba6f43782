// fic_device.cuh -- device-side helpers shared by the kernels of libfic_b200.
//
// Geometry follows the reference exactly (file:line refer to
// src/bvk_ss19/FractalCompression.java = FC); float helpers pin Java semantics:
// binary32 with round-to-nearest on every operation, never contracted into FMA.
#pragma once

#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "fic_internal.h"

namespace fic {

// FC:516-545 getDomainBlockIndex: index of the domain block "above" range (xr, yr).
__host__ __device__ inline int domain_block_index(int xr, int yr, int rpw, int rph, int dpw)
{
    if (yr == 0) yr = 1;
    if (xr == 0) xr = 1;
    if (yr == rph - 1) yr = yr - 1;
    if (xr == rpw - 1) xr = xr - 1;
    int i = 0;
    if (xr > 1) {
        i = (yr == 0) ? xr : (xr * 2) - 2 + (yr + yr - 1) * dpw;
    } else if (xr == 1) {
        i = (yr == 0) ? xr : xr + (yr + yr - 1) * dpw;
    }
    return i;
}

// FC:84-100 generateKernel (= FC:868-879): clamped origin of the wk x wk window.
__host__ __device__ inline void window_origin(int index, int dpw, int dph, int wk, int *dy, int *dx)
{
    int y = index / dpw - wk / 2;
    int x = index % dpw - wk / 2;
    if (x < 0) x = 0;
    if (y < 0) y = 0;
    if (x + wk >= dpw) x = dpw - wk;
    if (y + wk >= dph) y = dph - wk;
    *dy = y;
    *dx = x;
}

// Window origin of range block j (raster order).
__host__ __device__ inline void range_window(const Geom &g, int64_t j, int *dy, int *dx)
{
    int xr = (int)(j % g.rpw), yr = (int)(j / g.rpw);
    int i = domain_block_index(xr, yr, g.rpw, g.rph, g.dpw);
    window_origin(i, g.dpw, g.dph, g.wk, dy, dx);
}

// Java (int)float: truncate toward zero, saturate, NaN -> 0 (== cvt.rzi.s32.f32 on the device).
__host__ __device__ __forceinline__ int j_f2i(float f)
{
#ifdef __CUDA_ARCH__
    return __float2int_rz(f);
#else
    if (f != f) return 0;
    if (f >= 2147483648.0f) return INT32_MAX;
    if (f <= -2147483648.0f) return INT32_MIN;
    return (int)f;
#endif
}

// FC:853-893 calculateIndices for range block j: the window-local index c of its code -> codebook index, with Java's
// float division and float remainder (FC:882-886); -1 when it falls outside the pool (the reference would throw).
__host__ __device__ inline int64_t code_pool_index(const Geom &g, int64_t j, float c)
{
    int dy, dx;
    range_window(g, j, &dy, &dx);
    const float fwk = (float)g.wk;
    const int yd = j_f2i(c / fwk), xd = j_f2i(fmodf(c, fwk));
    const int64_t r = (int64_t)xd + dx + (int64_t)(yd + dy) * g.dpw;
    return r < 0 || r >= g.ND ? -1 : r;
}

// ---- quadtree extension: the tree of one top block ----
// Range index at level L + 1 of child k (0 TL, 1 TR, 2 BL, 3 BR) of range j at level L.
__host__ __device__ inline int64_t qt_child(const QtGeom &q, int L, int64_t j, int k)
{
    const int64_t y = 2 * (j / q.g[L].rpw) + (k >> 1), x = 2 * (j % q.g[L].rpw) + (k & 1);
    return y * q.g[L + 1].rpw + x;
}

// A flag byte may set bit 0 (the top block is split) when there is a level below, and bit 1 + k (child k is split)
// only when bit 0 is set and there are two levels below.
__host__ __device__ inline bool qt_flags_legal(const QtGeom &q, uint32_t f)
{
    const uint32_t allowed = q.nl == 1 ? 0u : (q.nl == 2 || !(f & 1u) ? 1u : 0x1fu);
    return (f & ~allowed) == 0;
}

__host__ __device__ inline int qt_leaf_count(uint32_t f)
{
    if (!(f & 1u)) return 1;
    int n = 0;
    for (int k = 0; k < 4; k++) n += (f >> (1 + k)) & 1u ? 4 : 1;
    return n;
}

// Calls visit(level, range index) for every leaf of top block t in stream order: depth first, children in raster order.
#pragma nv_exec_check_disable
template <class V>
__host__ __device__ inline void qt_visit_leaves(const QtGeom &q, int64_t t, uint32_t f, V &&visit)
{
    if (!(f & 1u)) {
        visit(0, t);
        return;
    }
    for (int k = 0; k < 4; k++) {
        const int64_t c = qt_child(q, 0, t, k);
        if (!((f >> (1 + k)) & 1u)) {
            visit(1, c);
            continue;
        }
        for (int k2 = 0; k2 < 4; k2++) visit(2, qt_child(q, 1, c, k2));
    }
}

// Isometry extension (not in the reference): T_k maps range pixel (ry, rx) of a B x B block to the domain
// pixel (sy, sx) it is compared with / reconstructed from.  0 identity, 1-3 rotations, 4 mirror x, 5 mirror y,
// 6 transpose, 7 anti-transpose.
__host__ __device__ inline void iso_map(int k, int B, int ry, int rx, int *sy, int *sx)
{
    const int m = B - 1;
    switch (k & 7) {
    case 0: *sy = ry;     *sx = rx;     break;
    case 1: *sy = m - rx; *sx = ry;     break;
    case 2: *sy = m - ry; *sx = m - rx; break;
    case 3: *sy = rx;     *sx = m - ry; break;
    case 4: *sy = ry;     *sx = m - rx; break;
    case 5: *sy = m - ry; *sx = rx;     break;
    case 6: *sy = rx;     *sx = ry;     break;
    default: *sy = m - rx; *sx = m - ry; break;
    }
}
// iso_map(iso_inverse(k)) undoes iso_map(k): the rotations by 90 and 270 degrees swap, the rest are involutions.
__host__ __device__ inline int iso_inverse(int k) { return k == 1 ? 3 : (k == 3 ? 1 : k); }

#ifdef __CUDACC__

// FC:72 getMittelwert: the integer mean of a block from its pixel sum, mean = sum / n.  Returns
// sum (x - mean) = sum - n * mean (FC:671, FC:790), the exact integer in [0, n) that the reference's scores divide by.
__device__ __forceinline__ int centred_sum(int sum, int n, int *mean)
{
    const int m = sum / n;
    *mean = m;
    return sum - n * m;
}

// RGB (FC:760-791): the three channel means m[c] of block j, from per-channel sums stored as sum[c * count + j];
// returns the centred sums added over the channels (vR of a range block, vD of a domain).
__device__ __forceinline__ int centred_sum_rgb(const int32_t *__restrict__ sum, int64_t count, int64_t j, int n, int m[3])
{
    int v = 0;
#pragma unroll
    for (int c = 0; c < 3; c++) v += centred_sum(sum[c * count + j], n, &m[c]);
    return v;
}

// The reference's grey "error" of one candidate (FC:677-683), from exact integers:
// kov = sum (r-rmean)(d-dmean), vR = sum (r-rmean), varD = sum (d-dmean)^2.
// sqd must be the correctly rounded double sqrt of varD.
__device__ __forceinline__ float grey_error(int kov, int vR, double sqd)
{
    float fvR = (float)vR;
    float r = 0.0f;
    if (!(fvR == 0.0f || sqd == 0.0)) {
        double den = __dmul_rn((double)fvR, sqd);
        r = __double2float_rn(__ddiv_rn((double)(float)kov, den));
    }
    r = __fmul_rn(r, r);
    return __fmul_rn(__fmul_rn(fvR, fvR), __fsub_rn(1.0f, r));
}

// One step of the reference's RGB covariance, kov += gR * gD in binary32 (FC:789), gR and gD being the channel-summed
// centred pixels (FC:783-786).  |gR|, |gD| <= 765 are exact small integers, so their product is exact and one rounding
// of kov + product equals the reference's multiply-then-add -- also at B = 16, where kov may pass 2^24 and round.
__device__ __forceinline__ float rgb_kov_step(float kov, float gR, float gD) { return __fmaf_rn(gR, gD, kov); }

// The reference's RGB "error" of one candidate (FC:797-803): r = kov / (vR * vD), error = vR^2 (1 - r^2), all binary32.
// vR, vD are the channel-summed centred sums (FC:790-791): the domain's `variance` stays 0 on the RGB path.
__device__ __forceinline__ float rgb_error(float kov, float vR, float vD)
{
    float r = 0.0f;
    if (!(vR == 0.0f || vD == 0.0f)) r = __fdiv_rn(kov, __fmul_rn(vR, vD));
    r = __fmul_rn(r, r);
    return __fmul_rn(__fmul_rn(vR, vR), __fsub_rn(1.0f, r));
}

// Lexicographic (error, index) minimum: with the candidates visited in ascending index order, the reference's strict
// `error < best` (FC:627, FC:710) keeps the lowest index among equal errors, and so does this order.
__device__ __forceinline__ void argmin_merge(float &err, int &idx, float e2, int i2)
{
    if (e2 < err || (e2 == err && i2 < idx)) { err = e2; idx = i2; }
}

// argmin_merge over the 32 lanes of a warp; lane 0 ends with the warp's minimum.
__device__ __forceinline__ void warp_argmin(float &err, int &idx)
{
    for (int o = 16; o > 0; o >>= 1) {
        const float e2 = __shfl_down_sync(0xffffffffu, err, o);
        const int i2 = __shfl_down_sync(0xffffffffu, idx, o);
        argmin_merge(err, idx, e2, i2);
    }
}

// varD = sum d^2 - 2*dmean*sum d + n*dmean^2 with dmean = floor(sum d / n) (DB:92-115).
__device__ __forceinline__ int dom_var(int dsum, int dsq, int n, int *dmean)
{
    int m = dsum / n;
    *dmean = m;
    return dsq - m * (2 * dsum - n * m);
}

// One pixel of the 2x decimation (K1b in fic_kernels.cu) from the taps p00, p10 (row y), p01, p11 (row y + 1) of source
// column x.  Used by the pool builder and by the decoder sweeps, which decimate the image they write.
__device__ __forceinline__ int dec_tap4(int p00, int p10, int p01, int p11, int x, int H, bool rgb)
{
    int fourth = (x + 1 >= H) ? 128 : (rgb ? p01 : p11);
    return (p00 + p10 + p01 + fourth) / 4;
}

// A reconstructed pixel, (int)(a * domain + b) -- float multiply, then float add (FC:396 / FC:482) -- clamped to
// [0, 255] (FC:396-402, FC:743-749).  cvt.rzi.u8.f32 does the cast and the clamp in one instruction: it truncates
// toward zero and saturates to the destination range, NaN -> 0, like Java's cast followed by applyThreshold.
__device__ __forceinline__ uint32_t decode_px(float a, float b, uint32_t domain)
{
    uint32_t r;
    asm("cvt.rzi.u8.f32 %0, %1;" : "=r"(r) : "f"(__fadd_rn(__fmul_rn(a, (float)domain), b)));
    return r;
}

// Quantisation scales of the code stream: written by FC:242-244 / FC:250-254, read back by FC:372-374 / FC:446-450.
constexpr float kGreyAScale = 100.0f, kRgbAScale = 1000000.0f, kRgbBScale = 100000.0f;

#endif  // __CUDACC__

}  // namespace fic
