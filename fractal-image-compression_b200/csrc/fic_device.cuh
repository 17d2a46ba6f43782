// fic_device.cuh -- device-side helpers shared by the kernels of libfic_b200.
//
// Geometry follows the reference exactly (file:line refer to
// src/bvk_ss19/FractalCompression.java = FC); float helpers pin Java semantics:
// binary32 with round-to-nearest on every operation, never contracted into FMA.
#pragma once

#include <cuda_runtime.h>
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

// Java (int)float: truncate toward zero, saturate, NaN -> 0 == cvt.rzi.s32.f32.
__device__ __forceinline__ int j_f2i(float f) { return __float2int_rz(f); }

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

// Quantisation scales of the code stream: written by FC:242-244 / FC:250-254, read back by FC:372-374 / FC:446-450.
constexpr float kGreyAScale = 100.0f, kRgbAScale = 1000000.0f, kRgbBScale = 100000.0f;

#endif  // __CUDACC__

}  // namespace fic
