// fic_kernels.cu -- HBM-bound kernels of libfic_b200 (sm_100a):
//   K1  pool builder: ARGB unpack, 2x decimation, per-domain / per-range integer sums
//   K2w direct windowed search (grey + RGB), the reference's default widthKernel path
//   K3s code solve + quantisation (shared by the direct and the tcgen05 search)
//   K4  iterative decoder sweep (+ one-shot collage), exact avgError bookkeeping
//
// file:line citations refer to the reference, src/bvk_ss19/FractalCompression.java (FC)
// and src/bvk_ss19/Domainblock.java (DB).
#include "fic_device.cuh"

namespace fic {

// ------------------------------------------------------------------------------------
// K1a: ARGB int32 -> 8-bit planes.  Grey keeps the red channel only (FC:596, FC:977).
// 16-byte loads, 4-byte stores per plane.
// ------------------------------------------------------------------------------------
template <int C>
__global__ void k_unpack(const int4 *__restrict__ argb, uchar4 *__restrict__ planes, int64_t quads,
                         int64_t plane_quads)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < quads; i += stride) {
        int4 p = __ldg(argb + i);
        planes[i] = make_uchar4((p.x >> 16) & 0xff, (p.y >> 16) & 0xff, (p.z >> 16) & 0xff, (p.w >> 16) & 0xff);
        if (C == 3) {
            planes[plane_quads + i] =
                make_uchar4((p.x >> 8) & 0xff, (p.y >> 8) & 0xff, (p.z >> 8) & 0xff, (p.w >> 8) & 0xff);
            planes[2 * plane_quads + i] = make_uchar4(p.x & 0xff, p.y & 0xff, p.z & 0xff, p.w & 0xff);
        }
    }
}

int launch_unpack(const int32_t *d_argb, uint8_t *d_planes, int W, int H, int C, cudaStream_t s)
{
    int64_t quads = (int64_t)W * H / 4;  // W % 4 == 0 is guaranteed by make_geom
    int blocks = (int)((quads + 255) / 256 < 148 * 16 ? (quads + 255) / 256 : 148 * 16);
    if (blocks < 1) blocks = 1;
    if (C == 1)
        k_unpack<1><<<blocks, 256, 0, s>>>((const int4 *)d_argb, (uchar4 *)d_planes, quads, quads);
    else
        k_unpack<3><<<blocks, 256, 0, s>>>((const int4 *)d_argb, (uchar4 *)d_planes, quads, quads);
    return 1;
}

// planes -> ARGB (0xff alpha), grey replicates the plane (FC:404, FC:490).  Grid-stride over quads of pixels with
// blockDim.x == 256.
template <int C>
__device__ __forceinline__ void pack_argb(const uchar4 *planes, int4 *argb, int64_t quads)
{
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < quads; i += (int64_t)gridDim.x * 256) {
        const uchar4 r = planes[i];
        uchar4 g = r, b = r;
        if (C == 3) {
            g = planes[quads + i];
            b = planes[2 * quads + i];
        }
        auto px = [](uint32_t r, uint32_t g, uint32_t b) { return (int)(0xff000000u | (r << 16) | (g << 8) | b); };
        argb[i] = make_int4(px(r.x, g.x, b.x), px(r.y, g.y, b.y), px(r.z, g.z, b.z), px(r.w, g.w, b.w));
    }
}

template <int C>
__global__ void k_pack_argb(const uchar4 *__restrict__ planes, int4 *__restrict__ argb, int64_t quads)
{
    pack_argb<C>(planes, argb, quads);
}

int launch_pack_argb(const uint8_t *d_planes, int32_t *d_argb, int W, int H, int C, cudaStream_t s)
{
    int64_t quads = (int64_t)W * H / 4;
    int blocks = (int)((quads + 255) / 256 < 148 * 16 ? (quads + 255) / 256 : 148 * 16);
    if (blocks < 1) blocks = 1;
    if (C == 1)
        k_pack_argb<1><<<blocks, 256, 0, s>>>((const uchar4 *)d_planes, (int4 *)d_argb, quads);
    else
        k_pack_argb<3><<<blocks, 256, 0, s>>>((const uchar4 *)d_planes, (int4 *)d_argb, quads);
    return 1;
}

// ------------------------------------------------------------------------------------
// K1b: 2x decimation (FC:970-1007 grey, FC:901-962 RGB).
//   grey: (p00 + p10 + p01 + p11) / 4;  RGB: (p00 + p10 + 2*p01) / 4 (FC:945 re-reads
//   (x, y+1)).  With W, H even the only live border branch is the reference's
//   `x + 1 >= image.height` test (FC:993, FC:940), which substitutes 128 for the fourth
//   tap on landscape images; it is reproduced here.
// One thread makes 2 output pixels from two 4-byte loads; stores are 2 bytes.
// ------------------------------------------------------------------------------------
__device__ __forceinline__ int dec_tap4(int p00, int p10, int p01, int p11, int x, int H, bool rgb)
{
    int fourth = (x + 1 >= H) ? 128 : (rgb ? p01 : p11);
    return (p00 + p10 + p01 + fourth) / 4;
}

__global__ void k_decimate(const uint8_t *__restrict__ src, uint8_t *__restrict__ dec, int W, int H, int C)
{
    int sw = W / 2, sh = H / 2;
    int64_t pairs_per_plane = (int64_t)(sw / 2) * sh;
    int64_t total = pairs_per_plane * C;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    bool rgb = C == 3;
    for (; i < total; i += stride) {
        int c = (int)(i / pairs_per_plane);
        int64_t k = i - c * pairs_per_plane;
        int qy = (int)(k / (sw / 2)), qx2 = (int)(k % (sw / 2));
        const uint8_t *p = src + (int64_t)c * W * H + (int64_t)(2 * qy) * W + 4 * qx2;
        uchar4 a = *(const uchar4 *)p;
        uchar4 b = *(const uchar4 *)(p + W);
        int x0 = 4 * qx2;
        uchar2 o;
        o.x = (unsigned char)dec_tap4(a.x, a.y, b.x, b.y, x0, H, rgb);
        o.y = (unsigned char)dec_tap4(a.z, a.w, b.z, b.w, x0 + 2, H, rgb);
        *(uchar2 *)(dec + (int64_t)c * sw * sh + (int64_t)qy * sw + 2 * qx2) = o;
    }
}

// Vector path (W % 16 == 0): one thread makes 8 output pixels from two 16-byte loads, one 8-byte store.
__global__ void k_decimate_v8(const uint8_t *__restrict__ src, uint8_t *__restrict__ dec, int W, int H, int C)
{
    const int sw = W / 2, sh = H / 2;
    const int64_t oct_per_plane = (int64_t)(sw / 8) * sh;
    const int64_t total = oct_per_plane * C;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const bool rgb = C == 3;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int c = (int)(i / oct_per_plane);
        const int64_t k = i - c * oct_per_plane;
        const int qy = (int)(k / (sw / 8)), o8 = (int)(k % (sw / 8));
        const uint8_t *p = src + (int64_t)c * W * H + (int64_t)(2 * qy) * W + 16 * o8;
        const uint4 a = __ldg((const uint4 *)p);
        const uint4 b = __ldg((const uint4 *)(p + W));
        const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
        uint32_t out[2] = {0, 0};
#pragma unroll
        for (int w = 0; w < 4; w++) {
            const int x0 = 16 * o8 + 4 * w;
            const int v0 = dec_tap4(aw[w] & 0xff, (aw[w] >> 8) & 0xff, bw[w] & 0xff, (bw[w] >> 8) & 0xff, x0, H, rgb);
            const int v1 = dec_tap4((aw[w] >> 16) & 0xff, aw[w] >> 24, (bw[w] >> 16) & 0xff, bw[w] >> 24, x0 + 2, H, rgb);
            out[w >> 1] |= ((uint32_t)v0 | ((uint32_t)v1 << 8)) << (16 * (w & 1));
        }
        *(uint2 *)(dec + (int64_t)c * sw * sh + (int64_t)qy * sw + 8 * o8) = make_uint2(out[0], out[1]);
    }
}

int launch_decimate(const uint8_t *d_src, uint8_t *d_dec, const Geom &g, cudaStream_t s)
{
    if (g.W % 16 == 0) {
        int64_t total = (int64_t)(g.sw / 8) * g.sh * g.C;
        int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
        if (blocks < 1) blocks = 1;
        k_decimate_v8<<<blocks, 256, 0, s>>>(d_src, d_dec, g.W, g.H, g.C);
        return 1;
    }
    int64_t total = (int64_t)(g.sw / 2) * g.sh * g.C;
    int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
    if (blocks < 1) blocks = 1;
    k_decimate<<<blocks, 256, 0, s>>>(d_src, d_dec, g.W, g.H, g.C);
    return 1;
}

// ------------------------------------------------------------------------------------
// K1c: per-domain integer sums (DB:92-115).  Domain j = (gy, gx) covers the BxB block
// of the decimated plane at (gx*step, gy*step) (FC:1027-1047).  sum d and sum d^2 are
// exact in s32; mean and variance follow from them (dom_var()).
// ------------------------------------------------------------------------------------
__global__ void k_domain_stats(const uint8_t *__restrict__ dec, int32_t *__restrict__ dsum,
                               int32_t *__restrict__ dsq, Geom g)
{
    int64_t total = g.ND * g.C;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int c = (int)(i / g.ND);
    int64_t j = i - c * g.ND;
    int gx = (int)(j % g.dpw), gy = (int)(j / g.dpw);
    const uint8_t *p = dec + (int64_t)c * g.sw * g.sh + (int64_t)(gy * g.step) * g.sw + gx * g.step;
    int s1 = 0, s2 = 0;
    for (int ry = 0; ry < g.B; ry++) {
        const uint8_t *row = p + (int64_t)ry * g.sw;
        for (int rx = 0; rx < g.B; rx++) {
            int v = __ldg(row + rx);
            s1 += v;
            s2 += v * v;
        }
    }
    dsum[i] = s1;
    dsq[i] = s2;
}

int launch_domain_stats(const uint8_t *d_dec, int32_t *d_dsum, int32_t *d_dsq, const Geom &g, cudaStream_t s)
{
    int64_t total = g.ND * g.C;
    k_domain_stats<<<(unsigned)((total + 127) / 128), 128, 0, s>>>(d_dec, d_dsum, d_dsq, g);
    return 1;
}

// K1d: per-range pixel sums (FC:67-73 getMittelwert of FC:588-602 getRangeblock).
__global__ void k_range_stats(const uint8_t *__restrict__ src, int32_t *__restrict__ rsum, Geom g)
{
    int64_t total = g.NR * g.C;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int c = (int)(i / g.NR);
    int64_t j = i - c * g.NR;
    int xr = (int)(j % g.rpw), yr = (int)(j / g.rpw);
    const uint8_t *p = src + (int64_t)c * g.W * g.H + (int64_t)(yr * g.B) * g.W + xr * g.B;
    int s1 = 0;
    for (int ry = 0; ry < g.B; ry++) {
        const uchar4 *row = (const uchar4 *)(p + (int64_t)ry * g.W);
        for (int rx = 0; rx < g.B / 4; rx++) {
            uchar4 v = __ldg(row + rx);
            s1 += v.x + v.y + v.z + v.w;
        }
    }
    rsum[i] = s1;
}

int launch_range_stats(const uint8_t *d_src, int32_t *d_rsum, const Geom &g, cudaStream_t s)
{
    int64_t total = g.NR * g.C;
    k_range_stats<<<(unsigned)((total + 127) / 128), 128, 0, s>>>(d_src, d_rsum, g);
    return 1;
}

// ------------------------------------------------------------------------------------
// K2w: direct windowed search.  One CTA per range block; threads stride over the wk*wk
// window candidates in ascending order, score each exactly as the reference does and
// keep the strict-< running minimum (FC:619-632); a lexicographic (error, index) block
// reduction then picks the lowest index among equal errors, which is what the
// reference's ascending loop with strict < yields.
// ------------------------------------------------------------------------------------
constexpr int kDirectThreads = 128;

__device__ __forceinline__ void block_argmin(float &err, int &c, float *s_err, int *s_c)
{
    warp_argmin(err, c);
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { s_err[warp] = err; s_c[warp] = c; }
    __syncthreads();
    if (threadIdx.x == 0)
        for (int w = 1; w < kDirectThreads / 32; w++) argmin_merge(err, c, s_err[w], s_c[w]);
}

// sum r * d over one candidate block with packed-byte dot products: kov = sum r d - rmean * sum d - dmean * vR
// (exact in s32).  s_rw = the range block as packed u8 words (raster order).  A block row of the decimated plane
// starts at a multiple of B / 4 bytes: 4-, 2- and 1-byte loads for B = 16, 8, 4.
template <int B>
__device__ __forceinline__ int grey_dot_raw(const uint32_t *s_rw, const uint8_t *__restrict__ p, int sw)
{
    int dot = 0;
#pragma unroll 4
    for (int ry = 0; ry < B; ry++) {
        const uint8_t *row = p + (int64_t)ry * sw;
#pragma unroll
        for (int w = 0; w < B / 4; w++) {
            uint32_t d4;
            if (B == 16) d4 = __ldg((const uint32_t *)(row + 4 * w));
            else if (B == 8) d4 = (uint32_t)__ldg((const uint16_t *)(row + 4 * w)) | ((uint32_t)__ldg((const uint16_t *)(row + 4 * w + 2)) << 16);
            else d4 = (uint32_t)__ldg(row) | ((uint32_t)__ldg(row + 1) << 8) | ((uint32_t)__ldg(row + 2) << 16) | ((uint32_t)__ldg(row + 3) << 24);
            dot = (int)__dp4a(s_rw[ry * (B / 4) + w], d4, (uint32_t)dot);
        }
    }
    return dot;
}

template <int B>
__global__ void __launch_bounds__(kDirectThreads)
k_search_direct_grey(const uint8_t *__restrict__ src, const uint8_t *__restrict__ dec,
                     const int32_t *__restrict__ dsum, const int32_t *__restrict__ dsq,
                     const int32_t *__restrict__ rsum, int32_t *__restrict__ best, Geom g, int64_t j0)
{
    constexpr int n = B * B;
    __shared__ uint32_t s_rw[n / 4];  // the range block, packed bytes
    __shared__ float s_err[kDirectThreads / 32];
    __shared__ int s_c[kDirectThreads / 32];
    int64_t j = j0 + blockIdx.x;
    int xr = (int)(j % g.rpw), yr = (int)(j / g.rpw);
    int rmean;
    const int vR = centred_sum(rsum[j], n, &rmean);
    for (int t = threadIdx.x; t < n / 4; t += kDirectThreads) {
        int ry = (4 * t) / B, rx = (4 * t) % B;  // 4-byte aligned: W, xr * B and rx are multiples of 4
        s_rw[t] = *(const uint32_t *)(src + (int64_t)(yr * B + ry) * g.W + xr * B + rx);
    }
    __syncthreads();
    int dy, dx;
    range_window(g, j, &dy, &dx);
    float best_err = 10000000.0f;  // FC:615
    int best_c = 0;
    int ncand = g.wk * g.wk;
    for (int c = threadIdx.x; c < ncand; c += kDirectThreads) {
        int ky = c / g.wk, kx = c - ky * g.wk;
        int gx = dx + kx, gy = dy + ky;
        int64_t idx = gx + (int64_t)gy * g.dpw;  // FC:145
        const uint8_t *p = dec + (int64_t)(gy * g.step) * g.sw + gx * g.step;
        const int ds = dsum[idx];
        int dmean;
        int varD = dom_var(ds, dsq[idx], n, &dmean);
        int kov = grey_dot_raw<B>(s_rw, p, g.sw) - rmean * ds - dmean * vR;  // sum (r-rmean)(d-dmean)
        float err = grey_error(kov, vR, __dsqrt_rn((double)varD));
        if (err < best_err) { best_err = err; best_c = c; }  // FC:627
    }
    block_argmin(best_err, best_c, s_err, s_c);
    if (threadIdx.x == 0) best[j] = best_c;
}

// RGB: one shared domain and contrast for the three channels (FC:760-808).  The
// covariance is accumulated sequentially in binary32 in pixel order exactly as the
// reference does (it is only guaranteed to be an exact integer for B <= 4).
struct RgbScore {
    float err, kov;
};

template <int B>
__device__ __forceinline__ RgbScore rgb_score(const float *s_gR, float vR, const uint16_t *dec3, const Geom &g,
                                              int gx, int gy, int dmsum, int vDi)
{
    // dec3 = R + G + B of the decimated planes, dmsum = the sum of the three integer channel means:
    // gD = (dR - mR) + (dG - mG) + (dB - mB) (FC:783-784, exact small integers in binary32) = dec3 - dmsum.
    // A block row starts at a multiple of B / 4 pixels: 2-, 4- and 8-byte loads for B = 4, 8, 16.
    constexpr int LW = B / 4;  // pixels per load
    const uint16_t *p = dec3 + (int64_t)(gy * g.step) * g.sw + gx * g.step;
    float kov = 0.0f;  // FC:775
#pragma unroll 2
    for (int ry = 0; ry < B; ry++) {
        const uint16_t *row = p + (int64_t)ry * g.sw;
#pragma unroll
        for (int rx = 0; rx < B; rx += LW) {
            uint32_t w[2];
            if (LW == 1) w[0] = __ldg(row + rx);
            else if (LW == 2) w[0] = __ldg((const uint32_t *)(row + rx));
            else { const uint2 v = __ldg((const uint2 *)(row + rx)); w[0] = v.x; w[1] = v.y; }
#pragma unroll
            for (int e = 0; e < LW; e++) {
                const float gD = (float)((int)((w[e >> 1] >> (16 * (e & 1))) & 0xffffu) - dmsum);
                kov = rgb_kov_step(kov, s_gR[ry * B + rx + e], gD);
            }
        }
    }
    RgbScore o;
    o.err = rgb_error(kov, vR, (float)vDi);
    o.kov = kov;
    return o;
}

// Loads (r - rmean) summed over the channels for the range block into smem (FC:785-786)
// and returns vR = sum of it (FC:790).  rm[] receives the per-channel integer means.
__device__ __forceinline__ float rgb_range_prep(const uint8_t *src, const int32_t *rsum, const Geom &g, int64_t j,
                                                float *s_gR, int rm[3])
{
    int xr = (int)(j % g.rpw), yr = (int)(j / g.rpw);
    int64_t plane = (int64_t)g.W * g.H;
    const int v = centred_sum_rgb(rsum, g.NR, j, g.n, rm);
    for (int t = threadIdx.x; t < g.n; t += blockDim.x) {
        int ry = t / g.B, rx = t % g.B;
        int64_t o = (int64_t)(yr * g.B + ry) * g.W + xr * g.B + rx;
        s_gR[t] = (float)(((int)src[o] - rm[0]) + ((int)src[plane + o] - rm[1]) + ((int)src[2 * plane + o] - rm[2]));
    }
    return (float)v;
}

template <int B>
__global__ void __launch_bounds__(kDirectThreads)
k_search_direct_rgb(const uint8_t *__restrict__ src, const uint16_t *__restrict__ dec3,
                    const int32_t *__restrict__ dsum, const int32_t *__restrict__ rsum,
                    int32_t *__restrict__ best, Geom g, int64_t j0)
{
    __shared__ float s_gR[256];
    __shared__ float s_err[kDirectThreads / 32];
    __shared__ int s_c[kDirectThreads / 32];
    int64_t j = j0 + blockIdx.x;
    int rm[3];
    float vR = rgb_range_prep(src, rsum, g, j, s_gR, rm);
    __syncthreads();
    int dy, dx;
    range_window(g, j, &dy, &dx);
    float best_err = 10000000.0f;  // FC:698
    int best_c = 0;
    int ncand = g.wk * g.wk;
    for (int c = threadIdx.x; c < ncand; c += kDirectThreads) {
        int ky = c / g.wk, kx = c - ky * g.wk;
        int gx = dx + kx, gy = dy + ky;
        int64_t idx = gx + (int64_t)gy * g.dpw;
        int dm[3];
        const int vDi = centred_sum_rgb(dsum, g.ND, idx, g.n, dm);
        RgbScore sc = rgb_score<B>(s_gR, vR, dec3, g, gx, gy, dm[0] + dm[1] + dm[2], vDi);
        if (sc.err < best_err) { best_err = sc.err; best_c = c; }  // FC:710
    }
    block_argmin(best_err, best_c, s_err, s_c);
    if (threadIdx.x == 0) best[j] = best_c;
}

// Isometry extension of k_search_direct_grey: every candidate is scored under the 8 isometries (inner loop,
// k ascending); best[j] = c * 8 + k of the lexicographic (error, c, k) minimum -- what an ascending
// (c, k) double loop with strict < yields.  s_rt[k][p] holds (r - rmean) of the range pixel that isometry k
// maps onto domain pixel p, so one pass over the domain block feeds all eight dot products.
__global__ void __launch_bounds__(kDirectThreads)
k_search_direct_grey_iso(const uint8_t *__restrict__ src, const uint8_t *__restrict__ dec,
                         const int32_t *__restrict__ dsum, const int32_t *__restrict__ dsq,
                         const int32_t *__restrict__ rsum, int32_t *__restrict__ best, Geom g, int64_t j0)
{
    __shared__ short s_rt[8][256];  // B <= 16
    __shared__ float s_err[kDirectThreads / 32];
    __shared__ int s_c[kDirectThreads / 32];
    int64_t j = j0 + blockIdx.x;
    int xr = (int)(j % g.rpw), yr = (int)(j / g.rpw);
    int rmean;
    const int vR = centred_sum(rsum[j], g.n, &rmean);
    for (int t = threadIdx.x; t < 8 * g.n; t += kDirectThreads) {
        int k = t / g.n, p = t % g.n;
        int ry, rx;  // the range pixel that T_k sends to domain pixel p
        iso_map(iso_inverse(k), g.B, p / g.B, p % g.B, &ry, &rx);
        s_rt[k][p] = (short)((int)src[(int64_t)(yr * g.B + ry) * g.W + xr * g.B + rx] - rmean);
    }
    __syncthreads();
    int dy, dx;
    range_window(g, j, &dy, &dx);
    float best_err = 10000000.0f;
    int best_c = 0;
    int ncand = g.wk * g.wk;
    for (int c = threadIdx.x; c < ncand; c += kDirectThreads) {
        int ky = c / g.wk, kx = c - ky * g.wk;
        int gx = dx + kx, gy = dy + ky;
        int64_t idx = gx + (int64_t)gy * g.dpw;
        const uint8_t *p = dec + (int64_t)(gy * g.step) * g.sw + gx * g.step;
        int dot[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (int sy = 0; sy < g.B; sy++) {
            const uint8_t *row = p + (int64_t)sy * g.sw;
            for (int sx = 0; sx < g.B; sx++) {
                const int d = (int)__ldg(row + sx);
#pragma unroll
                for (int k = 0; k < 8; k++) dot[k] += (int)s_rt[k][sy * g.B + sx] * d;
            }
        }
        int dmean;
        int varD = dom_var(dsum[idx], dsq[idx], g.n, &dmean);
        const double sqd = __dsqrt_rn((double)varD);
#pragma unroll
        for (int k = 0; k < 8; k++) {
            float err = grey_error(dot[k] - dmean * vR, vR, sqd);
            if (err < best_err) { best_err = err; best_c = c * 8 + k; }
        }
    }
    block_argmin(best_err, best_c, s_err, s_c);
    if (threadIdx.x == 0) best[j] = best_c;
}

// RGB: dec3 = R + G + B of the decimated planes (what k_search_direct_rgb reads instead of three planes).
__global__ void k_sum_planes(const uint8_t *__restrict__ dec, uint16_t *__restrict__ dec3, int64_t count)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) dec3[i] = (uint16_t)((int)dec[i] + (int)dec[count + i] + (int)dec[2 * count + i]);
}

int launch_sum_planes(const uint8_t *d_dec, uint16_t *d_dec3, const Geom &g, cudaStream_t s)
{
    const int64_t count = (int64_t)g.sw * g.sh;
    k_sum_planes<<<(unsigned)((count + 255) / 256), 256, 0, s>>>(d_dec, d_dec3, count);
    return 1;
}

int launch_search_direct(const Work &w, const Geom &g, int64_t j0, int64_t j1, cudaStream_t s)
{
    if (j1 <= j0) return 0;
    int64_t left = j1 - j0, at = j0;
    int launches = 0;
    while (left > 0) {  // grid.x limit is 2^31-1; chunk anyway to keep launches bounded
        unsigned chunk = (unsigned)(left < (1 << 30) ? left : (1 << 30));
        if (g.C == 1 && g.n_iso > 1)
            k_search_direct_grey_iso<<<chunk, kDirectThreads, 0, s>>>(w.src, w.dec, w.dsum, w.dsq, w.rsum, w.best, g, at);
        else if (g.C == 1 && g.B == 4)
            k_search_direct_grey<4><<<chunk, kDirectThreads, 0, s>>>(w.src, w.dec, w.dsum, w.dsq, w.rsum, w.best, g, at);
        else if (g.C == 1 && g.B == 8)
            k_search_direct_grey<8><<<chunk, kDirectThreads, 0, s>>>(w.src, w.dec, w.dsum, w.dsq, w.rsum, w.best, g, at);
        else if (g.C == 1)
            k_search_direct_grey<16><<<chunk, kDirectThreads, 0, s>>>(w.src, w.dec, w.dsum, w.dsq, w.rsum, w.best, g, at);
        else if (g.B == 4)
            k_search_direct_rgb<4><<<chunk, kDirectThreads, 0, s>>>(w.src, w.dec3, w.dsum, w.rsum, w.best, g, at);
        else if (g.B == 8)
            k_search_direct_rgb<8><<<chunk, kDirectThreads, 0, s>>>(w.src, w.dec3, w.dsum, w.rsum, w.best, g, at);
        else
            k_search_direct_rgb<16><<<chunk, kDirectThreads, 0, s>>>(w.src, w.dec3, w.dsum, w.rsum, w.best, g, at);
        left -= chunk;
        at += chunk;
        launches++;
    }
    return launches;
}


// ------------------------------------------------------------------------------------
// Solve + quantisation of a winning candidate, shared by the fused encode (K2f) and the code solve (K3s).
// ------------------------------------------------------------------------------------
// Quantisation scales of the code stream: written by FC:242-244 / FC:250-254, read back by FC:372-374 / FC:446-450.
constexpr float kGreyAScale = 100.0f, kRgbAScale = 1000000.0f, kRgbBScale = 100000.0f;

// Grey (FC:634-641): contrast a = kov / varD clamped to [-1, 1] -- 0/0 gives NaN on flat winners and NaN passes the
// clamp -- and brightness b = rmean - a * dmean.
__device__ __forceinline__ float2 grey_solve(int kov, int varD, int rmean, int dmean)
{
    float a = __fdiv_rn((float)kov, (float)varD);
    if (a < -1.0f) a = -1.0f;
    else if (a > 1.0f) a = 1.0f;
    return make_float2(a, __fsub_rn((float)rmean, __fmul_rn(a, (float)dmean)));
}

// RGB (FC:718-731): one contrast for the three channels over varianzSquare, which the reference computes as
// varianceR + varianceG + mittelWertB (FC:776, sic); one brightness per channel.  Returns {a, bR, bG, bB}.
__device__ __forceinline__ float4 rgb_solve(float kov, const int dv[3], const int dm[3], const int rm[3])
{
    float a = __fdiv_rn(kov, __fadd_rn(__fadd_rn((float)dv[0], (float)dv[1]), (float)dm[2]));
    if (a > 1.0f) a = 1.0f;
    if (a < -1.0f) a = -1.0f;
    return make_float4(a, __fsub_rn((float)rm[0], __fmul_rn(a, (float)dm[0])), __fsub_rn((float)rm[1], __fmul_rn(a, (float)dm[1])),
                       __fsub_rn((float)rm[2], __fmul_rn(a, (float)dm[2])));
}

// Code of range j for window candidate c: the floats into info and the quantised ints into q (FC:242-244), either
// optional.  iso: the isometry extension's fourth column kiso.
__device__ __forceinline__ void write_grey_code(float *info, int32_t *q, int64_t j, int c, float2 ab, bool iso, int kiso)
{
    const int S = iso ? 4 : 3;
    const float fc = (float)c;
    if (info) {
        info[S * j + 0] = fc;
        info[S * j + 1] = ab.x;
        info[S * j + 2] = ab.y;
        if (iso) info[S * j + 3] = (float)kiso;
    }
    if (q) {
        q[S * j + 0] = j_f2i(fc);
        q[S * j + 1] = j_f2i(__fmul_rn(ab.x, kGreyAScale));
        q[S * j + 2] = j_f2i(ab.y);
        if (iso) q[S * j + 3] = kiso;
    }
}

// RGB (FC:250-254): code = {c, a, bR, bG, bB}.
__device__ __forceinline__ void write_rgb_code(float *info, int32_t *q, int64_t j, int c, float4 ab)
{
    const float fc = (float)c;
    if (info) {
        info[5 * j + 0] = fc;
        info[5 * j + 1] = ab.x;
        info[5 * j + 2] = ab.y;
        info[5 * j + 3] = ab.z;
        info[5 * j + 4] = ab.w;
    }
    if (q) {
        q[5 * j + 0] = j_f2i(fc);
        q[5 * j + 1] = j_f2i(__fmul_rn(ab.x, kRgbAScale));
        q[5 * j + 2] = j_f2i(__fmul_rn(ab.y, kRgbBScale));
        q[5 * j + 3] = j_f2i(__fmul_rn(ab.z, kRgbBScale));
        q[5 * j + 4] = j_f2i(ab.w);
    }
}

// ------------------------------------------------------------------------------------
// K2f: fused windowed encode -- the reference's default configuration in ONE launch.
//
// For the windows the reference's GUI offers (widthKernel <= 16, RLEAppView.fxml:104) the whole chain
// scaleImage -> createCodebuch -> Domainblock stats -> window search -> solve -> quantise (FC:119-159 /
// FC:181-215) fits one CTA per range block: the CTA decimates the (wk-1)*B/4 + B pixel square of the source that
// its window covers into shared memory (a few KB; neighbouring ranges redo the overlap, which is cheaper than four
// more launches and three intermediate arrays), takes the range block's mean, scores the wk*wk candidates straight
// from shared memory with the same integer sums and the same float/double expression as the other paths, reduces
// to the lexicographic (error, index) minimum and lets thread 0 solve and quantise the winner.  Pixels come from the
// caller's ARGB ints (no unpack pass) or from 8-bit planes.  256^2, B = 8, wk = 2: 1024 CTAs, a few microseconds.
// ------------------------------------------------------------------------------------
template <int C, bool ARGB>
__device__ __forceinline__ void fused_px(const void *__restrict__ src, int64_t plane, int64_t o, int v[C])
{
    if (ARGB) {
        const uint32_t p = (uint32_t)__ldg((const int32_t *)src + o);
        v[0] = (p >> 16) & 0xff;  // grey: the red channel (FC:596, FC:977)
        if (C == 3) { v[1] = (p >> 8) & 0xff; v[C - 1] = p & 0xff; }
    } else {
#pragma unroll
        for (int c = 0; c < C; c++) v[c] = __ldg((const uint8_t *)src + c * plane + o);
    }
}

template <int B, int C, bool ARGB>
__global__ void __launch_bounds__(kDirectThreads)
k_encode_fused(const void *__restrict__ src, float *__restrict__ info, int32_t *__restrict__ q, Geom g, int64_t j0)
{
    constexpr int n = B * B, step = B / 4;
    extern __shared__ __align__(16) uint8_t s_tile[];  // C planes of TW x TW decimated pixels
    __shared__ int s_r[C][n];                          // the range block, per channel
    __shared__ float s_gR[C == 3 ? n : 1];             // RGB: sum over the channels of (r - rmean_c), FC:785-786
    __shared__ int s_sum[C][kDirectThreads / 32];
    __shared__ float s_err[kDirectThreads / 32];
    __shared__ int s_c[kDirectThreads / 32];
    const int64_t j = j0 + blockIdx.x;
    const int xr = (int)(j % g.rpw), yr = (int)(j / g.rpw);
    const int64_t plane = (int64_t)g.W * g.H;
    int dy, dx;
    range_window(g, j, &dy, &dx);
    const int TW = (g.wk - 1) * step + B;
    // ---- the window's decimated pixels (FC:970-1007 / FC:901-962, tap quirks as k_decimate)
    for (int t = threadIdx.x; t < TW * TW; t += kDirectThreads) {
        const int ty = t / TW, tx = t - ty * TW;
        const int x = 2 * (dx * step + tx), y = 2 * (dy * step + ty);
        int p00[C], p10[C], p01[C], p11[C];
        const int64_t o = (int64_t)y * g.W + x;
        fused_px<C, ARGB>(src, plane, o, p00);
        fused_px<C, ARGB>(src, plane, o + 1, p10);
        fused_px<C, ARGB>(src, plane, o + g.W, p01);
        fused_px<C, ARGB>(src, plane, o + g.W + 1, p11);
#pragma unroll
        for (int c = 0; c < C; c++) s_tile[c * TW * TW + t] = (uint8_t)dec_tap4(p00[c], p10[c], p01[c], p11[c], x, g.H, C == 3);
    }
    // ---- the range block and its integer means (FC:588-602, FC:67-73)
    int part[C];
#pragma unroll
    for (int c = 0; c < C; c++) part[c] = 0;
    for (int t = threadIdx.x; t < n; t += kDirectThreads) {
        int v[C];
        fused_px<C, ARGB>(src, plane, (int64_t)(yr * B + t / B) * g.W + xr * B + t % B, v);
#pragma unroll
        for (int c = 0; c < C; c++) { s_r[c][t] = v[c]; part[c] += v[c]; }
    }
#pragma unroll
    for (int c = 0; c < C; c++) {
        for (int o = 16; o > 0; o >>= 1) part[c] += __shfl_xor_sync(0xffffffffu, part[c], o);
        if ((threadIdx.x & 31) == 0) s_sum[c][threadIdx.x >> 5] = part[c];
    }
    __syncthreads();
    int rm[C], vR = 0;
#pragma unroll
    for (int c = 0; c < C; c++) {
        int rs = 0;
        for (int w = 0; w < kDirectThreads / 32; w++) rs += s_sum[c][w];
        vR += centred_sum(rs, n, &rm[c]);
    }
    if (C == 3) {
        for (int t = threadIdx.x; t < n; t += kDirectThreads)
            s_gR[t] = (float)((s_r[0][t] - rm[0]) + (s_r[C == 3 ? 1 : 0][t] - rm[C == 3 ? 1 : 0]) + (s_r[C - 1][t] - rm[C - 1]));
        __syncthreads();
    }
    // ---- candidates in ascending order per thread, strict < (FC:619-632 / FC:702-713)
    float best_err = 10000000.0f;  // FC:615 / FC:698
    int best_c = 0;
    const int ncand = g.wk * g.wk;
    for (int c = threadIdx.x; c < ncand; c += kDirectThreads) {
        const int ky = c / g.wk, kx = c - ky * g.wk;
        const uint8_t *p = s_tile + (ky * step) * TW + kx * step;
        float err;
        if (C == 1) {
            int ds = 0, dsq = 0, dot = 0;
            for (int ry = 0; ry < B; ry++)
#pragma unroll
                for (int rx = 0; rx < B; rx++) {
                    const int d = p[ry * TW + rx];
                    ds += d;
                    dsq += d * d;
                    dot += s_r[0][ry * B + rx] * d;
                }
            int dmean;
            const int varD = dom_var(ds, dsq, n, &dmean);
            const int kov = dot - rm[0] * ds - dmean * vR;  // sum (r - rmean)(d - dmean)
            err = grey_error(kov, vR, __dsqrt_rn((double)varD));
        } else {
            int dmsum = 0, vDi = 0;
#pragma unroll
            for (int ch = 0; ch < C; ch++) {
                int ds = 0;
                for (int ry = 0; ry < B; ry++)
#pragma unroll
                    for (int rx = 0; rx < B; rx++) ds += p[ch * TW * TW + ry * TW + rx];
                int dm;
                vDi += centred_sum(ds, n, &dm);
                dmsum += dm;
            }
            float kov = 0.0f;  // FC:775: sequential binary32 accumulation in pixel order
            for (int ry = 0; ry < B; ry++)
#pragma unroll
                for (int rx = 0; rx < B; rx++) {
                    const int o = ry * TW + rx;
                    const float gD = (float)((int)p[o] + (int)p[(C == 3 ? 1 : 0) * TW * TW + o] + (int)p[(C - 1) * TW * TW + o] - dmsum);
                    kov = rgb_kov_step(kov, s_gR[ry * B + rx], gD);
                }
            err = rgb_error(kov, (float)vR, (float)vDi);
        }
        if (err < best_err) { best_err = err; best_c = c; }  // FC:627 / FC:710
    }
    block_argmin(best_err, best_c, s_err, s_c);
    if (threadIdx.x != 0) return;
    // ---- solve + quantise the winner
    const int c = best_c;
    const int ky = c / g.wk, kx = c - ky * g.wk;
    const uint8_t *p = s_tile + (ky * step) * TW + kx * step;
    if constexpr (C == 1) {
        int ds = 0, dsq = 0, dot = 0;
        for (int ry = 0; ry < B; ry++)
            for (int rx = 0; rx < B; rx++) {
                const int d = p[ry * TW + rx];
                ds += d;
                dsq += d * d;
                dot += (s_r[0][ry * B + rx] - rm[0]) * d;
            }
        int dmean;
        const int varD = dom_var(ds, dsq, n, &dmean);
        write_grey_code(info, q, j, c, grey_solve(dot - dmean * vR, varD, rm[0], dmean), false, 0);
    } else {
        int dm[3], dv[3], dmsum = 0;
#pragma unroll
        for (int ch = 0; ch < C; ch++) {
            int ds = 0, dsq = 0;
            for (int ry = 0; ry < B; ry++)
                for (int rx = 0; rx < B; rx++) {
                    const int d = p[ch * TW * TW + ry * TW + rx];
                    ds += d;
                    dsq += d * d;
                }
            dv[ch] = dom_var(ds, dsq, n, &dm[ch]);
            dmsum += dm[ch];
        }
        float kov = 0.0f;
        for (int ry = 0; ry < B; ry++)
            for (int rx = 0; rx < B; rx++) {
                const int o = ry * TW + rx;
                const float gD = (float)((int)p[o] + (int)p[(C == 3 ? 1 : 0) * TW * TW + o] + (int)p[(C - 1) * TW * TW + o] - dmsum);
                kov = rgb_kov_step(kov, s_gR[ry * B + rx], gD);
            }
        write_rgb_code(info, q, j, c, rgb_solve(kov, dv, dm, rm));
    }
}

bool fused_encode_applicable(const Geom &g) { return g.wk <= 16 && g.n_iso == 1; }

template <int C, bool ARGB>
static int launch_fused_t(const void *d_src, const Geom &g, int64_t j0, int64_t j1, float *d_info, int32_t *d_q, cudaStream_t s)
{
    const int step = g.B / 4, TW = (g.wk - 1) * step + g.B;
    const size_t smem = (size_t)C * TW * TW;  // <= 3 * 76 * 76 = 17 KB
    int launches = 0;
    for (int64_t at = j0; at < j1;) {
        const unsigned chunk = (unsigned)(j1 - at < (1 << 30) ? j1 - at : (1 << 30));
        if (g.B == 4) k_encode_fused<4, C, ARGB><<<chunk, kDirectThreads, smem, s>>>(d_src, d_info, d_q, g, at);
        else if (g.B == 8) k_encode_fused<8, C, ARGB><<<chunk, kDirectThreads, smem, s>>>(d_src, d_info, d_q, g, at);
        else k_encode_fused<16, C, ARGB><<<chunk, kDirectThreads, smem, s>>>(d_src, d_info, d_q, g, at);
        at += chunk;
        launches++;
    }
    return launches;
}

int launch_encode_fused(const void *d_src, int src_is_argb, const Geom &g, int64_t j0, int64_t j1, float *d_info, int32_t *d_q,
                        cudaStream_t s)
{
    if (j1 <= j0) return 0;
    if (g.C == 1) return src_is_argb ? launch_fused_t<1, true>(d_src, g, j0, j1, d_info, d_q, s) : launch_fused_t<1, false>(d_src, g, j0, j1, d_info, d_q, s);
    return src_is_argb ? launch_fused_t<3, true>(d_src, g, j0, j1, d_info, d_q, s) : launch_fused_t<3, false>(d_src, g, j0, j1, d_info, d_q, s);
}

// ------------------------------------------------------------------------------------
// K3s: code solve + quantisation for the winning candidate.  One thread per range block.
// ------------------------------------------------------------------------------------
__global__ void k_solve_grey(const uint8_t *__restrict__ src, const uint8_t *__restrict__ dec,
                             const int32_t *__restrict__ dsum, const int32_t *__restrict__ dsq,
                             const int32_t *__restrict__ rsum, const int32_t *__restrict__ best,
                             float *__restrict__ info, int32_t *__restrict__ q, Geom g, int64_t j0, int64_t j1)
{
    int64_t j = j0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= j1) return;
    int xr = (int)(j % g.rpw), yr = (int)(j / g.rpw);
    const bool iso = g.n_iso > 1;  // extension: best = c * 8 + isometry
    int c = iso ? best[j] >> 3 : best[j];
    const int kiso = iso ? best[j] & 7 : 0;
    int dy, dx;
    range_window(g, j, &dy, &dx);
    int ky = c / g.wk, kx = c - ky * g.wk;
    int gx = dx + kx, gy = dy + ky;
    int64_t idx = gx + (int64_t)gy * g.dpw;
    int rmean;
    const int vR = centred_sum(rsum[j], g.n, &rmean);
    const uint8_t *pr = src + (int64_t)(yr * g.B) * g.W + xr * g.B;
    const uint8_t *pd = dec + (int64_t)(gy * g.step) * g.sw + gx * g.step;
    int dot = 0;
    for (int ry = 0; ry < g.B; ry++)
        for (int rx = 0; rx < g.B; rx++) {
            int sy = ry, sx = rx;
            if (iso) iso_map(kiso, g.B, ry, rx, &sy, &sx);
            dot += ((int)pr[(int64_t)ry * g.W + rx] - rmean) * (int)pd[(int64_t)sy * g.sw + sx];
        }
    int dmean;
    int varD = dom_var(dsum[idx], dsq[idx], g.n, &dmean);
    write_grey_code(info, q, j, c, grey_solve(dot - dmean * vR, varD, rmean, dmean), iso, kiso);
}

__global__ void k_solve_rgb(const uint8_t *__restrict__ src, const uint8_t *__restrict__ dec,
                            const int32_t *__restrict__ dsum, const int32_t *__restrict__ dsq,
                            const int32_t *__restrict__ rsum, const int32_t *__restrict__ best,
                            float *__restrict__ info, int32_t *__restrict__ q, Geom g, int64_t j0, int64_t j1)
{
    int64_t j = j0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= j1) return;
    int xr = (int)(j % g.rpw), yr = (int)(j / g.rpw);
    int c = best[j];
    int dy, dx;
    range_window(g, j, &dy, &dx);
    int ky = c / g.wk, kx = c - ky * g.wk;
    int gx = dx + kx, gy = dy + ky;
    int64_t idx = gx + (int64_t)gy * g.dpw;
    int rm[3], dm[3], dv[3];
    centred_sum_rgb(rsum, g.NR, j, g.n, rm);
    for (int ch = 0; ch < 3; ch++) dv[ch] = dom_var(dsum[(int64_t)ch * g.ND + idx], dsq[(int64_t)ch * g.ND + idx], g.n, &dm[ch]);
    const int dmsum = dm[0] + dm[1] + dm[2];
    int64_t planeS = (int64_t)g.W * g.H, planeD = (int64_t)g.sw * g.sh;
    const uint8_t *pr = src + (int64_t)(yr * g.B) * g.W + xr * g.B;
    const uint8_t *pd = dec + (int64_t)(gy * g.step) * g.sw + gx * g.step;
    float kov = 0.0f;
    for (int ry = 0; ry < g.B; ry++)
        for (int rx = 0; rx < g.B; rx++) {
            int64_t os = (int64_t)ry * g.W + rx, od = (int64_t)ry * g.sw + rx;
            const int gD = (int)pd[od] + (int)pd[planeD + od] + (int)pd[2 * planeD + od] - dmsum;
            const int gR = ((int)pr[os] - rm[0]) + ((int)pr[planeS + os] - rm[1]) + ((int)pr[2 * planeS + os] - rm[2]);
            kov = rgb_kov_step(kov, (float)gR, (float)gD);
        }
    write_rgb_code(info, q, j, c, rgb_solve(kov, dv, dm, rm));
}

int launch_solve(const Work &w, const Geom &g, int64_t j0, int64_t j1, float *d_info, int32_t *d_q, cudaStream_t s)
{
    if (j1 <= j0) return 0;
    unsigned blocks = (unsigned)((j1 - j0 + 127) / 128);
    if (g.C == 1)
        k_solve_grey<<<blocks, 128, 0, s>>>(w.src, w.dec, w.dsum, w.dsq, w.rsum, w.best, d_info, d_q, g, j0, j1);
    else
        k_solve_rgb<<<blocks, 128, 0, s>>>(w.src, w.dec, w.dsum, w.dsq, w.rsum, w.best, d_info, d_q, g, j0, j1);
    return 1;
}

// ------------------------------------------------------------------------------------
// K4: decoder.
// ------------------------------------------------------------------------------------

// Stream ints -> float codes (FC:372-374 / FC:446-450) and window-local -> codebook
// index (FC:853-893 calculateIndices, float division / float remainder as in Java).
// With `unquantised` the float codes of an encode are used instead (collage, FC:271).
// acc[1] is set when an index falls outside the pool (the reference would throw).
// packed != 0 (decoder loop over the row-pair interleaved plane, k_decode_sweep_il): doff[j] is the domain block's
// position in the decimated plane as (row << 16) | column instead of its byte offset.
__device__ __forceinline__ void dequant_one(int64_t j, const int32_t *__restrict__ q, const float *__restrict__ info_in,
                                            float *__restrict__ code, int32_t *__restrict__ doff, const Geom &g, int unquantised,
                                            unsigned long long *acc, int packed)
{
    int S = code_stride(g);
    float v[5];
    if (unquantised) {
        for (int k = 0; k < S; k++) v[k] = info_in[S * j + k];
    } else if (g.C == 1) {
        v[0] = (float)q[S * j];
        v[1] = __fdiv_rn((float)q[S * j + 1], kGreyAScale);
        v[2] = (float)q[S * j + 2];
        if (S == 4) v[3] = (float)(q[S * j + 3] & 7);  // isometry index (extension)
    } else {
        v[0] = (float)q[5 * j];
        v[1] = __fdiv_rn((float)q[5 * j + 1], kRgbAScale);
        v[2] = __fdiv_rn((float)q[5 * j + 2], kRgbBScale);
        v[3] = __fdiv_rn((float)q[5 * j + 3], kRgbBScale);
        v[4] = (float)q[5 * j + 4];
    }
    int dy, dx;
    range_window(g, j, &dy, &dx);
    float fwk = (float)g.wk;
    int yd = j_f2i(__fdiv_rn(v[0], fwk));  // FC:882
    int xd = j_f2i(fmodf(v[0], fwk));      // FC:883
    int64_t result = (int64_t)xd + dx + (int64_t)(yd + dy) * g.dpw;  // FC:886
    if (result < 0 || result >= g.ND) {
        atomicOr(acc + 1, 1ull);
        result = 0;
    }
    v[0] = (float)(int)result;  // FC:888 stores the index back into the float table
    for (int k = 0; k < S; k++) code[S * j + k] = v[k];
    // position of the domain block (FC:394 codebuch[(int) imgData[i][0]]) inside a decimated plane: its byte offset, or
    // (packed) row and column
    const int idx = j_f2i(v[0]);
    const int drow = (idx / g.dpw) * g.step, dcol = (idx % g.dpw) * g.step;
    doff[j] = packed ? (int32_t)(((uint32_t)drow << 16) | (uint32_t)dcol) : drow * g.sw + dcol;
}

__global__ void k_dequant(const int32_t *__restrict__ q, const float *__restrict__ info_in,
                          float *__restrict__ code, int32_t *__restrict__ doff, Geom g, int unquantised,
                          unsigned long long *acc, int packed)
{
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= g.NR) return;
    dequant_one(j, q, info_in, code, doff, g, unquantised, acc, packed);
}

int launch_dequant(const int32_t *d_q, float *d_code, int32_t *d_off, const Geom &g, int unquantised,
                   const float *d_info, unsigned long long *d_acc, int packed, cudaStream_t s)
{
    k_dequant<<<(unsigned)((g.NR + 127) / 128), 128, 0, s>>>(d_q, d_info, d_code, d_off, g, unquantised, d_acc, packed);
    return 1;
}

__global__ void k_fill(uint4 *p, int64_t n16, uint32_t v)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n16; i += stride) p[i] = make_uint4(v, v, v, v);
}

int launch_fill(uint8_t *d_planes, size_t bytes, int value, cudaStream_t s)
{
    uint32_t v = (uint32_t)(value & 0xff) * 0x01010101u;
    int64_t n16 = (int64_t)(bytes / 16);  // plane sizes are multiples of 16 (W % 4 == 0, H % 4 == 0)
    int blocks = (int)((n16 + 255) / 256 < 148 * 8 ? (n16 + 255) / 256 : 148 * 8);
    if (blocks < 1) blocks = 1;
    k_fill<<<blocks, 256, 0, s>>>((uint4 *)d_planes, n16, v);
    return 1;
}

// Decoder state block (device memory, 8 x u64; fic_api.cu owns it): [0] sum of squared pixel changes of the running
// sweep, [1] "a code indexes outside the pool", then as 32-bit words from [2]: ticket counter of the running sweep,
// done flag, sweeps executed, avgError bits.
enum { ST_TICKET = 4, ST_DONE = 5, ST_ITERS = 6, ST_AVG = 7 };  // indices into (uint32_t *)st

// Sweeps are enqueued ahead of the host's knowledge of convergence (FC:414): once the done flag is set every later
// sweep returns at once, so the image stays the converged one.
__device__ __forceinline__ bool sweep_done(const SweepCtl &ctl)
{
    return ctl.st && ((volatile const uint32_t *)ctl.st)[ST_DONE] != 0;
}

// Records sweep `it` whose float running sum of squared changes is `sum` (FC:407 / FC:493): avgError = sum / (W*H)
// (FC:413); below 1 the decode has converged and stops with that value (FC:414), otherwise the value is kept only
// after the last allowed sweep (FC:416-417).
__device__ __forceinline__ void record_sweep(uint32_t *w, int it, float sum, float fwh, bool last)
{
    const float avg = __fdiv_rn(sum, fwh);
    w[ST_ITERS] = (uint32_t)(it + 1);
    if (avg < 1.0f) {
        w[ST_AVG] = __float_as_uint(avg);
        w[ST_DONE] = 1u;
    } else {
        w[ST_AVG] = last ? __float_as_uint(avg) : 0u;
    }
}

// Sum of `local` over the CTA (blockDim.x == 256), valid in thread 0.
__device__ __forceinline__ unsigned long long cta_sum(unsigned long long local)
{
    __shared__ unsigned long long s_part[8];
    for (int o = 16; o > 0; o >>= 1) local += __shfl_down_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = local;
    __syncthreads();
    unsigned long long tot = 0;
    if (threadIdx.x == 0)
        for (int wv = 0; wv < 8; wv++) tot += s_part[wv];
    return tot;
}

// Common tail of the sweep kernels: add the CTA's squared changes to st[0]; with ctl.finish the last CTA to get
// here records the sweep (no separate kernel, no host round trip per sweep).  fic_api.cu only asks for that on
// sweeps whose float running sum needs no replay: it is the exact integer S when S < 2^24 (every float partial sum
// is then exact); S >= 2^24 >= W*H means "not converged" and the value is discarded (never the last sweep here).
__device__ __forceinline__ void sweep_tail(const SweepCtl &ctl, unsigned long long local)
{
    if (!ctl.st) return;
    const unsigned long long tot = cta_sum(local);
    if (threadIdx.x == 0) {
        if (tot) atomicAdd(ctl.st, tot);
        if (!ctl.finish) return;
        __threadfence();
        uint32_t *w = (uint32_t *)ctl.st;
        if (atomicAdd(w + ST_TICKET, 1u) == gridDim.x - 1) {
            __threadfence();
            const unsigned long long S = atomicExch(ctl.st, 0ull);
            w[ST_TICKET] = 0u;
            record_sweep(w, ctl.it, S < (1ull << 24) ? (float)S : 2.0f * ctl.fwh, ctl.fwh, false);
        }
    }
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

// One Jacobi sweep of FC:386-412 / FC:463-499.  The reference snapshots the codebook
// of the current image (FC:382), then rewrites every pixel from it; here the snapshot
// is the 2x-decimated plane `dec_in` of the current image, and the sweep emits the
// decimated plane of the image it writes (`dec_out`), so the next sweep needs no
// separate decimation pass.  One thread owns a 2x2 pixel quad (same range block, same
// code): 4 gathered domain bytes in, 4 image bytes + 1 decimated byte out per channel.
//   acc[0] += sum of squared pixel changes (exact integer; see fic_api.cu for how this
//   reproduces the reference's float avgError), perr (optional) gets the per-pixel
//   squared change in the reference's accumulation order (range-major, ry, rx).
template <int C>
__global__ void __launch_bounds__(256)
k_decode_sweep(const uint8_t *__restrict__ dec_in, uint8_t *__restrict__ img, uint8_t *__restrict__ dec_out,
               const float *__restrict__ code, const int32_t *__restrict__ doff, Geom g, SweepCtl ctl,
               int32_t *__restrict__ perr)
{
    if (sweep_done(ctl)) return;
    unsigned long long *const acc = ctl.st;
    int qw = g.W / 2;
    int64_t quads = (int64_t)qw * (g.H / 2);
    unsigned long long local = 0;
    // grid-stride: a bounded number of CTAs, so that the sweep's sum costs one atomic per CTA, not per warp
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < quads; t += (int64_t)gridDim.x * blockDim.x) {
        int qy = (int)(t / qw), qx = (int)(t - (int64_t)qy * qw);
        int x = 2 * qx, y = 2 * qy;
        int xr = x / g.B, yr = y / g.B;
        int rx = x - xr * g.B, ry = y - yr * g.B;
        int64_t j = (int64_t)yr * g.rpw + xr;
        const int S = code_stride(g);
        const float *cd = code + S * j;
        float a = cd[1];
        const int off = doff[j];
        int64_t planeI = (int64_t)g.W * g.H, planeD = (int64_t)g.sw * g.sh;
        int e[4] = {0, 0, 0, 0};
        // domain pixel of each of the quad's four range pixels: the same position, or (isometry extension,
        // grey only) the position the range's isometry maps it to
        int o00 = ry * g.sw + rx, o10 = o00 + 1, o01 = o00 + g.sw, o11 = o01 + 1;
        if (C == 1 && g.n_iso > 1) {
            const int kiso = j_f2i(cd[3]);
            int sy, sx;
            iso_map(kiso, g.B, ry, rx, &sy, &sx);         o00 = sy * g.sw + sx;
            iso_map(kiso, g.B, ry, rx + 1, &sy, &sx);     o10 = sy * g.sw + sx;
            iso_map(kiso, g.B, ry + 1, rx, &sy, &sx);     o01 = sy * g.sw + sx;
            iso_map(kiso, g.B, ry + 1, rx + 1, &sy, &sx); o11 = sy * g.sw + sx;
        }
#pragma unroll
        for (int c = 0; c < C; c++) {
            float b = cd[2 + c];
            const uint8_t *pd = dec_in + c * planeD + off;
            const int v00 = (int)decode_px(a, b, pd[o00]), v10 = (int)decode_px(a, b, pd[o10]);
            const int v01 = (int)decode_px(a, b, pd[o01]), v11 = (int)decode_px(a, b, pd[o11]);
            uint8_t *pi = img + c * planeI + (int64_t)y * g.W + x;
            uchar2 o0 = *(uchar2 *)pi, o1 = *(uchar2 *)(pi + g.W);
            e[0] += (o0.x - v00) * (o0.x - v00);  // FC:407 / FC:493
            e[1] += (o0.y - v10) * (o0.y - v10);
            e[2] += (o1.x - v01) * (o1.x - v01);
            e[3] += (o1.y - v11) * (o1.y - v11);
            *(uchar2 *)pi = make_uchar2(v00, v10);
            *(uchar2 *)(pi + g.W) = make_uchar2(v01, v11);
            if (dec_out) dec_out[c * planeD + (int64_t)qy * g.sw + qx] = (uint8_t)dec_tap4(v00, v10, v01, v11, x, g.H, C == 3);
        }
        local += (unsigned long long)(e[0] + e[1] + e[2] + e[3]);
        if (perr) {
            int32_t *pe = perr + j * g.n + ry * g.B + rx;
            pe[0] = e[0];
            pe[1] = e[1];
            pe[g.B] = e[2];
            pe[g.B + 1] = e[3];
        }
    }
    sweep_tail(ctl, local);
}

// Vector path (W % 8 == 0): one thread owns an 8 x 2 pixel strip (four quads): 8-byte loads of the old
// pixels, 8-byte stores of the new ones, one 4-byte store of the new decimated pixels; the 16 domain
// bytes are gathered from the (L2-resident) decimated plane.

// FIRST: the sweep that starts from the constant-128 image (FC:360): every old pixel and every domain pixel is 128,
// so nothing is read -- the start image and its decimated plane are never materialised (B >= 8 only).
template <int C, bool FIRST = false>
__global__ void __launch_bounds__(256)
k_decode_sweep_v8(const uint8_t *__restrict__ dec_in, uint8_t *__restrict__ img, uint8_t *__restrict__ dec_out,
                  const float *__restrict__ code, const int32_t *__restrict__ doff, Geom g, SweepCtl ctl,
                  int32_t *__restrict__ perr)
{
    if (sweep_done(ctl)) return;
    const int sw8 = g.W / 8;
    const int64_t strips = (int64_t)sw8 * (g.H / 2);
    unsigned long long local = 0;
    constexpr int S = C == 1 ? 3 : 5;
    const int64_t planeI = (int64_t)g.W * g.H, planeD = (int64_t)g.sw * g.sh;
    const int lb = __ffs(g.B) - 1, bm = g.B - 1;  // B is a power of two
    // B >= 8: the strip lies inside ONE range block -- one code, one domain offset, and the 2 x 8 domain bytes
    // are two runs of 8 contiguous bytes, read as 16-bit words at B = 8 (2-byte aligned: the domain grid stride B/4
    // is even) and as 32-bit words at B = 16 (stride 4).  B = 4: a strip spans two range blocks; every quad fetches
    // its own code and bytes.
    const bool one_range = g.B >= 8;
    const bool wide = (g.step & 3) == 0;
    // 32-bit strip arithmetic (strips = W * H / 16 < 2^31): a 64-bit division per strip was a quarter of the kernel's instructions
    const uint32_t nstrips = (uint32_t)strips, usw8 = (uint32_t)sw8;
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < nstrips; t += gridDim.x * blockDim.x) {
        const uint32_t uqy = t / usw8;
        const int qy = (int)uqy, s8 = (int)(t - uqy * usw8);
        const int y = 2 * qy, x0 = 8 * s8;
        const int yr = y >> lb, ry = y & bm;
        const int jr0 = yr * g.rpw + (x0 >> lb);
        float a0 = 0.0f;
        int off0 = 0;
        if (one_range) {
            a0 = __ldg(code + S * jr0 + 1);
            if (!FIRST) off0 = __ldg(doff + jr0) + ry * g.sw + (x0 & bm);
        }
        uint32_t esq[4][C];  // per quad: packed |old - new| of its four pixels (only unpacked when perr is asked for)
#pragma unroll
        for (int c = 0; c < C; c++) {
            uint8_t *pi = img + c * planeI + (int64_t)y * g.W + x0;
            uint2 o0 = make_uint2(0x80808080u, 0x80808080u), o1 = o0;
            if (!FIRST) {
                o0 = *(const uint2 *)pi;
                o1 = *(const uint2 *)(pi + g.W);
            }
            const uint32_t old0[2] = {o0.x, o0.y}, old1[2] = {o1.x, o1.y};
            uint32_t n0[2] = {0, 0}, n1[2] = {0, 0}, nd = 0;
            uint32_t dr0[4], dr1[4];  // domain bytes of the four quads: row ry (low 16 bits hold 2 pixels) and ry + 1
            float bq = 0.0f;
            if (one_range) {
                bq = __ldg(code + S * jr0 + 2 + c);
                if (FIRST) {
#pragma unroll
                    for (int qd = 0; qd < 4; qd++) dr0[qd] = dr1[qd] = 0x8080u;
                } else if (wide) {
                    const uint32_t *pw = (const uint32_t *)(dec_in + c * planeD + off0);
                    const uint32_t *pw1 = (const uint32_t *)(dec_in + c * planeD + off0 + g.sw);
#pragma unroll
                    for (int h = 0; h < 2; h++) {
                        const uint32_t w0 = __ldg(pw + h), w1 = __ldg(pw1 + h);
                        dr0[2 * h] = w0 & 0xffffu; dr0[2 * h + 1] = w0 >> 16;
                        dr1[2 * h] = w1 & 0xffffu; dr1[2 * h + 1] = w1 >> 16;
                    }
                } else {
                    const uint16_t *pd = (const uint16_t *)(dec_in + c * planeD + off0);
                    const uint16_t *pd1 = (const uint16_t *)(dec_in + c * planeD + off0 + g.sw);
#pragma unroll
                    for (int qd = 0; qd < 4; qd++) {
                        dr0[qd] = __ldg(pd + qd);
                        dr1[qd] = __ldg(pd1 + qd);
                    }
                }
            }
#pragma unroll
            for (int qd = 0; qd < 4; qd++) {
                const int x = x0 + 2 * qd;
                float a = a0, b = bq;
                if (!one_range) {
                    const int xr = x >> lb, rx = x & bm;
                    const int64_t jr = (int64_t)yr * g.rpw + xr;
                    const float *cd = code + S * jr;
                    a = cd[1];
                    b = cd[2 + c];
                    const uint8_t *pd = dec_in + c * planeD + doff[jr] + ry * g.sw + rx;
                    dr0[qd] = (uint32_t)pd[0] | ((uint32_t)pd[1] << 8);
                    dr1[qd] = (uint32_t)pd[g.sw] | ((uint32_t)pd[g.sw + 1] << 8);
                }
                const uint32_t v00 = decode_px(a, b, dr0[qd] & 0xffu), v10 = decode_px(a, b, dr0[qd] >> 8);
                const uint32_t v01 = decode_px(a, b, dr1[qd] & 0xffu), v11 = decode_px(a, b, dr1[qd] >> 8);
                const int sh = 16 * (qd & 1);
                const uint32_t newq = v00 | (v10 << 8) | (v01 << 16) | (v11 << 24);
                const uint32_t oldq = ((old0[qd >> 1] >> sh) & 0xffffu) | (((old1[qd >> 1] >> sh) & 0xffffu) << 16);
                const uint32_t ad = __vabsdiffu4(oldq, newq);
                esq[qd][c] = ad;
                local += (unsigned long long)__dp4a(ad, ad, 0u);  // FC:407 / FC:493: sum of the squared pixel changes
                n0[qd >> 1] |= (newq & 0xffffu) << sh;
                n1[qd >> 1] |= (newq >> 16) << sh;
                nd |= (uint32_t)dec_tap4((int)v00, (int)v10, (int)v01, (int)v11, x, g.H, C == 3) << (8 * qd);
            }
            *(uint2 *)pi = make_uint2(n0[0], n0[1]);
            *(uint2 *)(pi + g.W) = make_uint2(n1[0], n1[1]);
            if (dec_out) *(uint32_t *)(dec_out + c * planeD + (int64_t)qy * g.sw + 4 * s8) = nd;
        }
        if (perr) {  // per-pixel squared change, summed over the channels, in the reference's loop order
#pragma unroll
            for (int qd = 0; qd < 4; qd++) {
                const int x = x0 + 2 * qd;
                const int xr = x >> lb, rx = x & bm;
                int e[4] = {0, 0, 0, 0};
#pragma unroll
                for (int c = 0; c < C; c++)
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const int d = (int)((esq[qd][c] >> (8 * k)) & 0xffu);
                        e[k] += d * d;
                    }
                int32_t *pe = perr + ((int64_t)yr * g.rpw + xr) * g.n + ry * g.B + rx;
                pe[0] = e[0];
                pe[1] = e[1];
                pe[g.B] = e[2];
                pe[g.B + 1] = e[3];
            }
        }
    }
    sweep_tail(ctl, local);
}

// Decoder-loop sweep for B >= 8 and W % 16 == 0 over a ROW-PAIR INTERLEAVED decimated plane.  What a sweep pays for is
// L2 sectors (DESIGN 4.5): on a plain plane the two 8-byte domain row pieces of a strip lie in two different 32-byte
// sectors (2.4 sectors per strip with the pieces that straddle one), three quarters of which is over-fetch.  A strip
// always needs the decimated rows 2k and 2k + 1 of one pair (domain rows start at multiples of B/4 >= 2, strips at even
// rows), and the decoder owns both sides of the plane -- every sweep writes the plane the next one reads.  It
// therefore keeps the two rows of a pair interleaved at 8-byte granularity,
//     byte (y, x)  ->  (y >> 1) * 2 sw + (x >> 3) * 16 + (y & 1) * 8 + (x & 7),
// so that both pieces of a strip sit in one aligned 16-byte group, or in two adjacent groups when the domain column is
// not a multiple of 8: one or two 16-byte loads (1.4 sectors per strip) instead of eight 2-byte loads, and the writer
// still stores its four decimated bytes as one aligned word.  Arithmetic, error sums and the perr order are those
// of k_decode_sweep_v8; dpos[j] = (row << 16) | column of range j's domain block (k_dequant, packed).
// Used while the image and the two decimated planes stay L2-resident from sweep to sweep (48 MB: grey up to ~5800^2,
// RGB up to ~3300^2): there the sweep is bound by L2 sectors and the interleaved plane saves a quarter of them (grey
// 4096^2: 18.9 -> 15.7 us per sweep; RGB 3072^2: 26.1 -> 22.5).  Beyond L2 it measured slower than the plain plane
// (RGB at 4096^2, 75 MB of planes: 72-95 against 40 us per sweep), so larger images keep k_decode_sweep_v8.
__host__ __device__ inline bool sweep_interleaved(const Geom &g)
{
    return g.B >= 8 && g.W % 16 == 0 && g.n_iso == 1 && g.C * ((int64_t)g.W * g.H + 2 * (int64_t)g.sw * g.sh) <= ((int64_t)48 << 20);
}

__device__ __forceinline__ uint32_t decode_row4(float a, float b, uint32_t dom4)
{
    return decode_px(a, b, dom4 & 0xffu) | (decode_px(a, b, (dom4 >> 8) & 0xffu) << 8) |
           (decode_px(a, b, (dom4 >> 16) & 0xffu) << 16) | (decode_px(a, b, dom4 >> 24) << 24);
}

// The sweep itself (all strips this CTA owns); returns the thread's sum of squared pixel changes.  NC: the codes and
// the plane read are constant for the lifetime of the kernel (one launch per sweep) and go through the read-only path;
// the one-launch decoder (k_decode_small) rewrites them between its barriers and reads them with ordinary loads.
template <bool NC, class T>
__device__ __forceinline__ T sweep_ld(const T *p)
{
    if (NC) return __ldg(p);
    return *p;
}

template <int C, int B, bool PERR, bool FIRST, bool NC = true>
__device__ __forceinline__ unsigned long long sweep_il_body(const uint8_t *__restrict__ dec_in, uint8_t *__restrict__ img,
                                                            uint8_t *__restrict__ dec_out, const float *__restrict__ code,
                                                            const int32_t *__restrict__ dpos, const Geom &g, int32_t *__restrict__ perr)
{
    constexpr int LB = B == 8 ? 3 : 4, BM = B - 1, S = C == 1 ? 3 : 5;
    const uint32_t W = (uint32_t)g.W, sw = (uint32_t)g.sw, rpw = (uint32_t)g.rpw;
    const uint32_t sw8 = W >> 3;
    const size_t planeI = (size_t)g.W * g.H, planeD = (size_t)g.sw * g.sh;
    const uint32_t tap_x = (uint32_t)g.H - 1u;  // dec_tap4: columns x >= H - 1 take the constant 128 as their fourth tap
    unsigned long long local = 0;
    // A warp owns a tile of 16 x 2 strips: lanes 0-15 the strips of decimated row 2 tr, lanes 16-31 the same columns of
    // row 2 tr + 1 -- the two rows of one interleaved pair, so that the warp's one store of decimated pixels writes whole
    // 32-byte sectors (half-written sectors cost a read-modify-write once the planes no longer fit in L2).
    const uint32_t tiles_x = (sw8 + 15u) >> 4, tiles = tiles_x * ((uint32_t)g.H >> 2);
    const uint32_t lane = threadIdx.x & 31u;
    for (uint32_t wt = blockIdx.x * 8u + (threadIdx.x >> 5); wt < tiles; wt += gridDim.x * 8u) {
        const uint32_t tr = wt / tiles_x, tx = wt - tr * tiles_x;
        const uint32_t qy = 2u * tr + (lane >> 4), s8 = 16u * tx + (lane & 15u);
        if (s8 >= sw8) continue;
        const uint32_t y = 2u * qy, x0 = 8u * s8;
        const uint32_t jr = (y >> LB) * rpw + (x0 >> LB);
        const float a = sweep_ld<NC>(code + S * jr + 1);
        uint32_t gbase = 0, o = 0;
        if (!FIRST) {
            const uint32_t pos = (uint32_t)sweep_ld<NC>(dpos + jr);
            const uint32_t yd = (pos >> 16) + (y & BM), xd = (pos & 0xffffu) + (x0 & BM);  // yd is even
            gbase = (yd >> 1) * (2u * sw) + (xd >> 3) * 16u;
            o = xd & 7u;  // even
        }
        uint8_t *pi = img + (size_t)y * W + x0;
        uint32_t sq = 0;
        uint32_t e[PERR ? 16 : 1];
        if (PERR)
#pragma unroll
            for (int k = 0; k < 16; k++) e[k] = 0;
#pragma unroll
        for (int c = 0; c < C; c++) {
            const float b = sweep_ld<NC>(code + S * jr + 2 + c);
            uint2 d0 = make_uint2(0x80808080u, 0x80808080u), d1 = d0, o0 = d0, o1 = d0;
            if (!FIRST) {
                const uint8_t *pg = dec_in + c * planeD + gbase;
                const uint4 ga = sweep_ld<NC>((const uint4 *)pg);
                uint4 gb = ga;  // not used when the column is a multiple of 8
                if (o) gb = sweep_ld<NC>((const uint4 *)(pg + 16));
                // row ry: bytes o .. o + 7 of the words {ga.x, ga.y, gb.x, gb.y}; row ry + 1: of {ga.z, ga.w, gb.z, gb.w}
                const uint32_t sh = (o & 3u) * 8u;
                const bool up = o >= 4u;
                d0.x = __funnelshift_r(up ? ga.y : ga.x, up ? gb.x : ga.y, sh);
                d0.y = __funnelshift_r(up ? gb.x : ga.y, up ? gb.y : gb.x, sh);
                d1.x = __funnelshift_r(up ? ga.w : ga.z, up ? gb.z : ga.w, sh);
                d1.y = __funnelshift_r(up ? gb.z : ga.w, up ? gb.w : gb.z, sh);
                o0 = *(const uint2 *)(pi + c * planeI);
                o1 = *(const uint2 *)(pi + c * planeI + W);
            }
            uint2 n0, n1;
            n0.x = decode_row4(a, b, d0.x);
            if (FIRST) {  // one domain value: every pixel of the strip is the same
                n0.y = n0.x; n1 = n0;
            } else {
                n0.y = decode_row4(a, b, d0.y);
                n1.x = decode_row4(a, b, d1.x);
                n1.y = decode_row4(a, b, d1.y);
            }
            *(uint2 *)(pi + c * planeI) = n0;
            *(uint2 *)(pi + c * planeI + W) = n1;
            const uint32_t ad[4] = {__vabsdiffu4(o0.x, n0.x), __vabsdiffu4(o0.y, n0.y), __vabsdiffu4(o1.x, n1.x), __vabsdiffu4(o1.y, n1.y)};
#pragma unroll
            for (int k = 0; k < 4; k++) {
                sq = __dp4a(ad[k], ad[k], sq);  // FC:407 / FC:493: sum of the squared pixel changes
                if (PERR)
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        const uint32_t d = (ad[k] >> (8 * i)) & 0xffu;
                        e[4 * k + i] += d * d;
                    }
            }
            if (dec_out) {
                // 2x decimation of the new pixels (dec_tap4): quads (x0 + 2 qd, y), bytes {p00, p10, p01, p11}
                const uint32_t quad[4] = {__byte_perm(n0.x, n1.x, 0x5410), __byte_perm(n0.x, n1.x, 0x7632),
                                          __byte_perm(n0.y, n1.y, 0x5410), __byte_perm(n0.y, n1.y, 0x7632)};
                uint32_t nd = 0;
#pragma unroll
                for (int qd = 0; qd < 4; qd++) {
                    const bool edge = x0 + 2u * qd >= tap_x;
                    const uint32_t wts = edge ? 0x00010101u : (C == 3 ? 0x00020101u : 0x01010101u);
                    nd |= ((__dp4a(quad[qd], wts, edge ? 128u : 0u) >> 2) & 0xffu) << (8 * qd);
                }
                // decimated row qy, columns 4 s8 .. 4 s8 + 3, in the interleaved plane
                *(uint32_t *)(dec_out + c * planeD + (size_t)(qy >> 1) * (2u * sw) + (s8 >> 1) * 16u + (qy & 1u) * 8u + (s8 & 1u) * 4u) = nd;
            }
        }
        local += sq;
        if (PERR) {  // per-pixel squared change, summed over the channels, in the reference's loop order
            int4 *pe = (int4 *)(perr + (size_t)jr * (B * B) + (y & BM) * B + (x0 & BM));
            pe[0] = make_int4((int)e[0], (int)e[1], (int)e[2], (int)e[3]);
            pe[1] = make_int4((int)e[4], (int)e[5], (int)e[6], (int)e[7]);
            pe[B / 4] = make_int4((int)e[8], (int)e[9], (int)e[10], (int)e[11]);
            pe[B / 4 + 1] = make_int4((int)e[12], (int)e[13], (int)e[14], (int)e[15]);
        }
    }
    return local;
}

template <int C, int B, bool PERR, bool FIRST>
__global__ void __launch_bounds__(256)
k_decode_sweep_il(const uint8_t *__restrict__ dec_in, uint8_t *__restrict__ img, uint8_t *__restrict__ dec_out,
                  const float *__restrict__ code, const int32_t *__restrict__ dpos, Geom g, SweepCtl ctl,
                  int32_t *__restrict__ perr)
{
    if (sweep_done(ctl)) return;
    sweep_tail(ctl, sweep_il_body<C, B, PERR, FIRST>(dec_in, img, dec_out, code, dpos, g, perr));
}

// ---- small images: the whole decode in ONE cooperative launch ------------------------------------------------------
// The reference's default setting (256^2, B = 8) is launch bound on the GPU: code dequantisation, five to nine sweeps of
// ~2 us each, the output conversion -- a dozen launches of ~2.5 us each.  k_decode_small runs all of it in one
// cooperative kernel (every CTA resident; a grid barrier on a counter in the state block between the phases): dequantise,
// then sweep / barrier / fold (one thread decides FC:413-417) / barrier until the sweep converges, then write the ARGB
// ints.  It takes the cases whose avgError needs no replay of the float sum: the exact total is below 2^24 and nothing
// is carried in (the float sum IS that integer), or the total is so large that the sweep certainly did not converge
// (skip_from_of) and is not the last allowed one.  Anything else -- a last sweep that has not converged, a
// carried-in avgError on a sweep that might converge -- sets the bail word and the host repeats the decode through the
// per-sweep kernels.
enum { ST_BARRIER = 8, ST_BAIL = 9 };  // further 32-bit words of the state block

__device__ __forceinline__ void grid_barrier(uint32_t *counter, uint32_t &epoch)
{
    __syncthreads();
    if (threadIdx.x == 0) {
        epoch += gridDim.x;
        __threadfence();
        atomicAdd(counter, 1u);
        while (*(volatile uint32_t *)counter < epoch) {}
        __threadfence();
    }
    __syncthreads();
}

template <int C, int B>
__global__ void __launch_bounds__(256)
k_decode_small(const int32_t *__restrict__ q, float *__restrict__ code, int32_t *__restrict__ dpos, uint8_t *__restrict__ img,
               uint8_t *__restrict__ dec_a, uint8_t *__restrict__ dec_b, int32_t *__restrict__ argb_out, Geom g,
               unsigned long long *st, int max_iters, float carry, float fwh, unsigned long long skip_from)
{
    uint32_t *w = (uint32_t *)st;
    uint32_t epoch = 0;
    for (int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x; j < g.NR; j += (int64_t)gridDim.x * 256)
        dequant_one(j, q, nullptr, code, dpos, g, 0, st, 1);
    grid_barrier(w + ST_BARRIER, epoch);
    uint8_t *din = dec_a, *dout = dec_b;
    bool ok = false;
    for (int it = 0; it < max_iters; it++) {
        unsigned long long local = it == 0 ? sweep_il_body<C, B, false, true, false>(din, img, dout, code, dpos, g, nullptr)
                                           : sweep_il_body<C, B, false, false, false>(din, img, dout, code, dpos, g, nullptr);
        const unsigned long long tot = cta_sum(local);
        if (threadIdx.x == 0 && tot) atomicAdd(st, tot);
        grid_barrier(w + ST_BARRIER, epoch);
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            const unsigned long long S = atomicExch(st, 0ull);
            const bool last = it == max_iters - 1;
            const float c0 = it == 0 ? carry : 0.0f;
            if (c0 == 0.0f && S < (1ull << 24)) {  // the float sum is the exact integer
                record_sweep(w, it, (float)S, fwh, last);
            } else if (!last && c0 >= 0.0f && S >= skip_from) {  // certainly not converged; the value is discarded
                w[ST_ITERS] = (uint32_t)(it + 1);
                w[ST_AVG] = 0u;
            } else {
                w[ST_BAIL] = 1u;
            }
            __threadfence();
        }
        grid_barrier(w + ST_BARRIER, epoch);
        const uint32_t done = ((volatile uint32_t *)w)[ST_DONE], bail = ((volatile uint32_t *)w)[ST_BAIL];
        if (bail) return;
        if (done || it == max_iters - 1) { ok = true; break; }
        uint8_t *t = din; din = dout; dout = t;
    }
    if (ok && argb_out) pack_argb<C>((const uchar4 *)img, (int4 *)argb_out, (int64_t)g.W * g.H / 4);
}

// The sweeps are grid-stride over exactly one wave of resident CTAs (SMs x occupancy of the kernel): a second, partly
// filled wave cost a third of the sweep at 4096^2 (1184 CTAs on 740 slots, profiles/README.md).
template <class K>
static int64_t sweep_wave_ctas(K kernel)
{
    int dev = 0, sms = 148, per_sm = 4;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, 0) != cudaSuccess || per_sm < 1) per_sm = 4;
    return (int64_t)sms * per_sm;
}

// skip_from: exact totals from which a sweep over `count` pixels certainly did not converge (only its value < W*H would
// be kept, FC:413-417).  Every float add loses at most half an ulp, and below W*H an ulp is at most ulp(W*H): with
// S >= W*H + count * ulp / 2 the float sum cannot end below W*H.  (~0 when no total qualifies.)
static unsigned long long skip_from_of(float fwh, int64_t count)
{
    if (fwh < 1.0f) return ~0ull;
    int ex = 0;
    frexpf(fwh, &ex);  // fwh = m * 2^ex, 0.5 <= m < 1: ulp(fwh) = 2^(ex - 24)
    return (unsigned long long)((double)fwh + (double)count * ldexp(1.0, ex - 25)) + 2ull;
}

// Small images: the whole decode in one cooperative launch (k_decode_small).  Returns 1 if the kernel was launched (the
// state block then tells whether it finished or bailed), 0 if this geometry / device does not take the fused path.
// The state block must be zero.
template <int C, int B>
static int launch_small_t(const int32_t *d_q, float *d_code, int32_t *d_pos, uint8_t *d_img, uint8_t *d_dec_a, uint8_t *d_dec_b,
                          int32_t *d_argb, const Geom &g, unsigned long long *d_state, int max_iters, float carry, float fwh,
                          unsigned long long skip_from, cudaStream_t s)
{
    static int coop = -1, per_sm = 0, sms = 0;
    if (coop < 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_decode_small<C, B>, 256, 0) != cudaSuccess) per_sm = 0;
        cudaGetLastError();
    }
    if (coop <= 0 || per_sm < 1) return 0;
    const int64_t tiles = (int64_t)((g.W / 8 + 15) / 16) * (g.H / 4);
    int64_t grid = (tiles + 7) / 8;
    if (grid > (int64_t)sms * per_sm) grid = (int64_t)sms * per_sm;
    Geom gg = g;
    void *args[] = {(void *)&d_q, (void *)&d_code, (void *)&d_pos, (void *)&d_img, (void *)&d_dec_a, (void *)&d_dec_b, (void *)&d_argb,
                    (void *)&gg, (void *)&d_state, (void *)&max_iters, (void *)&carry, (void *)&fwh, (void *)&skip_from};
    if (cudaLaunchCooperativeKernel((const void *)k_decode_small<C, B>, dim3((unsigned)grid), dim3(256), args, 0, s) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return 1;
}

int launch_decode_small(const int32_t *d_q, float *d_code, int32_t *d_pos, uint8_t *d_img, uint8_t *d_dec_a, uint8_t *d_dec_b,
                        int32_t *d_argb, const Geom &g, unsigned long long *d_state, int max_iters, float carry, float fwh,
                        cudaStream_t s)
{
    if (!sweep_interleaved(g) || (int64_t)g.W * g.H > ((int64_t)1 << 20)) return 0;
    const unsigned long long skip_from = skip_from_of(fwh, (int64_t)g.W * g.H);
    if (g.B == 8)
        return g.C == 1 ? launch_small_t<1, 8>(d_q, d_code, d_pos, d_img, d_dec_a, d_dec_b, d_argb, g, d_state, max_iters, carry, fwh, skip_from, s)
                        : launch_small_t<3, 8>(d_q, d_code, d_pos, d_img, d_dec_a, d_dec_b, d_argb, g, d_state, max_iters, carry, fwh, skip_from, s);
    return g.C == 1 ? launch_small_t<1, 16>(d_q, d_code, d_pos, d_img, d_dec_a, d_dec_b, d_argb, g, d_state, max_iters, carry, fwh, skip_from, s)
                    : launch_small_t<3, 16>(d_q, d_code, d_pos, d_img, d_dec_a, d_dec_b, d_argb, g, d_state, max_iters, carry, fwh, skip_from, s);
}

bool decode_sweep_has_first(const Geom &g) { return g.W % 8 == 0 && g.n_iso == 1 && g.B >= 8; }
bool decode_sweep_interleaved(const Geom &g) { return sweep_interleaved(g); }

template <int C, int B>
static void launch_sweep_il(const uint8_t *d_dec_in, uint8_t *d_img, uint8_t *d_dec_out, const float *d_code, const int32_t *d_pos,
                            const Geom &g, const SweepCtl &ctl, int32_t *d_perr, int first, cudaStream_t s)
{
    static const int64_t wave[4] = {sweep_wave_ctas(k_decode_sweep_il<C, B, false, false>), sweep_wave_ctas(k_decode_sweep_il<C, B, false, true>),
                                    sweep_wave_ctas(k_decode_sweep_il<C, B, true, false>), sweep_wave_ctas(k_decode_sweep_il<C, B, true, true>)};
    const int64_t tiles = (int64_t)((g.W / 8 + 15) / 16) * (g.H / 4), need = (tiles + 7) / 8;  // one warp per 16 x 2 strips
    const int v = (d_perr ? 2 : 0) + (first ? 1 : 0);
    const unsigned grid = (unsigned)(need < wave[v] ? need : wave[v]);
    switch (v) {
    case 0: k_decode_sweep_il<C, B, false, false><<<grid, 256, 0, s>>>(d_dec_in, d_img, d_dec_out, d_code, d_pos, g, ctl, d_perr); break;
    case 1: k_decode_sweep_il<C, B, false, true><<<grid, 256, 0, s>>>(d_dec_in, d_img, d_dec_out, d_code, d_pos, g, ctl, d_perr); break;
    case 2: k_decode_sweep_il<C, B, true, false><<<grid, 256, 0, s>>>(d_dec_in, d_img, d_dec_out, d_code, d_pos, g, ctl, d_perr); break;
    default: k_decode_sweep_il<C, B, true, true><<<grid, 256, 0, s>>>(d_dec_in, d_img, d_dec_out, d_code, d_pos, g, ctl, d_perr); break;
    }
}

// first != 0 (only where decode_sweep_has_first): the sweep starts from the constant-128 image and reads neither
// d_img nor d_dec_in.
// interleaved != 0 (only where decode_sweep_interleaved): the decimated planes are row-pair interleaved and d_off holds
// packed positions (launch_dequant with packed = 1).
int launch_decode_sweep(const uint8_t *d_dec_in, uint8_t *d_img, uint8_t *d_dec_out, const float *d_code,
                        const int32_t *d_off, const Geom &g, const SweepCtl &ctl, int32_t *d_perr, int first, int interleaved,
                        cudaStream_t s)
{
    if (interleaved && sweep_interleaved(g)) {
        if (g.B == 8) {
            if (g.C == 1) launch_sweep_il<1, 8>(d_dec_in, d_img, d_dec_out, d_code, d_off, g, ctl, d_perr, first, s);
            else launch_sweep_il<3, 8>(d_dec_in, d_img, d_dec_out, d_code, d_off, g, ctl, d_perr, first, s);
        } else {
            if (g.C == 1) launch_sweep_il<1, 16>(d_dec_in, d_img, d_dec_out, d_code, d_off, g, ctl, d_perr, first, s);
            else launch_sweep_il<3, 16>(d_dec_in, d_img, d_dec_out, d_code, d_off, g, ctl, d_perr, first, s);
        }
        return 1;
    }
    if (first && decode_sweep_has_first(g)) {
        static const int64_t wave_f_1 = sweep_wave_ctas(k_decode_sweep_v8<1, true>), wave_f_3 = sweep_wave_ctas(k_decode_sweep_v8<3, true>);
        const int64_t strips = (int64_t)(g.W / 8) * (g.H / 2), need = (strips + 255) / 256;
        if (g.C == 1)
            k_decode_sweep_v8<1, true><<<(unsigned)(need < wave_f_1 ? need : wave_f_1), 256, 0, s>>>(d_dec_in, d_img, d_dec_out, d_code, d_off, g, ctl, d_perr);
        else
            k_decode_sweep_v8<3, true><<<(unsigned)(need < wave_f_3 ? need : wave_f_3), 256, 0, s>>>(d_dec_in, d_img, d_dec_out, d_code, d_off, g, ctl, d_perr);
        return 1;
    }
    static const int64_t wave_v8_1 = sweep_wave_ctas(k_decode_sweep_v8<1>), wave_v8_3 = sweep_wave_ctas(k_decode_sweep_v8<3>);
    static const int64_t wave_q_1 = sweep_wave_ctas(k_decode_sweep<1>), wave_q_3 = sweep_wave_ctas(k_decode_sweep<3>);
    if (g.W % 8 == 0 && g.n_iso == 1) {  // the isometry extension uses the quad kernel (per-pixel gather)
        const int64_t strips = (int64_t)(g.W / 8) * (g.H / 2), need = (strips + 255) / 256;
        if (g.C == 1)
            k_decode_sweep_v8<1><<<(unsigned)(need < wave_v8_1 ? need : wave_v8_1), 256, 0, s>>>(d_dec_in, d_img, d_dec_out, d_code, d_off, g, ctl, d_perr);
        else
            k_decode_sweep_v8<3><<<(unsigned)(need < wave_v8_3 ? need : wave_v8_3), 256, 0, s>>>(d_dec_in, d_img, d_dec_out, d_code, d_off, g, ctl, d_perr);
        return 1;
    }
    const int64_t quads = (int64_t)(g.W / 2) * (g.H / 2), need = (quads + 255) / 256;
    if (g.C == 1)
        k_decode_sweep<1><<<(unsigned)(need < wave_q_1 ? need : wave_q_1), 256, 0, s>>>(d_dec_in, d_img, d_dec_out, d_code, d_off, g, ctl, d_perr);
    else
        k_decode_sweep<3><<<(unsigned)(need < wave_q_3 ? need : wave_q_3), 256, 0, s>>>(d_dec_in, d_img, d_dec_out, d_code, d_off, g, ctl, d_perr);
    return 1;
}

// Folds a sweep that may need the reference's float accumulation replayed (FC:407 / FC:493): the first sweep when
// the never-reset static avgError (FC:20) carries a value in, the last allowed sweep (its value is kept whatever it is,
// FC:416), and every sweep of an image above 2^24 pixels (where the sum may pass 2^24 and still converge).
// One warp.  The running binary32 sum is order dependent once it passes 2^24, so it is replayed in loop order over
// the per-pixel squared changes -- with three shortcuts, none of which changes a bit of the result:
//   * while the sum is an integer below 2^24 every add is exact, so a whole 128-element group is added at once; if the
//     sweep's exact total S is below 2^24 (and nothing is carried in) the sum is S and nothing is replayed;
//   * a group of zeros is skipped, and inside a group only lanes that hold a non-zero term are visited (x + 0 == x);
//   * the sum never decreases (the terms are >= 0): on a sweep whose value is discarded unless it converged
//     (FC:413-417) the replay stops once the sum reaches W*H.
__global__ void k_sweep_finish(const int32_t *__restrict__ perr, int64_t count, unsigned long long *st, int it, int last,
                               float carry, float fwh)
{
    if (blockIdx.x || threadIdx.x >= 32) return;
    uint32_t *w = (uint32_t *)st;
    if (((volatile uint32_t *)w)[ST_DONE]) return;
    const int lane = threadIdx.x;
    const unsigned long long S = *(volatile unsigned long long *)st;
    float a = carry;  // FC:20: the first sweep starts from whatever the previous decode left; later ones from 0
    if (!(a == 0.0f && S < (1ull << 24))) {
        const float limit = last ? __int_as_float(0x7f800000) : fwh;
        for (int64_t base = 0; base < count && a < limit; base += 128) {
            const int64_t i = base + 4 * lane;
            int4 v = make_int4(0, 0, 0, 0);
            if (i + 4 <= count) v = *(const int4 *)(perr + i);
            else
                for (int k = 0; k < 4; k++)
                    if (i + k < count) (&v.x)[k] = perr[i + k];
            const int s = v.x + v.y + v.z + v.w;  // <= 4 * 3 * 255^2
            int tot = s;
            for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
            if (tot == 0) continue;
            if (a == floorf(a) && __fadd_rn(a, (float)tot) <= 16777216.0f) {  // every partial sum is an exact integer
                a = __fadd_rn(a, (float)tot);
                continue;
            }
            unsigned m = __ballot_sync(0xffffffffu, s != 0);
            while (m) {
                const int l = __ffs(m) - 1;
                m &= m - 1;
                a = __fadd_rn(a, (float)__shfl_sync(0xffffffffu, v.x, l));
                a = __fadd_rn(a, (float)__shfl_sync(0xffffffffu, v.y, l));
                a = __fadd_rn(a, (float)__shfl_sync(0xffffffffu, v.z, l));
                a = __fadd_rn(a, (float)__shfl_sync(0xffffffffu, v.w, l));
            }
        }
    } else {
        a = (float)S;
    }
    if (lane == 0) {
        *st = 0ull;
        record_sweep(w, it, a, fwh, last);
    }
}

// ---- chunked replay (large images) -------------------------------------------------------------------------------
// The literal replay above is one dependent float add per pixel: 0.2 s per sweep at 8192^2, where EVERY sweep passes
// 2^24.  Above 2^24 the running sum a = A * u (u = ulp = 2^(k-23), 2^23 <= A < 2^24) stays a multiple of u, and
// adding an integer e = m * u + r rounds to A + m + c with c = [r > u/2], or, on a tie r == u/2, the parity of A + m
// (round to nearest even).  So while the sum stays inside one binade a run of pixels acts on A only through its
// parity: the run is a two-state transducer (delta[0], delta[1]) = what it adds to A for an even / odd A on entry, and
// transducers compose (associatively).  Per chunk of 4096 pixels: k_replay_sums takes the exact integer sum,
// k_replay_scan guesses the chunk's binade from the exact prefix, k_replay_transducers composes the chunk's
// transducers for that binade and the one below (the float sum falls behind the exact one -- on a grid of 2 an added 1
// is a tie that an even mantissa drops -- but rarely by more than a binade), all in parallel; one
// warp (k_replay_walk) then walks the chunks with the true float sum: exact integer adds below 2^24, the transducer
// where the guess holds and the chunk provably stays inside the binade, and the literal loop for the few chunks
// around a binade crossing; 32 chunks at a time through their composed transducer (k_replay_groups) where that holds
// for all of them.  Bit-identical to the sequential float sum.
constexpr int kRepChunk = 4096;                 // pixels per chunk = 256 threads x 16
struct ReplayChunk { uint32_t sum; int32_t k; uint32_t d0, d1, e0, e1; };  // exact sum, guessed binade (0: none), transducers for binades k and k - 1

// skip_from: see skip_from_of.
__device__ __forceinline__ bool replay_not_needed(const unsigned long long *st, float carry, unsigned long long skip_from)
{
    // done already; or the sweep's exact total is below 2^24 and nothing is carried in: the float sum is that integer
    const unsigned long long S = *(volatile const unsigned long long *)st;
    return ((volatile const uint32_t *)st)[ST_DONE] != 0 || (carry == 0.0f && S < (1ull << 24)) || S >= skip_from;
}

__device__ __forceinline__ void replay_load16(const int32_t *__restrict__ perr, int64_t count, int64_t i0, int (&v)[16])
{
    if (i0 + 16 <= count) {
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int4 t = __ldg((const int4 *)(perr + i0) + q);
            v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w;
        }
    } else {
#pragma unroll
        for (int q = 0; q < 16; q++) v[q] = i0 + q < count ? perr[i0 + q] : 0;
    }
}

__global__ void __launch_bounds__(256) k_replay_sums(const int32_t *__restrict__ perr, int64_t count, ReplayChunk *__restrict__ ch,
                                                     const unsigned long long *st, float carry, unsigned long long skip_from)
{
    if (replay_not_needed(st, carry, skip_from)) return;
    __shared__ uint32_t s_part[8];
    int v[16];
    replay_load16(perr, count, (int64_t)blockIdx.x * kRepChunk + 16 * threadIdx.x, v);
    uint32_t t = 0;
#pragma unroll
    for (int q = 0; q < 16; q++) t += (uint32_t)v[q];   // <= 4096 * 3 * 255^2 < 2^32 per chunk
    for (int o = 16; o > 0; o >>= 1) t += __shfl_down_sync(0xffffffffu, t, o);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t tot = 0;
        for (int w = 0; w < 8; w++) tot += s_part[w];
        ch[blockIdx.x].sum = tot;
    }
}

// One CTA: exact prefix sums of the chunk totals -> the binade each chunk's running sum is expected to start in.
__global__ void __launch_bounds__(1024) k_replay_scan(ReplayChunk *__restrict__ ch, int nchunks, const unsigned long long *st, float carry,
                                                      unsigned long long skip_from)
{
    if (replay_not_needed(st, carry, skip_from)) return;
    __shared__ unsigned long long s_tot[1024];
    const int per = (nchunks + 1023) / 1024, c0 = threadIdx.x * per, c1 = min(nchunks, c0 + per);
    unsigned long long t = 0;
    for (int c = c0; c < c1; c++) t += ch[c].sum;
    s_tot[threadIdx.x] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long run = 0;
        for (int i = 0; i < 1024; i++) { const unsigned long long x = s_tot[i]; s_tot[i] = run; run += x; }
    }
    __syncthreads();
    unsigned long long pre = s_tot[threadIdx.x];
    for (int c = c0; c < c1; c++) {
        const double g = (double)carry + (double)pre;
        ch[c].k = g >= 16777216.0 ? ilogb(g) : 0;
        pre += ch[c].sum;
    }
}

// ordered composition: first `l`, then `r`
__device__ __forceinline__ uint2 replay_compose(uint2 l, uint2 r)
{
    return make_uint2(l.x + (((l.x) & 1u) ? r.y : r.x), l.y + (((1u + l.y) & 1u) ? r.y : r.x));
}

__global__ void __launch_bounds__(256) k_replay_transducers(const int32_t *__restrict__ perr, int64_t count, ReplayChunk *__restrict__ ch,
                                                            const unsigned long long *st, float carry, unsigned long long skip_from)
{
    if (replay_not_needed(st, carry, skip_from)) return;
    const int k = ch[blockIdx.x].k;
    if (k == 0) return;
    __shared__ uint4 s_part[8];
    int v[16];
    replay_load16(perr, count, (int64_t)blockIdx.x * kRepChunk + 16 * threadIdx.x, v);
    // binade k: u = 2^sh; binade k - 1 (only if it is still >= 24): u = 2^(sh - 1)
    const int sh = k - 23, shl = sh > 1 ? sh - 1 : 1;
    uint32_t d[4] = {0u, 0u, 0u, 0u}, par[4] = {0u, 1u, 0u, 1u};
#pragma unroll
    for (int q = 0; q < 16; q++) {
        const uint32_t e = (uint32_t)v[q];
#pragma unroll
        for (int b = 0; b < 2; b++) {
            const int s2 = b ? shl : sh;
            const uint32_t m = e >> s2, r = e & ((1u << s2) - 1u), h = 1u << (s2 - 1);
#pragma unroll
            for (int p = 0; p < 2; p++) {
                const uint32_t t = par[2 * b + p] ^ (m & 1u);              // parity of A + m
                const uint32_t c = r > h ? 1u : (r == h ? t : 0u);         // round to nearest, ties to even
                d[2 * b + p] += m + c;
                par[2 * b + p] = t ^ c;
            }
        }
    }
    uint4 T = make_uint4(d[0], d[1], d[2], d[3]);
    auto compose4 = [](uint4 l, uint4 r) {
        const uint2 hi = replay_compose(make_uint2(l.x, l.y), make_uint2(r.x, r.y));
        const uint2 lo = replay_compose(make_uint2(l.z, l.w), make_uint2(r.z, r.w));
        return make_uint4(hi.x, hi.y, lo.x, lo.y);
    };
    const int lane = threadIdx.x & 31;
    for (int o = 1; o < 32; o <<= 1) {
        uint4 other;
        other.x = __shfl_down_sync(0xffffffffu, T.x, o);
        other.y = __shfl_down_sync(0xffffffffu, T.y, o);
        other.z = __shfl_down_sync(0xffffffffu, T.z, o);
        other.w = __shfl_down_sync(0xffffffffu, T.w, o);
        if ((lane & (2 * o - 1)) == 0) T = compose4(T, other);
    }
    if (lane == 0) s_part[threadIdx.x >> 5] = T;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint4 tot = s_part[0];
        for (int w = 1; w < 8; w++) tot = compose4(tot, s_part[w]);
        ch[blockIdx.x].d0 = tot.x;
        ch[blockIdx.x].d1 = tot.y;
        ch[blockIdx.x].e0 = tot.z;
        ch[blockIdx.x].e1 = tot.w;
    }
}

// The literal float accumulation over perr[begin, end) (one warp; every lane returns the same sum).
__device__ float replay_literal(const int32_t *__restrict__ perr, int64_t begin, int64_t end, float a, float limit)
{
    const int lane = threadIdx.x & 31;
    for (int64_t base = begin; base < end && a < limit; base += 128) {
        const int64_t i = base + 4 * lane;
        int4 v = make_int4(0, 0, 0, 0);
        if (i + 4 <= end) v = *(const int4 *)(perr + i);
        else
            for (int k = 0; k < 4; k++)
                if (i + k < end) (&v.x)[k] = perr[i + k];
        unsigned m = __ballot_sync(0xffffffffu, (v.x | v.y | v.z | v.w) != 0);
        while (m) {
            const int l = __ffs(m) - 1;
            m &= m - 1;
            a = __fadd_rn(a, (float)__shfl_sync(0xffffffffu, v.x, l));
            a = __fadd_rn(a, (float)__shfl_sync(0xffffffffu, v.y, l));
            a = __fadd_rn(a, (float)__shfl_sync(0xffffffffu, v.z, l));
            a = __fadd_rn(a, (float)__shfl_sync(0xffffffffu, v.w, l));
        }
    }
    return a;
}

// A group of 32 chunks composed into one record (valid when its non-empty chunks share one binade guess), so that the
// walker steps over 131 072 pixels at a time wherever the sum is far from a binade crossing.
struct ReplayGroup { unsigned long long sum; int32_t k; uint32_t d0, d1, e0, e1; };
constexpr int kRepGroup = 32;

__global__ void k_replay_groups(const ReplayChunk *__restrict__ ch, int nchunks, ReplayGroup *__restrict__ gr, int ngroups,
                                const unsigned long long *st, float carry, unsigned long long skip_from)
{
    if (replay_not_needed(st, carry, skip_from)) return;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= ngroups) return;
    unsigned long long sum = 0, d[2] = {0, 0}, e[2] = {0, 0};
    int k = -1;  // -1: no non-empty chunk yet; 0: no common transducer
    for (int c = g * kRepGroup; c < min(nchunks, (g + 1) * kRepGroup); c++) {
        const ReplayChunk x = ch[c];
        if (x.sum == 0u) continue;  // identity
        sum += x.sum;
        if (k == -1) k = x.k;
        if (x.k == 0 || x.k != k) k = 0;
        if (k == 0) continue;
        // ordered composition (replay_compose) in 64 bits: a total of 2^24 or more can never be applied
        const unsigned long long d0 = d[0] + ((d[0] & 1ull) ? x.d1 : x.d0), d1 = d[1] + (((1ull + d[1]) & 1ull) ? x.d1 : x.d0);
        const unsigned long long e0 = e[0] + ((e[0] & 1ull) ? x.e1 : x.e0), e1 = e[1] + (((1ull + e[1]) & 1ull) ? x.e1 : x.e0);
        d[0] = d0; d[1] = d1; e[0] = e0; e[1] = e1;
    }
    ReplayGroup out;
    out.sum = sum;
    const bool fits = (d[0] | d[1] | e[0] | e[1]) < (1ull << 24);
    out.k = (k > 0 && fits) ? k : 0;
    out.d0 = (uint32_t)d[0]; out.d1 = (uint32_t)d[1]; out.e0 = (uint32_t)e[0]; out.e1 = (uint32_t)e[1];
    gr[g] = out;
}

__global__ void k_replay_walk(const int32_t *__restrict__ perr, int64_t count, const ReplayChunk *__restrict__ ch, int nchunks,
                              const ReplayGroup *__restrict__ gr, int ngroups, unsigned long long *st, int it, int last, float carry,
                              float fwh, unsigned long long skip_from)
{
    if (blockIdx.x || threadIdx.x >= 32) return;
    uint32_t *w = (uint32_t *)st;
    if (((volatile uint32_t *)w)[ST_DONE]) return;
    const int lane = threadIdx.x;
    const unsigned long long S = *(volatile unsigned long long *)st;
    float a = carry;  // FC:20
    // One step over `px` pixels with exact total `sum` (> 0), binade guess kk and transducers d (binade kk) / e (kk - 1),
    // identical in all lanes.  True if the step could be taken without looking at the pixels.
    auto step = [&](unsigned long long sum, int kk, uint32_t d0, uint32_t d1, uint32_t e0, uint32_t e1, unsigned long long px) -> bool {
        const uint32_t bits = __float_as_uint(a);
        const int k = (int)(bits >> 23) - 127;
        if (k < 24) {
            // below 2^24: while the sum is an integer and stays <= 2^24 every add is exact
            if (a == floorf(a) && a >= 0.0f && (unsigned long long)a + sum <= (1ull << 24)) {
                a = (float)((uint32_t)a + (uint32_t)sum);
                return true;
            }
            return false;
        }
        const int below = kk - k;
        if (k >= 62 || kk == 0 || (below != 0 && below != 1)) return false;
        // a = A * 2^(k-23).  If even the largest sum the span can reach (its exact total plus half an ulp per add)
        // stays inside the binade, every add rounds on this grid: apply the span's transducer to A.
        const uint32_t A = (bits & 0x7fffffu) | 0x800000u;
        const unsigned long long ai = (unsigned long long)A << (k - 23);
        if (ai + sum + (px << (k - 24)) >= (2ull << k)) return false;
        const uint32_t d = (A & 1u) ? (below ? e1 : d1) : (below ? e0 : d0);
        a = __uint_as_float((bits & 0xff800000u) | ((A + d) & 0x7fffffu));   // A + d < 2^24
        return true;
    };
    if (carry == 0.0f && S < (1ull << 24)) {
        a = (float)S;
    } else if (S >= skip_from) {
        a = __fmul_rn(fwh, 2.0f);  // certainly not converged (see replay_not_needed); the value is discarded
    } else {
        const float limit = last ? __int_as_float(0x7f800000) : fwh;  // FC:416-417: an unconverged value is only kept on the last sweep
        for (int gb = 0; gb < ngroups && a < limit; gb += 32) {
            ReplayGroup mine = {0ull, 0, 0u, 0u, 0u, 0u};
            if (gb + lane < ngroups) mine = gr[gb + lane];
            for (int j = 0; j < 32 && gb + j < ngroups && a < limit; j++) {
                const unsigned long long gsum = __shfl_sync(0xffffffffu, mine.sum, j);
                if (gsum == 0ull) continue;  // x + 0 == x
                if (step(gsum, __shfl_sync(0xffffffffu, mine.k, j), __shfl_sync(0xffffffffu, mine.d0, j), __shfl_sync(0xffffffffu, mine.d1, j),
                         __shfl_sync(0xffffffffu, mine.e0, j), __shfl_sync(0xffffffffu, mine.e1, j), (unsigned long long)kRepGroup * kRepChunk))
                    continue;
                // chunk by chunk; a chunk that cannot be stepped over either is replayed literally
                const int c0 = (gb + j) * kRepGroup;
                ReplayChunk cm = {0u, 0, 0u, 0u, 0u, 0u};
                if (c0 + lane < nchunks) cm = ch[c0 + lane];
                for (int i = 0; i < kRepGroup && c0 + i < nchunks && a < limit; i++) {
                    const uint32_t csum = __shfl_sync(0xffffffffu, cm.sum, i);
                    if (csum == 0u) continue;
                    if (step(csum, __shfl_sync(0xffffffffu, cm.k, i), __shfl_sync(0xffffffffu, cm.d0, i), __shfl_sync(0xffffffffu, cm.d1, i),
                             __shfl_sync(0xffffffffu, cm.e0, i), __shfl_sync(0xffffffffu, cm.e1, i), (unsigned long long)kRepChunk))
                        continue;
                    const int64_t b0 = (int64_t)(c0 + i) * kRepChunk, b1 = b0 + kRepChunk < count ? b0 + kRepChunk : count;
                    a = replay_literal(perr, b0, b1, a, __int_as_float(0x7f800000));
                }
            }
        }
    }
    if (lane == 0) {
        *st = 0ull;
        record_sweep(w, it, a, fwh, last);
    }
}

static int64_t replay_chunks(int64_t count) { return (count + kRepChunk - 1) / kRepChunk; }
static int64_t replay_groups(int64_t count) { return (replay_chunks(count) + kRepGroup - 1) / kRepGroup; }

size_t sweep_finish_workspace(int64_t count)
{
    if (count < ((int64_t)1 << 22)) return 0;
    return sizeof(ReplayGroup) * (size_t)replay_groups(count) + sizeof(ReplayChunk) * (size_t)replay_chunks(count);
}

int launch_sweep_finish(const int32_t *d_perr, int64_t count, unsigned long long *d_state, int it, int last, float carry,
                        float fwh, void *d_workspace, cudaStream_t s)
{
    if (d_workspace && sweep_finish_workspace(count)) {
        const int nchunks = (int)replay_chunks(count), ngroups = (int)replay_groups(count);
        ReplayGroup *gr = (ReplayGroup *)d_workspace;
        ReplayChunk *ch = (ReplayChunk *)(gr + ngroups);
        // the last allowed sweep keeps its value whatever it is
        const unsigned long long skip_from = !last && carry >= 0.0f ? skip_from_of(fwh, count) : ~0ull;
        k_replay_sums<<<nchunks, 256, 0, s>>>(d_perr, count, ch, d_state, carry, skip_from);
        k_replay_scan<<<1, 1024, 0, s>>>(ch, nchunks, d_state, carry, skip_from);
        k_replay_transducers<<<nchunks, 256, 0, s>>>(d_perr, count, ch, d_state, carry, skip_from);
        k_replay_groups<<<(ngroups + 127) / 128, 128, 0, s>>>(ch, nchunks, gr, ngroups, d_state, carry, skip_from);
        k_replay_walk<<<1, 32, 0, s>>>(d_perr, count, ch, nchunks, gr, ngroups, d_state, it, last, carry, fwh, skip_from);
        return 5;
    }
    k_sweep_finish<<<1, 32, 0, s>>>(d_perr, count, d_state, it, last, carry, fwh);
    return 1;
}

}  // namespace fic
