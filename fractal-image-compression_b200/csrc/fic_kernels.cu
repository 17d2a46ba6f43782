// fic_kernels.cu -- HBM-bound encoder kernels of libfic_b200 (sm_100a):
//   K1  pool builder: ARGB unpack, 2x decimation, per-domain / per-range integer sums
//   K2w direct windowed search (grey + RGB), the reference's default widthKernel path
//   K2f fused one-launch windowed encode
//   K3s code solve + quantisation (shared by the direct and the tcgen05 search)
// The decoder (K4) is fic_decode.cu.
//
// file:line citations refer to the reference, src/bvk_ss19/FractalCompression.java (FC)
// and src/bvk_ss19/Domainblock.java (DB).
#include "fic_device.cuh"

namespace fic {

// ------------------------------------------------------------------------------------
// K1a: ARGB int32 -> 8-bit planes.  Grey keeps the red channel only (FC:596, FC:977).
// 16-byte loads, 4-byte stores per plane.
// ------------------------------------------------------------------------------------
// Several images: quads runs over all of them; image i's planes start 3 * plane_quads quads after image i - 1's (grey:
// the one plane of each image directly follows the previous one, so the flat index needs no image).
template <int C>
__global__ void k_unpack(const int4 *__restrict__ argb, uchar4 *__restrict__ planes, int64_t quads,
                         int64_t plane_quads)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < quads; i += stride) {
        int4 p = __ldg(argb + i);
        if (C == 1) {
            planes[i] = make_uchar4((p.x >> 16) & 0xff, (p.y >> 16) & 0xff, (p.z >> 16) & 0xff, (p.w >> 16) & 0xff);
        } else {
            const int64_t image = i >= plane_quads ? i / plane_quads : 0, o = i + 2 * image * plane_quads;  // quad of image's R plane
            planes[o] = make_uchar4((p.x >> 16) & 0xff, (p.y >> 16) & 0xff, (p.z >> 16) & 0xff, (p.w >> 16) & 0xff);
            planes[plane_quads + o] =
                make_uchar4((p.x >> 8) & 0xff, (p.y >> 8) & 0xff, (p.z >> 8) & 0xff, (p.w >> 8) & 0xff);
            planes[2 * plane_quads + o] = make_uchar4(p.x & 0xff, p.y & 0xff, p.z & 0xff, p.w & 0xff);
        }
    }
}

int launch_unpack(const int32_t *d_argb, uint8_t *d_planes, int W, int H, int C, cudaStream_t s, int n_images)
{
    int64_t quads = (int64_t)W * H / 4 * n_images;  // W % 4 == 0 is guaranteed by make_geom
    int blocks = (int)((quads + 255) / 256 < 148 * 16 ? (quads + 255) / 256 : 148 * 16);
    if (blocks < 1) blocks = 1;
    if (C == 1)
        k_unpack<1><<<blocks, 256, 0, s>>>((const int4 *)d_argb, (uchar4 *)d_planes, quads, quads);
    else
        k_unpack<3><<<blocks, 256, 0, s>>>((const int4 *)d_argb, (uchar4 *)d_planes, quads, quads / n_images);
    return 1;
}

// ------------------------------------------------------------------------------------
// K1b: 2x decimation (FC:970-1007 grey, FC:901-962 RGB).
//   grey: (p00 + p10 + p01 + p11) / 4;  RGB: (p00 + p10 + 2*p01) / 4 (FC:945 re-reads
//   (x, y+1)).  With W, H even the only live border branch is the reference's
//   `x + 1 >= image.height` test (FC:993, FC:940), which substitutes 128 for the fourth
//   tap on landscape images; it is reproduced here.
// One thread makes 2 output pixels from two 4-byte loads; stores are 2 bytes.  `planes` = C * images: the planes of a
// group of images follow each other in source and output alike.
// ------------------------------------------------------------------------------------
__global__ void k_decimate(const uint8_t *__restrict__ src, uint8_t *__restrict__ dec, int W, int H, int planes, bool rgb)
{
    int sw = W / 2, sh = H / 2;
    int64_t pairs_per_plane = (int64_t)(sw / 2) * sh;
    int64_t total = pairs_per_plane * planes;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
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
__global__ void k_decimate_v8(const uint8_t *__restrict__ src, uint8_t *__restrict__ dec, int W, int H, int planes, bool rgb)
{
    const int sw = W / 2, sh = H / 2;
    const int64_t oct_per_plane = (int64_t)(sw / 8) * sh;
    const int64_t total = oct_per_plane * planes;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
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

int launch_decimate(const uint8_t *d_src, uint8_t *d_dec, const Geom &g, cudaStream_t s, int n_images)
{
    const int planes = g.C * n_images;
    if (g.W % 16 == 0) {
        int64_t total = (int64_t)(g.sw / 8) * g.sh * planes;
        int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
        if (blocks < 1) blocks = 1;
        k_decimate_v8<<<blocks, 256, 0, s>>>(d_src, d_dec, g.W, g.H, planes, g.C == 3);
        return 1;
    }
    int64_t total = (int64_t)(g.sw / 2) * g.sh * planes;
    int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
    if (blocks < 1) blocks = 1;
    k_decimate<<<blocks, 256, 0, s>>>(d_src, d_dec, g.W, g.H, planes, g.C == 3);
    return 1;
}

// ------------------------------------------------------------------------------------
// K1c: per-domain integer sums (DB:92-115).  Domain j = (gy, gx) covers the BxB block
// of the decimated plane at (gx*step, gy*step) (FC:1027-1047).  sum d and sum d^2 are
// exact in s32; mean and variance follow from them (dom_var()).
// ------------------------------------------------------------------------------------
__global__ void k_domain_stats(const uint8_t *__restrict__ dec, int32_t *__restrict__ dsum,
                               int32_t *__restrict__ dsq, Geom g, int planes)  // planes = C * images
{
    int64_t total = g.ND * planes;
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

int launch_domain_stats(const uint8_t *d_dec, int32_t *d_dsum, int32_t *d_dsq, const Geom &g, cudaStream_t s, int n_images)
{
    int64_t total = g.ND * g.C * n_images;
    k_domain_stats<<<(unsigned)((total + 127) / 128), 128, 0, s>>>(d_dec, d_dsum, d_dsq, g, g.C * n_images);
    return 1;
}

// K1d: per-range pixel sums (FC:67-73 getMittelwert of FC:588-602 getRangeblock).
__global__ void k_range_stats(const uint8_t *__restrict__ src, int32_t *__restrict__ rsum, Geom g, int planes)  // C * images
{
    int64_t total = g.NR * planes;
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

int launch_range_stats(const uint8_t *d_src, int32_t *d_rsum, const Geom &g, cudaStream_t s, int n_images)
{
    int64_t total = g.NR * g.C * n_images;
    k_range_stats<<<(unsigned)((total + 127) / 128), 128, 0, s>>>(d_src, d_rsum, g, g.C * n_images);
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

// RGB: dec3 = R + G + B of the decimated planes (what k_search_direct_rgb reads instead of three planes); `total`
// pixels of images of `count` pixels each.
__global__ void k_sum_planes(const uint8_t *__restrict__ dec, uint16_t *__restrict__ dec3, int64_t count, int64_t total)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const uint8_t *d = dec + 2 * (i >= count ? i / count : 0) * count + i;  // pixel i % count of its image's R plane
    dec3[i] = (uint16_t)((int)d[0] + (int)d[count] + (int)d[2 * count]);
}

int launch_sum_planes(const uint8_t *d_dec, uint16_t *d_dec3, const Geom &g, cudaStream_t s, int n_images)
{
    const int64_t count = (int64_t)g.sw * g.sh, total = count * n_images;
    k_sum_planes<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(d_dec, d_dec3, count, total);
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

// A batch of same-size images (fic_encode_batch) is one launch over n * NR CTAs: the flat CTA index jf = image * NR + j
// picks the image, whose pixels start img_stride elements (ARGB ints or bytes of its C planes) after the previous
// image's, and the codes go to row jf of the [n][NR] code tables.
template <int B, int C, bool ARGB>
__global__ void __launch_bounds__(kDirectThreads)
k_encode_fused(const void *__restrict__ src, float *__restrict__ info, int32_t *__restrict__ q, Geom g, int64_t j0,
               size_t img_stride)
{
    constexpr int n = B * B, step = B / 4;
    extern __shared__ __align__(16) uint8_t s_tile[];  // C planes of TW x TW decimated pixels
    __shared__ int s_r[C][n];                          // the range block, per channel
    __shared__ float s_gR[C == 3 ? n : 1];             // RGB: sum over the channels of (r - rmean_c), FC:785-786
    __shared__ int s_sum[C][kDirectThreads / 32];
    __shared__ float s_err[kDirectThreads / 32];
    __shared__ int s_c[kDirectThreads / 32];
    const int64_t jf = j0 + blockIdx.x;
    const int64_t image = jf / g.NR, j = jf - image * g.NR;
    src = ARGB ? (const void *)((const int32_t *)src + image * img_stride) : (const void *)((const uint8_t *)src + image * img_stride);
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
        write_grey_code(info, q, jf, c, grey_solve(dot - dmean * vR, varD, rm[0], dmean), false, 0);
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
        write_rgb_code(info, q, jf, c, rgb_solve(kov, dv, dm, rm));
    }
}

bool fused_encode_applicable(const Geom &g) { return g.wk <= 16 && g.n_iso == 1; }

template <int C, bool ARGB>
static int launch_fused_t(const void *d_src, const Geom &g, int64_t j0, int64_t j1, size_t img_stride, float *d_info, int32_t *d_q,
                          cudaStream_t s)
{
    const int step = g.B / 4, TW = (g.wk - 1) * step + g.B;
    const size_t smem = (size_t)C * TW * TW;  // <= 3 * 76 * 76 = 17 KB
    int launches = 0;
    for (int64_t at = j0; at < j1;) {
        const unsigned chunk = (unsigned)(j1 - at < (1 << 30) ? j1 - at : (1 << 30));
        if (g.B == 4) k_encode_fused<4, C, ARGB><<<chunk, kDirectThreads, smem, s>>>(d_src, d_info, d_q, g, at, img_stride);
        else if (g.B == 8) k_encode_fused<8, C, ARGB><<<chunk, kDirectThreads, smem, s>>>(d_src, d_info, d_q, g, at, img_stride);
        else k_encode_fused<16, C, ARGB><<<chunk, kDirectThreads, smem, s>>>(d_src, d_info, d_q, g, at, img_stride);
        at += chunk;
        launches++;
    }
    return launches;
}

int launch_encode_fused(const void *d_src, int src_is_argb, const Geom &g, int64_t j0, int64_t j1, float *d_info, int32_t *d_q,
                        cudaStream_t s, int n_images)
{
    if (j1 <= j0) return 0;
    const size_t plane = (size_t)g.W * g.H, stride = src_is_argb ? plane : g.C * plane;
    if (n_images > 1) j1 = n_images * g.NR;  // a batch: every range of every image, the flat range [0, n NR)
    if (g.C == 1) return src_is_argb ? launch_fused_t<1, true>(d_src, g, j0, j1, stride, d_info, d_q, s) : launch_fused_t<1, false>(d_src, g, j0, j1, stride, d_info, d_q, s);
    return src_is_argb ? launch_fused_t<3, true>(d_src, g, j0, j1, stride, d_info, d_q, s) : launch_fused_t<3, false>(d_src, g, j0, j1, stride, d_info, d_q, s);
}

// ------------------------------------------------------------------------------------
// K3s: code solve + quantisation for the winning candidate.  One thread per range block.  A group of images passes
// the flat range [0, n NR): flat row jf = image * NR + j reads that image's planes and stats (as the pool builders lay
// them out) and writes row jf of best / info / q.
// ------------------------------------------------------------------------------------
__global__ void k_solve_grey(const uint8_t *__restrict__ src, const uint8_t *__restrict__ dec,
                             const int32_t *__restrict__ dsum, const int32_t *__restrict__ dsq,
                             const int32_t *__restrict__ rsum, const int32_t *__restrict__ best,
                             float *__restrict__ info, int32_t *__restrict__ q, Geom g, int64_t j0, int64_t j1)
{
    const int64_t jf = j0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (jf >= j1) return;
    const int64_t image = jf >= g.NR ? jf / g.NR : 0, j = jf - image * g.NR;  // (a single image divides nothing)
    src += image * g.W * g.H;
    dec += image * g.sw * g.sh;
    dsum += image * g.ND;
    dsq += image * g.ND;
    rsum += image * g.NR;
    best += image * g.NR;
    info = info ? info + image * g.NR * code_stride(g) : info;
    q = q ? q + image * g.NR * code_stride(g) : q;
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
    const int64_t jf = j0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // see k_solve_grey
    if (jf >= j1) return;
    const int64_t image = jf >= g.NR ? jf / g.NR : 0, j = jf - image * g.NR;
    src += image * 3 * g.W * g.H;
    dec += image * 3 * g.sw * g.sh;
    dsum += image * 3 * g.ND;
    dsq += image * 3 * g.ND;
    rsum += image * 3 * g.NR;
    best += image * g.NR;
    info = info ? info + image * g.NR * 5 : info;
    q = q ? q + image * g.NR * 5 : q;
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

}  // namespace fic
