// fic_decode.cu -- the decoder of libfic_b200 (K4, sm_100a): code dequantisation, the Jacobi sweeps of the iterative
// decode and the one-shot collage, the one-launch decoder for small images, the exact avgError bookkeeping (the
// state block and the replay of the reference's float sum), and the host driver that picks among them.
//
// file:line citations refer to the reference, src/bvk_ss19/FractalCompression.java (FC).
#include <math.h>
#include <string.h>

#include <vector>

#include "fic_device.cuh"

namespace fic {

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

// Stream ints -> float codes (FC:372-374 / FC:446-450) and window-local -> codebook
// index (FC:853-893 calculateIndices, float division / float remainder as in Java).
// With `unquantised` the float codes of an encode are used instead (collage, FC:271).
// st->bad_index is set when an index falls outside the pool (the reference would throw).
// packed != 0 (decoder loop over the row-pair interleaved plane, k_decode_sweep_il): doff[j] is the domain block's
// position in the decimated plane as (row << 16) | column instead of its byte offset.
__device__ __forceinline__ void dequant_one(int64_t j, const int32_t *__restrict__ q, const float *__restrict__ info_in,
                                            float *__restrict__ code, int32_t *__restrict__ doff, const Geom &g, int unquantised,
                                            DecodeState *st, int packed)
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
        atomicOr(&st->bad_index, 1ull);
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
                          DecodeState *st, int packed)
{
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= g.NR) return;
    dequant_one(j, q, info_in, code, doff, g, unquantised, st, packed);
}

__global__ void k_fill(uint4 *p, int64_t n16, uint32_t v)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n16; i += stride) p[i] = make_uint4(v, v, v, v);
}

// Control block of one decoder sweep.  st == nullptr: a plain sweep (the one-shot collage).  Otherwise the sweep
// returns at once when the done flag is set, adds its squared pixel changes to st->sq_sum and, with finish != 0, its
// last CTA folds the sweep into the state (avgError, iteration count, done flag; FC:413-417) so that the host need not
// look at every sweep.
struct SweepCtl {
    DecodeState *st;
    int it;      // sweep index (FC:381 counter)
    int finish;  // 1: fold inside the sweep kernel -- only when the float sum needs no replay (see k_sweep_finish)
    float fwh;   // (float)(W*H), FC:413
};

// A state word that another CTA or an earlier kernel may have written.
__device__ __forceinline__ uint32_t state_word(const uint32_t &x) { return *(volatile const uint32_t *)&x; }

// Sweeps are enqueued ahead of the host's knowledge of convergence (FC:414): once the done flag is set every later
// sweep returns at once, so the image stays the converged one.
__device__ __forceinline__ bool sweep_done(const SweepCtl &ctl)
{
    return ctl.st && state_word(ctl.st->done) != 0;
}

// Records sweep `it` whose float running sum of squared changes is `sum` (FC:407 / FC:493): avgError = sum / (W*H)
// (FC:413); below 1 the decode has converged and stops with that value (FC:414), otherwise the value is kept only
// after the last allowed sweep (FC:416-417).
__device__ __forceinline__ void record_sweep(DecodeState *st, int it, float sum, float fwh, bool last)
{
    const float avg = __fdiv_rn(sum, fwh);
    st->iters = (uint32_t)(it + 1);
    if (avg < 1.0f) {
        st->avg_bits = __float_as_uint(avg);
        st->done = 1u;
    } else {
        st->avg_bits = last ? __float_as_uint(avg) : 0u;
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

// Common tail of the sweep kernels: add the CTA's squared changes to st->sq_sum; with ctl.finish the last CTA to get
// here records the sweep (no separate kernel, no host round trip per sweep).  decode_run only asks for that on
// sweeps whose float running sum needs no replay: it is the exact integer S when S < 2^24 (every float partial sum
// is then exact); S >= 2^24 >= W*H means "not converged" and the value is discarded (never the last sweep here).
__device__ __forceinline__ void sweep_tail(const SweepCtl &ctl, unsigned long long local)
{
    if (!ctl.st) return;
    const unsigned long long tot = cta_sum(local);
    if (threadIdx.x == 0) {
        if (tot) atomicAdd(&ctl.st->sq_sum, tot);
        if (!ctl.finish) return;
        __threadfence();
        if (atomicAdd(&ctl.st->ticket, 1u) == gridDim.x - 1) {
            __threadfence();
            const unsigned long long S = atomicExch(&ctl.st->sq_sum, 0ull);
            ctl.st->ticket = 0u;
            record_sweep(ctl.st, ctl.it, S < (1ull << 24) ? (float)S : 2.0f * ctl.fwh, ctl.fwh, false);
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
//   st->sq_sum += sum of squared pixel changes (exact integer; see decode_run for how
//   this reproduces the reference's float avgError), perr (optional) gets the per-pixel
//   squared change in the reference's accumulation order (range-major, ry, rx).
template <int C>
__global__ void __launch_bounds__(256)
k_decode_sweep(const uint8_t *__restrict__ dec_in, uint8_t *__restrict__ img, uint8_t *__restrict__ dec_out,
               const float *__restrict__ code, const int32_t *__restrict__ doff, Geom g, SweepCtl ctl,
               int32_t *__restrict__ perr)
{
    if (sweep_done(ctl)) return;
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

// Warp tiles of a sweep over the interleaved plane: 16 x 2 strips each (see sweep_il_body).
__host__ __device__ inline uint32_t il_tiles(const Geom &g) { return (((uint32_t)g.W / 8u + 15u) >> 4) * ((uint32_t)g.H >> 2); }

// The warp sweeps tiles wt, wt + wt_step, ... below wt_end.
template <int C, int B, bool PERR, bool FIRST, bool NC = true>
__device__ __forceinline__ unsigned long long sweep_il_body(const uint8_t *__restrict__ dec_in, uint8_t *__restrict__ img,
                                                            uint8_t *__restrict__ dec_out, const float *__restrict__ code,
                                                            const int32_t *__restrict__ dpos, const Geom &g, int32_t *__restrict__ perr,
                                                            uint32_t wt, uint32_t wt_end, uint32_t wt_step)
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
    const uint32_t tiles_x = (sw8 + 15u) >> 4;
    const uint32_t lane = threadIdx.x & 31u;
    for (; wt < wt_end; wt += wt_step) {
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
    sweep_tail(ctl, sweep_il_body<C, B, PERR, FIRST>(dec_in, img, dec_out, code, dpos, g, perr, blockIdx.x * 8u + (threadIdx.x >> 5),
                                                     il_tiles(g), gridDim.x * 8u));
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
//
// A batch of n same-size images (fic_decode_batch) runs in the same launch: one state block per image, the images'
// buffers back to back.  A unit of work is (image, 8 consecutive warp tiles), one CTA's worth; CTAs grid-stride over
// the units of all images, so with one image unit blockIdx.x + k gridDim.x is exactly the tiles the per-sweep kernel's
// CTA visits.  A CTA sums its squared changes per image and adds them to that image's state when its next unit belongs
// to another image and at the end of the sweep.  The fold decides every image on its own; an image that converged or
// bailed is frozen (its units are skipped) while the others sweep on.

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

// MULTI: n_img images with their carried-in avgError at `carries`; otherwise the one image of a single decode with `carry`
// (n_img == 1 is then known at compile time, and what only a batch needs -- the flushes between images, the frozen
// images, the fold loop -- compiles away).  The batch form asks for 4 CTAs per SM (<= 64 registers): left to itself
// ptxas gives it 40 registers and a spill.
template <int C, int B, bool MULTI>
__global__ void __launch_bounds__(256, MULTI ? 4 : 0)
k_decode_small(const int32_t *__restrict__ q, float *__restrict__ code, int32_t *__restrict__ dpos, uint8_t *__restrict__ img,
               uint8_t *__restrict__ dec_a, uint8_t *__restrict__ dec_b, int32_t *__restrict__ argb_out, Geom g,
               DecodeState *st, int max_iters, float carry, float fwh, unsigned long long skip_from, uint32_t n_img,
               const float *__restrict__ carries)
{
    constexpr int S = C == 1 ? 3 : 5;
    const uint32_t NR = (uint32_t)g.NR, n = MULTI ? n_img : 1u;
    const size_t planeI = (size_t)C * g.W * g.H, planeD = (size_t)C * g.sw * g.sh;
    uint32_t epoch = 0;
    for (uint32_t jf = blockIdx.x * 256u + threadIdx.x; jf < n * NR; jf += gridDim.x * 256u) {
        const uint32_t im = MULTI ? jf / NR : 0u;
        dequant_one(jf - im * NR, q + (size_t)im * NR * S, nullptr, code + (size_t)im * NR * S, dpos + (size_t)im * NR, g, 0, st + im, 1);
    }
    grid_barrier(&st->barrier, epoch);
    const uint32_t tiles = il_tiles(g), per_img = (tiles + 7u) / 8u, units = n * per_img, warp = threadIdx.x >> 5;
    // unit u = im * per_img + lu, stepped by gridDim.x = dq * per_img + dr without a division per unit
    const uint32_t im0 = MULTI ? blockIdx.x / per_img : 0u, lu0 = blockIdx.x - im0 * per_img;
    const uint32_t dq = MULTI ? gridDim.x / per_img : 0u, dr = MULTI ? gridDim.x - dq * per_img : 0u;
    uint8_t *din = dec_a, *dout = dec_b;
    uint32_t bail0 = 0;  // the first image's bail word after the last fold
    for (int it = 0; it < max_iters; it++) {
        unsigned long long local = 0;  // this CTA's squared changes of image `cur` so far
        uint32_t cur = im0, im = im0, lu = lu0;
        bool pending = false;
        for (uint32_t u = blockIdx.x; u < units; u += gridDim.x, im += dq, lu += dr) {
            if (MULTI && lu >= per_img) {
                lu -= per_img;
                im++;
            }
            const uint32_t t0 = 8u * (MULTI ? lu : u);
            if (im != cur) {
                if (pending) {
                    const unsigned long long tot = cta_sum(local);
                    if (threadIdx.x == 0 && tot) atomicAdd(&st[cur].sq_sum, tot);
                    __syncthreads();  // cta_sum's shared partials are read by thread 0 before they are rewritten
                    local = 0;
                    pending = false;
                }
                cur = im;
            }
            // frozen (with one image the loop only runs while it sweeps)
            if (MULTI && (state_word(st[im].done) | state_word(st[im].bail))) continue;
            const uint32_t wt = t0 + warp, wt_end = min(tiles, t0 + 8u);
            uint8_t *const pi = img + im * planeI, *const pin = din + im * planeD, *const pout = dout + im * planeD;
            const float *const pc = code + (size_t)im * NR * S;
            const int32_t *const pp = dpos + (size_t)im * NR;
            local += it == 0 ? sweep_il_body<C, B, false, true, false>(pin, pi, pout, pc, pp, g, nullptr, wt, wt_end, 8u)
                             : sweep_il_body<C, B, false, false, false>(pin, pi, pout, pc, pp, g, nullptr, wt, wt_end, 8u);
            pending = true;
        }
        const unsigned long long tot = cta_sum(local);
        if (threadIdx.x == 0 && tot) atomicAdd(&st[cur].sq_sum, tot);
        grid_barrier(&st->barrier, epoch);
        if (blockIdx.x == 0) {
            const bool last = it == max_iters - 1;
            bool sweeping = false;  // some image of this thread sweeps again
            for (uint32_t i = threadIdx.x; i < n; i += 256u) {
                DecodeState *const si = st + i;
                // frozen images (one image is still sweeping whenever the loop runs: no state read on that path)
                if (MULTI && (si->done | si->bail)) continue;
                const unsigned long long sum = atomicExch(&si->sq_sum, 0ull);
                const float c0 = it == 0 ? (MULTI ? carries[i] : carry) : 0.0f;
                bool again;  // the image sweeps again
                if (c0 == 0.0f && sum < (1ull << 24)) {  // the float sum is the exact integer
                    record_sweep(si, it, (float)sum, fwh, last);
                    again = !(__fdiv_rn((float)sum, fwh) < 1.0f);  // not converged (record_sweep's test)
                } else if (!last && c0 >= 0.0f && sum >= skip_from) {  // certainly not converged; the value is discarded
                    si->iters = (uint32_t)(it + 1);
                    si->avg_bits = 0u;
                    again = true;
                } else {
                    si->bail = 1u;
                    again = false;
                }
                sweeping |= !last && again;
            }
            if (MULTI) sweeping = __syncthreads_or(sweeping);  // (one image: thread 0 folded it)
            if (threadIdx.x == 0) {
                st->ticket = sweeping ? 1u : 0u;
                __threadfence();
            }
        }
        grid_barrier(&st->barrier, epoch);
        bail0 = state_word(st->bail);  // read beside the ticket: the one image's verdict costs no extra round trip
        if (!state_word(st->ticket)) break;
        uint8_t *t = din; din = dout; dout = t;
    }
    if (argb_out)
        for (uint32_t i = 0; i < n; i++)
            if (!(i == 0 ? bail0 : state_word(st[i].bail))) pack_argb<C>((const uchar4 *)(img + i * planeI), (int4 *)(argb_out + (size_t)i * g.W * g.H), (int64_t)g.W * g.H / 4);
}

// The literal float accumulation (FC:407 / FC:493) over perr[begin, end), stopping once the sum reaches `limit` (one
// warp; every lane returns the same sum).  Zero terms are skipped (x + 0 == x).  GROUPS (k_sweep_finish): while the sum
// is an integer and stays <= 2^24 every add is exact, so a whole 128-term group is added at once.  That argument needs
// a sum >= 0: k_sweep_finish takes the shortcut from any carry, k_replay_walk never takes it.
template <bool GROUPS>
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
        if (GROUPS) {
            int tot = v.x + v.y + v.z + v.w;  // <= 4 * 3 * 255^2
            for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
            if (tot == 0) continue;
            if (a == floorf(a) && __fadd_rn(a, (float)tot) <= 16777216.0f) {  // every partial sum is an exact integer
                a = __fadd_rn(a, (float)tot);
                continue;
            }
        }
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

// Folds a sweep that may need the reference's float accumulation replayed (FC:407 / FC:493): the first sweep when
// the never-reset static avgError (FC:20) carries a value in, the last allowed sweep (its value is kept whatever it is,
// FC:416), and every sweep of an image above 2^24 pixels (where the sum may pass 2^24 and still converge).
// One warp.  The running binary32 sum is order dependent once it passes 2^24, so it is replayed in loop order over
// the per-pixel squared changes (replay_literal<true>); if the exact total S is below 2^24 and nothing is carried in,
// the sum is S.  The sum never decreases (the terms are >= 0): on a sweep whose value is discarded unless it converged
// (FC:413-417) the replay stops once the sum reaches W*H.
__global__ void k_sweep_finish(const int32_t *__restrict__ perr, int64_t count, DecodeState *st, int it, int last,
                               float carry, float fwh)
{
    if (blockIdx.x || threadIdx.x >= 32) return;
    if (state_word(st->done)) return;
    const unsigned long long S = *(volatile unsigned long long *)&st->sq_sum;
    float a = carry;  // FC:20: the first sweep starts from whatever the previous decode left; later ones from 0
    if (!(a == 0.0f && S < (1ull << 24))) a = replay_literal<true>(perr, 0, count, a, last ? __int_as_float(0x7f800000) : fwh);
    else a = (float)S;
    if (threadIdx.x == 0) {
        st->sq_sum = 0ull;
        record_sweep(st, it, a, fwh, last);
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
__device__ __forceinline__ bool replay_not_needed(const DecodeState *st, float carry, unsigned long long skip_from)
{
    // done already; or the sweep's exact total is below 2^24 and nothing is carried in: the float sum is that integer
    const unsigned long long S = *(volatile const unsigned long long *)&st->sq_sum;
    return state_word(st->done) != 0 || (carry == 0.0f && S < (1ull << 24)) || S >= skip_from;
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
                                                     const DecodeState *st, float carry, unsigned long long skip_from)
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
__global__ void __launch_bounds__(1024) k_replay_scan(ReplayChunk *__restrict__ ch, int nchunks, const DecodeState *st, float carry,
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
                                                            const DecodeState *st, float carry, unsigned long long skip_from)
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

// A group of 32 chunks composed into one record (valid when its non-empty chunks share one binade guess), so that the
// walker steps over 131 072 pixels at a time wherever the sum is far from a binade crossing.
struct ReplayGroup { unsigned long long sum; int32_t k; uint32_t d0, d1, e0, e1; };
constexpr int kRepGroup = 32;

__global__ void k_replay_groups(const ReplayChunk *__restrict__ ch, int nchunks, ReplayGroup *__restrict__ gr, int ngroups,
                                const DecodeState *st, float carry, unsigned long long skip_from)
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
                              const ReplayGroup *__restrict__ gr, int ngroups, DecodeState *st, int it, int last, float carry,
                              float fwh, unsigned long long skip_from)
{
    if (blockIdx.x || threadIdx.x >= 32) return;
    if (state_word(st->done)) return;
    const int lane = threadIdx.x;
    const unsigned long long S = *(volatile unsigned long long *)&st->sq_sum;
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
                    a = replay_literal<false>(perr, b0, b1, a, __int_as_float(0x7f800000));
                }
            }
        }
    }
    if (lane == 0) {
        st->sq_sum = 0ull;
        record_sweep(st, it, a, fwh, last);
    }
}

// ---- host side ------------------------------------------------------------------------------------------------------

#define DCU(call) \
    do { const cudaError_t e_ = (call); if (e_ != cudaSuccess) return DecodeStatus{FIC_E_CUDA, e_, #call, __FILE__, __LINE__}; } while (0)

// Which kernels a decode of geometry g runs, decided once per call.
enum class SweepFamily { IL, V8, QUAD };  // k_decode_sweep_il, k_decode_sweep_v8, k_decode_sweep
struct Plan {
    SweepFamily sweep;
    bool implicit_start;  // the first sweep starts from the constant-128 image and reads nothing (FIRST)
    bool one_launch;      // the whole decode may run as k_decode_small
};

// Sweeps over a plain (not interleaved) decimated plane; the isometry extension uses the quad kernel (per-pixel gather).
static Plan plain_plan(const Geom &g)
{
    return Plan{g.W % 8 == 0 && g.n_iso == 1 ? SweepFamily::V8 : SweepFamily::QUAD, false, false};
}

static Plan decode_plan(const Geom &g)
{
    const bool il = sweep_interleaved(g);
    return Plan{il ? SweepFamily::IL : plain_plan(g).sweep, g.W % 8 == 0 && g.n_iso == 1 && g.B >= 8,
                il && (int64_t)g.W * g.H <= ((int64_t)1 << 20)};
}

// Launches the grid-stride kernel K over min(need, one wave) CTAs of 256 threads.  The sweeps are grid-stride over
// exactly one wave of resident CTAs (SMs x occupancy of the kernel): a second, partly filled wave cost a third of the
// sweep at 4096^2 (1184 CTAs on 740 slots, profiles/README.md).  The wave is measured once per kernel.
template <auto K, class... A>
static void launch_wave(int64_t need, cudaStream_t s, A... args)
{
    static const int64_t wave = [] {
        int dev = 0, sms = 148, per_sm = 4;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, K, 256, 0) != cudaSuccess || per_sm < 1) per_sm = 4;
        return (int64_t)sms * per_sm;
    }();
    K<<<(unsigned)(need < wave ? need : wave), 256, 0, s>>>(args...);
}

template <int C, int B, class... A>
static void launch_sweep_il(int64_t need, bool perr, bool first, cudaStream_t s, A... args)
{
    if (perr) (first ? launch_wave<k_decode_sweep_il<C, B, true, true>, A...> : launch_wave<k_decode_sweep_il<C, B, true, false>, A...>)(need, s, args...);
    else (first ? launch_wave<k_decode_sweep_il<C, B, false, true>, A...> : launch_wave<k_decode_sweep_il<C, B, false, false>, A...>)(need, s, args...);
}

// One sweep of the family p chose.  first (p.implicit_start only): the sweep starts from the constant-128 image and
// reads neither img nor dec_in.  IL: the decimated planes are row-pair interleaved and doff holds packed positions.
template <int C>
static int launch_sweep(const Plan &p, const Geom &g, const uint8_t *dec_in, uint8_t *img, uint8_t *dec_out, const float *code,
                        const int32_t *doff, const SweepCtl &ctl, int32_t *perr, bool first, cudaStream_t s)
{
    if (p.sweep == SweepFamily::IL) {
        const int64_t tiles = (int64_t)((g.W / 8 + 15) / 16) * (g.H / 4), need = (tiles + 7) / 8;  // one warp per 16 x 2 strips
        if (g.B == 8) launch_sweep_il<C, 8>(need, perr, first, s, dec_in, img, dec_out, code, doff, g, ctl, perr);
        else launch_sweep_il<C, 16>(need, perr, first, s, dec_in, img, dec_out, code, doff, g, ctl, perr);
    } else if (p.sweep == SweepFamily::V8) {
        const int64_t strips = (int64_t)(g.W / 8) * (g.H / 2), need = (strips + 255) / 256;
        if (first) launch_wave<k_decode_sweep_v8<C, true>>(need, s, dec_in, img, dec_out, code, doff, g, ctl, perr);
        else launch_wave<k_decode_sweep_v8<C, false>>(need, s, dec_in, img, dec_out, code, doff, g, ctl, perr);
    } else {
        const int64_t quads = (int64_t)(g.W / 2) * (g.H / 2), need = (quads + 255) / 256;
        launch_wave<k_decode_sweep<C>>(need, s, dec_in, img, dec_out, code, doff, g, ctl, perr);
    }
    return 1;
}

// d_info != nullptr: the float codes of an encode (collage), not quantised ones.  packed: positions for k_decode_sweep_il.
static int launch_dequant(const int32_t *d_q, const float *d_info, float *d_code, int32_t *d_off, const Geom &g, bool packed,
                          DecodeState *d_state, cudaStream_t s)
{
    k_dequant<<<(unsigned)((g.NR + 127) / 128), 128, 0, s>>>(d_q, d_info, d_code, d_off, g, d_info ? 1 : 0, d_state, packed ? 1 : 0);
    return 1;
}

static int launch_fill(uint8_t *d_planes, size_t bytes, int value, cudaStream_t s)
{
    uint32_t v = (uint32_t)(value & 0xff) * 0x01010101u;
    int64_t n16 = (int64_t)(bytes / 16);  // plane sizes are multiples of 16 (W % 4 == 0, H % 4 == 0)
    int blocks = (int)((n16 + 255) / 256 < 148 * 8 ? (n16 + 255) / 256 : 148 * 8);
    if (blocks < 1) blocks = 1;
    k_fill<<<blocks, 256, 0, s>>>((uint4 *)d_planes, n16, v);
    return 1;
}

static int launch_pack_argb(const uint8_t *d_planes, int32_t *d_argb, const Geom &g, cudaStream_t s)
{
    int64_t quads = (int64_t)g.W * g.H / 4;
    int blocks = (int)((quads + 255) / 256 < 148 * 16 ? (quads + 255) / 256 : 148 * 16);
    if (blocks < 1) blocks = 1;
    if (g.C == 1)
        k_pack_argb<1><<<blocks, 256, 0, s>>>((const uchar4 *)d_planes, (int4 *)d_argb, quads);
    else
        k_pack_argb<3><<<blocks, 256, 0, s>>>((const uchar4 *)d_planes, (int4 *)d_argb, quads);
    return 1;
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

// The whole decode of n_img images in one cooperative launch (k_decode_small; p.one_launch only).  Returns 1 if the kernel
// was launched (the state blocks, zero on entry, then tell whether each image finished or bailed), 0 if this device does
// not take it.  MULTI (a batch): carries, device [n_img]; otherwise the one image of a single decode, `carry`.
template <int C, int B, bool MULTI>
static int launch_small(const Work &w, const Geom &g, const int32_t *d_q, int32_t *d_pos, uint8_t *d_img, int32_t *d_argb,
                        int max_iters, float carry, float fwh, cudaStream_t s, uint32_t n_img, const float *carries)
{
    static int coop = -1, per_sm = 0, sms = 0;
    if (coop < 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_decode_small<C, B, MULTI>, 256, 0) != cudaSuccess) per_sm = 0;
        cudaGetLastError();
    }
    if (coop <= 0 || per_sm < 1) return 0;
    int64_t grid = (int64_t)n_img * ((il_tiles(g) + 7) / 8);  // units of 8 warp tiles
    if (grid > (int64_t)sms * per_sm) grid = (int64_t)sms * per_sm;
    Geom gg = g;
    float *code = w.dcode;
    uint8_t *dec_a = w.dec, *dec_b = w.dec2;
    DecodeState *st = w.state;
    unsigned long long skip_from = skip_from_of(fwh, (int64_t)g.W * g.H);
    void *args[] = {(void *)&d_q, (void *)&code, (void *)&d_pos, (void *)&d_img, (void *)&dec_a, (void *)&dec_b, (void *)&d_argb,
                    (void *)&gg, (void *)&st, (void *)&max_iters, (void *)&carry, (void *)&fwh, (void *)&skip_from, (void *)&n_img,
                    (void *)&carries};
    if (cudaLaunchCooperativeKernel((const void *)k_decode_small<C, B, MULTI>, dim3((unsigned)grid), dim3(256), args, 0, s) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return 1;
}

static int64_t replay_chunks(int64_t count) { return (count + kRepChunk - 1) / kRepChunk; }
static int64_t replay_groups(int64_t count) { return (replay_chunks(count) + kRepGroup - 1) / kRepGroup; }

size_t decode_replay_bytes(int64_t pixels)
{
    if (pixels < ((int64_t)1 << 22)) return 0;
    return sizeof(ReplayGroup) * (size_t)replay_groups(pixels) + sizeof(ReplayChunk) * (size_t)replay_chunks(pixels);
}

// Folds a sweep over `count` pixels whose float running sum may have to be replayed in loop order (see k_sweep_finish):
// one warp below 2^22 pixels, the chunked replay in w.replay above.
static int launch_sweep_finish(const Work &w, int64_t count, int it, bool last, float carry, float fwh, cudaStream_t s)
{
    if (decode_replay_bytes(count)) {
        const int nchunks = (int)replay_chunks(count), ngroups = (int)replay_groups(count);
        ReplayGroup *gr = (ReplayGroup *)w.replay;
        ReplayChunk *ch = (ReplayChunk *)(gr + ngroups);
        // the last allowed sweep keeps its value whatever it is
        const unsigned long long skip_from = !last && carry >= 0.0f ? skip_from_of(fwh, count) : ~0ull;
        k_replay_sums<<<nchunks, 256, 0, s>>>(w.perr, count, ch, w.state, carry, skip_from);
        k_replay_scan<<<1, 1024, 0, s>>>(ch, nchunks, w.state, carry, skip_from);
        k_replay_transducers<<<nchunks, 256, 0, s>>>(w.perr, count, ch, w.state, carry, skip_from);
        k_replay_groups<<<(ngroups + 127) / 128, 128, 0, s>>>(ch, nchunks, gr, ngroups, w.state, carry, skip_from);
        k_replay_walk<<<1, 32, 0, s>>>(w.perr, count, ch, nchunks, gr, ngroups, w.state, it, last, carry, fwh, skip_from);
        return 5;
    }
    k_sweep_finish<<<1, 32, 0, s>>>(w.perr, count, w.state, it, last, carry, fwh);
    return 1;
}

// Waits for the stream, then reads the state block that was copied to h_state before.
static DecodeStatus sync_state(const DecodeState *h_state, cudaStream_t s)
{
    DCU(cudaStreamSynchronize(s));
    return DecodeStatus{h_state->bad_index ? FIC_E_STREAM : FIC_OK};
}

// avgError bookkeeping (FC:407-417).  The reference adds every squared pixel change to a binary32 running sum,
// divides by W*H after the sweep and stops below 1.  The sum is an exact integer while it stays below 2^24, so with
// W*H <= 2^24 the integer total S decides: S < 2^24 -> the float sum equals S; otherwise the float sum is
// >= 2^24 >= W*H and the sweep did not converge (its value is then discarded, FC:416-417).  Such sweeps are folded
// into the device-side state by the sweep kernel's last CTA.  Sweeps whose float sum may be both inexact and kept
// (carry-in on the first sweep, the last allowed sweep, images above 2^24 pixels) also write the per-pixel squared
// changes in loop order and are folded by k_sweep_finish or the chunked replay, which replay the float accumulation
// where they must.  Sweeps are enqueued eight at a time without looking at the result: once the done flag is set the
// remaining ones return immediately, and the host reads the state once per batch instead of once per sweep.
DecodeStatus decode_run(const Work &w, const Geom &g, const int32_t *d_q, uint8_t *img, int32_t *argb_out, uint8_t *planes_out,
                        int max_iters, float *avg_error, int *iterations, void *h_scratch, cudaEvent_t ev0, cudaEvent_t end,
                        fic_timings *tm, cudaStream_t s)
{
    const Plan p = decode_plan(g);
    const DecodeState *hs = (const DecodeState *)h_scratch;
    const size_t plane = (size_t)g.W * g.H;
    const bool big = (int64_t)plane > ((int64_t)1 << 24);
    const float carry = avg_error ? *avg_error : 0.0f;
    const float fwh = (float)(g.W * g.H);  // FC:413 (float)(width*height)
    int32_t *doff = (int32_t *)(w.dcode + g.NR * code_stride(g));
    int launches = 0;
    DecodeStatus st;
    auto enqueue_output = [&]() -> DecodeStatus {
        if (argb_out) {
            launches += launch_pack_argb(img, w.argb, g, s);
            DCU(cudaMemcpyAsync(argb_out, w.argb, sizeof(int32_t) * plane, cudaMemcpyDeviceToHost, s));
        } else if (planes_out) {
            DCU(cudaMemcpyAsync(planes_out, img, g.C * plane, cudaMemcpyDeviceToHost, s));
        }
        return DecodeStatus{};
    };
    DCU(cudaMemsetAsync(w.state, 0, sizeof(DecodeState), s));
    bool done = false;
    // Small images (the reference's own sizes): the whole decode in ONE cooperative launch (k_decode_small) -- unless its
    // avgError would need the float sum replayed (bail), in which case the decode is repeated below.
    const auto small = g.B == 8 ? (g.C == 1 ? launch_small<1, 8, false> : launch_small<3, 8, false>)
                                : (g.C == 1 ? launch_small<1, 16, false> : launch_small<3, 16, false>);
    if (p.one_launch && small(w, g, d_q, doff, img, argb_out ? w.argb : nullptr, max_iters, carry, fwh, s, 1u, nullptr)) {
        launches++;
        DCU(cudaMemcpyAsync(h_scratch, w.state, sizeof(DecodeState), cudaMemcpyDeviceToHost, s));
        // the output is copied without waiting for the verdict (<= 4 MB); a bailed decode overwrites it below
        if (argb_out) DCU(cudaMemcpyAsync(argb_out, w.argb, sizeof(int32_t) * plane, cudaMemcpyDeviceToHost, s));
        else if (planes_out) DCU(cudaMemcpyAsync(planes_out, img, g.C * plane, cudaMemcpyDeviceToHost, s));
        DCU(cudaEventRecord(end, s));
        if ((st = sync_state(hs, s)).rc) return st;
        done = !hs->bail;
        if (!done) DCU(cudaMemsetAsync(w.state, 0, sizeof(DecodeState), s));
    }
    if (!done) {
        launches += launch_dequant(d_q, nullptr, w.dcode, doff, g, p.sweep == SweepFamily::IL, w.state, s);
        // The start image is the constant 128 (FC:360, FC:1142-1148) and so is its 2x-decimated plane, for every tap rule
        // (FC:970-1007, FC:901-962).  For B >= 8 neither is materialised: the first sweep knows what it would read.
        if (!p.implicit_start) {
            launches += launch_fill(img, g.C * plane, 128, s);
            DCU(cudaMemsetAsync(w.dec, 128, (size_t)g.C * g.sw * g.sh, s));
        }
        uint8_t *dcur = w.dec, *dnext = w.dec2;
        // Small images: the output copy is enqueued behind every batch, so that a decode that converges within the batch
        // (the usual case) costs one host synchronisation in all; a later batch simply copies again.  Device-resident
        // output: the batch is the whole call (the end event must not wait for the host's state read).
        const bool host_out = argb_out || planes_out;
        const bool speculative_out = host_out && plane * (argb_out ? 4 : g.C) <= ((size_t)4 << 20);
        // a skipped sweep still costs a launch (~1.5 us), a second batch a host round trip (~40 us): grey decodes converge
        // in 5-9 sweeps, the reference's RGB quantisation (FC:250-254) needs 13-22
        const int batch = (g.C == 3 && speculative_out) ? 16 : 8;
        int it = 0;
        while (it < max_iters) {
            const int batch_end = it + batch < max_iters ? it + batch : max_iters;
            for (; it < batch_end; it++) {
                const bool last = it == max_iters - 1;
                const bool replay = big || last || (it == 0 && carry != 0.0f);
                const SweepCtl ctl = {w.state, it, replay ? 0 : 1, fwh};
                launches += (g.C == 1 ? launch_sweep<1> : launch_sweep<3>)(p, g, dcur, img, dnext, w.dcode, doff, ctl, replay ? w.perr : nullptr, it == 0 && p.implicit_start, s);
                if (replay) launches += launch_sweep_finish(w, (int64_t)plane, it, last, it == 0 ? carry : 0.0f, fwh, s);
                uint8_t *t = dcur; dcur = dnext; dnext = t;
            }
            DCU(cudaMemcpyAsync(h_scratch, w.state, sizeof(DecodeState), cudaMemcpyDeviceToHost, s));
            if (speculative_out && (st = enqueue_output()).rc) return st;
            if (speculative_out || !host_out) DCU(cudaEventRecord(end, s));
            if ((st = sync_state(hs, s)).rc) return st;
            if (hs->done) break;  // converged (FC:414)
        }
        if (host_out && !speculative_out) {
            if ((st = enqueue_output()).rc) return st;
            DCU(cudaEventRecord(end, s));
            DCU(cudaStreamSynchronize(s));
        }
    }
    DCU(cudaGetLastError());
    float ms = 0;
    if (cudaEventElapsedTime(&ms, ev0, end) == cudaSuccess) tm->total_ms = ms;
    tm->launches = launches;
    if (avg_error) memcpy(avg_error, &hs->avg_bits, sizeof *avg_error);
    if (iterations) *iterations = (int)hs->iters;
    return DecodeStatus{};
}

int decode_batch_group(const Geom &g)
{
    if (!decode_plan(g).one_launch) return 0;
    // the images of one launch stay L2-resident together, the budget sweep_interleaved gives one image (so at least 1)
    const int64_t per_image = (int64_t)g.C * ((int64_t)g.W * g.H + 2 * (int64_t)g.sw * g.sh);
    const int64_t n = ((int64_t)48 << 20) / per_image;
    return (int)(n < kDecodeBatchMax ? n : kDecodeBatchMax);
}

// Groups of `group` images through k_decode_small, then every image the one-launch decoder did not finish -- it bailed
// (its avgError needs the float sum replayed), the geometry has no one-launch form (group == 0) or the device cannot
// launch it cooperatively -- through decode_run, one image at a time: the path fic_decode takes.
DecodeStatus decode_batch_run(const Work &w, const Geom &g, int n, int group, const int32_t *qcodes, int32_t *argb_out,
                              uint8_t *planes_out, int max_iters, float *avg_error, int *iterations, void *h_stage,
                              void *h_scratch, cudaEvent_t ev0, cudaEvent_t end, fic_timings *tm, int *bad_image, cudaStream_t s)
{
    const size_t plane = (size_t)g.W * g.H, codes = (size_t)g.NR * code_stride(g);
    const float fwh = (float)(g.W * g.H);  // FC:413 (float)(width*height)
    int launches = 0;
    std::vector<char> redo((size_t)n, group == 0);
    const auto small = g.B == 8 ? (g.C == 1 ? launch_small<1, 8, true> : launch_small<3, 8, true>)
                                : (g.C == 1 ? launch_small<1, 16, true> : launch_small<3, 16, true>);
    const DecodeState *hs = (const DecodeState *)h_stage;
    for (int i0 = 0; group > 0 && i0 < n; i0 += group) {
        const int gn = n - i0 < group ? n - i0 : group;
        int32_t *dpos = (int32_t *)(w.dcode + (size_t)group * codes);
        float *d_carry = (float *)(w.state + group);
        DCU(cudaMemcpyAsync(w.q, qcodes + i0 * codes, sizeof(int32_t) * gn * codes, cudaMemcpyHostToDevice, s));
        DCU(cudaMemsetAsync(w.state, 0, sizeof(DecodeState) * gn, s));
        if (avg_error) DCU(cudaMemcpyAsync(d_carry, avg_error + i0, sizeof(float) * gn, cudaMemcpyHostToDevice, s));
        else DCU(cudaMemsetAsync(d_carry, 0, sizeof(float) * gn, s));
        if (!small(w, g, w.q, dpos, w.img, argb_out ? w.argb : nullptr, max_iters, 0.0f, fwh, s, (uint32_t)gn, d_carry)) {
            for (int i = i0; i < n; i++) redo[i] = 1;  // no cooperative launch on this device
            break;
        }
        launches++;
        DCU(cudaMemcpyAsync(h_stage, w.state, sizeof(DecodeState) * gn, cudaMemcpyDeviceToHost, s));
        if (argb_out) DCU(cudaMemcpyAsync(argb_out + i0 * plane, w.argb, sizeof(int32_t) * plane * gn, cudaMemcpyDeviceToHost, s));
        else DCU(cudaMemcpyAsync(planes_out + i0 * g.C * plane, w.img, g.C * plane * gn, cudaMemcpyDeviceToHost, s));
        DCU(cudaStreamSynchronize(s));
        for (int i = 0; i < gn; i++) {
            const DecodeState &x = hs[i];
            if (x.bad_index) {
                *bad_image = i0 + i;
                return DecodeStatus{FIC_E_STREAM};
            }
            if (x.bail) {
                redo[i0 + i] = 1;  // avg_error[i0 + i] still holds its carry
                continue;
            }
            if (avg_error) memcpy(avg_error + i0 + i, &x.avg_bits, sizeof(float));
            if (iterations) iterations[i0 + i] = (int)x.iters;
        }
    }
    for (int i = 0; i < n; i++) {
        if (!redo[i]) continue;
        DCU(cudaMemcpyAsync(w.q, qcodes + i * codes, sizeof(int32_t) * codes, cudaMemcpyHostToDevice, s));
        fic_timings one = {};
        const DecodeStatus st = decode_run(w, g, w.q, w.img, argb_out ? argb_out + i * plane : nullptr,
                                           planes_out ? planes_out + i * g.C * plane : nullptr, max_iters,
                                           avg_error ? avg_error + i : nullptr, iterations ? iterations + i : nullptr, h_scratch, ev0,
                                           end, &one, s);
        if (st.rc == FIC_E_STREAM) *bad_image = i;
        if (st.rc) return st;
        launches += one.launches;
    }
    DCU(cudaEventRecord(end, s));
    DCU(cudaStreamSynchronize(s));
    DCU(cudaGetLastError());
    float ms = 0;
    if (cudaEventElapsedTime(&ms, ev0, end) == cudaSuccess) tm->total_ms = ms;
    tm->launches = launches;
    return DecodeStatus{};
}

DecodeStatus collage_run(const Work &w, const Geom &g, int32_t *argb_out, float *info_out, void *h_scratch, cudaStream_t s)
{
    const Plan p = plain_plan(g);  // the source's codebook is the plain decimated plane of the pool builder
    const size_t plane = (size_t)g.W * g.H;
    const int S = code_stride(g);
    int32_t *doff = (int32_t *)(w.dcode + g.NR * S);
    DCU(cudaMemsetAsync(w.state, 0, sizeof(DecodeState), s));
    launch_dequant(nullptr, w.info, w.dcode, doff, g, false, w.state, s);  // FC:273 calculateIndices
    launch_fill(w.img, g.C * plane, 0xa0, s);                              // RasterImage.java:19,31
    (g.C == 1 ? launch_sweep<1> : launch_sweep<3>)(p, g, w.dec, w.img, nullptr, w.dcode, doff, SweepCtl{nullptr, 0, 0, 0.0f}, nullptr, false, s);
    launch_pack_argb(w.img, w.argb, g, s);
    DCU(cudaGetLastError());
    DCU(cudaMemcpyAsync(h_scratch, w.state, sizeof(DecodeState), cudaMemcpyDeviceToHost, s));
    DCU(cudaMemcpyAsync(argb_out, w.argb, sizeof(int32_t) * plane, cudaMemcpyDeviceToHost, s));
    DCU(cudaMemcpyAsync(info_out, w.dcode, sizeof(float) * g.NR * S, cudaMemcpyDeviceToHost, s));  // FC:888 in-place
    return sync_state((const DecodeState *)h_scratch, s);
}

DecodeStatus decode_float_sum(const Work &w, const int32_t *terms, int64_t count, float carry, void *h_scratch, float *sum,
                              cudaStream_t s)
{
    DecodeState state = {};
    for (int64_t i = 0; i < count; i++) state.sq_sum += (unsigned long long)terms[i];  // what a sweep leaves: the exact total
    DCU(cudaMemcpyAsync(w.perr, terms, sizeof(int32_t) * (size_t)count, cudaMemcpyHostToDevice, s));
    DCU(cudaMemcpyAsync(w.state, &state, sizeof state, cudaMemcpyHostToDevice, s));
    // "last sweep" keeps the value whatever it is; divided by 1 it is the sum itself
    launch_sweep_finish(w, count, 0, true, carry, 1.0f, s);
    DCU(cudaMemcpyAsync(h_scratch, w.state, sizeof(DecodeState), cudaMemcpyDeviceToHost, s));
    DCU(cudaStreamSynchronize(s));
    DCU(cudaGetLastError());
    memcpy(sum, &((const DecodeState *)h_scratch)->avg_bits, sizeof *sum);
    return DecodeStatus{};
}

}  // namespace fic
