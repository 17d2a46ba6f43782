// fic_quadtree.cu -- the quadtree extension (FIC_MODE_GREY_QT and FIC_MODE_RGB_QT, not in the reference): the stream's
// geometry and parser, and the kernels that turn every level's codes into the stream body on the device -- the collage
// error of each range block, the split flags of each top block, the leaf scan and the big-endian leaf scatter.  The
// per-level encodes are the library's ordinary grey or RGB encodes (fic_encode.cu); the decoder sweep lives with the
// other sweeps in fic_decode.cu.  The kernels take the channel count C (1 grey, 3 RGB) as a template parameter.
#include <string.h>

#include "fic_device.cuh"

namespace fic {

// ---- host: geometry and parser -----------------------------------------------------------------------------------------

int qt_geom(int mode, int W, int H, int b_max, int b_min, int wk, QtGeom *q, const char **why)
{
    if (mode != FIC_MODE_GREY_QT && mode != FIC_MODE_RGB_QT) { *why = "mode must be FIC_MODE_GREY_QT or FIC_MODE_RGB_QT"; return FIC_E_ARG; }
    if (!(b_max == 8 || b_max == 16)) { *why = "b_max must be 8 or 16"; return FIC_E_ARG; }
    if (!(b_min == 4 || b_min == 8 || b_min == 16) || b_min > b_max) { *why = "b_min must be 4, 8 or 16 and at most b_max"; return FIC_E_ARG; }
    if (W <= 0 || H <= 0 || W % b_max || H % b_max) { *why = "width and height must be positive multiples of b_max"; return FIC_E_ARG; }
    if (wk < 0 || (wk == 0 && W != H)) { *why = "widthKernel must be >= 1, or 0 (every level's whole pool) on a square image"; return FIC_E_ARG; }
    memset(q, 0, sizeof *q);
    q->wk = wk;
    for (int B = b_max; B >= b_min; B /= 2) {
        const int L = q->nl++;
        const int wk_l = wk ? wk : 2 * (W / B) - 3;  // the whole pool: domain blocks per width (== per height)
        const int rc = make_geom(W, H, B, wk_l, mode == FIC_MODE_RGB_QT ? FIC_MODE_RGB : FIC_MODE_GREY, &q->g[L], why);
        if (rc) return rc;
        q->first[L] = q->codes;
        q->codes += q->g[L].NR;
    }
    q->flag_bytes = (q->g[0].NR + 3) & ~(int64_t)3;
    return FIC_OK;
}

static int32_t be32(const uint8_t *p)
{
    return (int32_t)(((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3]);
}

size_t qt_leaf_bytes(const QtGeom &q) { return q.g[0].C == 3 ? 20 : 12; }

size_t qt_stream_bound(int mode, int W, int H, int b_max, int b_min)
{
    if (b_max <= 0 || b_min <= 0 || W <= 0 || H <= 0) return 0;
    const size_t top = (size_t)(W / b_max) * (size_t)(H / b_max), leaf = mode == FIC_MODE_RGB_QT ? 20 : 12;
    return kQtHeaderBytes + ((top + 3) & ~(size_t)3) + leaf * (size_t)(W / b_min) * (size_t)(H / b_min);
}

int qt_parse(int mode, const uint8_t *s, size_t nbytes, QtGeom *q, int32_t *base, bool check_leaves, const char **why)
{
    if (!s || nbytes < kQtHeaderBytes) { *why = "stream shorter than its 32-byte header"; return FIC_E_STREAM; }
    int32_t hd[8];
    for (int k = 0; k < 8; k++) hd[k] = be32(s + 4 * k);
    if (hd[0] != mode || hd[3] != 0) {
        *why = mode == FIC_MODE_RGB_QT ? "not an RGB quadtree stream (header 4, W, H, 0, ...)" : "not a grey quadtree stream (header 3, W, H, 0, ...)";
        return FIC_E_STREAM;
    }
    if (qt_geom(mode, hd[1], hd[2], hd[5], hd[6], hd[4], q, why)) return FIC_E_STREAM;
    const int64_t ntop = q->g[0].NR;
    if ((uint64_t)(nbytes - kQtHeaderBytes) < (uint64_t)q->flag_bytes) { *why = "stream truncated inside its split flags"; return FIC_E_STREAM; }
    const uint8_t *flags = s + kQtHeaderBytes;
    int64_t leaves = 0;
    for (int64_t t = 0; t < ntop; t++) {
        if (!qt_flags_legal(*q, flags[t])) { *why = "a split flag is set where no split is possible"; return FIC_E_STREAM; }
        if (base) base[t] = (int32_t)leaves;
        leaves += qt_leaf_count(flags[t]);
    }
    if (hd[7] != leaves) { *why = "n_leaves disagrees with the split flags"; return FIC_E_STREAM; }
    q->leaves = leaves;
    const size_t leaf_bytes = qt_leaf_bytes(*q);
    if ((uint64_t)(nbytes - kQtHeaderBytes - q->flag_bytes) / leaf_bytes < (uint64_t)leaves) { *why = "stream truncated inside its leaves"; return FIC_E_STREAM; }
    if (check_leaves) {
        const uint8_t *p = flags + q->flag_bytes;
        bool ok = true;
        for (int64_t t = 0; t < ntop && ok; t++)
            qt_visit_leaves(*q, t, flags[t], [&](int L, int64_t j) {
                ok = ok && code_pool_index(q->g[L], j, (float)be32(p)) >= 0;
                p += leaf_bytes;
            });
        if (!ok) { *why = "a leaf indexes outside its level's domain pool"; return FIC_E_STREAM; }
    }
    return FIC_OK;
}

// ---- device: collage error, split flags, leaf scatter --------------------------------------------------------------------

// qt_err layout for a group of n images: [0] leaf total, then the per-top-block in-warp prefixes (n * flag_bytes words),
// the per-warp totals (n * qt_warps), then the collage errors of every level (level-major, then image-major: level L of
// image i at n * QtGeom::first[L] + i * NR_L).  An image's top blocks start a new warp, so its prefixes and warp totals
// are its own; one scan over every warp total of the group gives each image's first leaf at its first warp.
__host__ __device__ inline int64_t qt_warps(const QtGeom &q) { return (q.flag_bytes + 31) / 32; }
static int64_t qt_err_at(const QtGeom &q, int n) { return 1 + n * (q.flag_bytes + qt_warps(q)); }
size_t qt_err_words(const QtGeom &q, int n) { return (size_t)(qt_err_at(q, n) + n * q.codes); }
__host__ __device__ inline int64_t qt_body_pitch(const QtGeom &q) { return q.flag_bytes + (q.g[0].C == 3 ? 20 : 12) * q.g[q.nl - 1].NR; }

// E(j) = sum over range block j (and its C channels) of (decode_px(a, b_c, d_c) - s_c)^2: the code dequantised as the
// decoder does (FC:372-374 grey, FC:446-450 RGB), the domain pixels d_c read from the source's decimated planes at the
// code's codebook index (FC:853-893).  B threads per range block, one row each (B divides 32: a block's rows share a warp
// and reduce with shuffles).  E < 2^32: at most 3 * 255^2 * 256.  BATCH: image blockIdx.y of a group -- its planes, and
// its rows of the level's [n][NR] code and error tables.
template <int C, bool BATCH>
__global__ void __launch_bounds__(256) k_qt_collage_sse(const uint8_t *__restrict__ src, const uint8_t *__restrict__ dec,
                                                        const int32_t *__restrict__ q, uint32_t *__restrict__ err, Geom g)
{
    if (BATCH) {
        const int64_t i = blockIdx.y;
        src += i * C * (int64_t)g.W * g.H;
        dec += i * C * (int64_t)g.sw * g.sh;
        q += i * (C == 1 ? 3 : 5) * g.NR;
        err += i * g.NR;
    }
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int B = g.B;
    const int64_t j = t / B;
    const int ry = (int)(t - j * B);
    uint32_t e = 0;
    if (j < g.NR) {
        const int32_t *c = q + (C == 1 ? 3 : 5) * j;
        const float a = __fdiv_rn((float)c[1], C == 1 ? kGreyAScale : kRgbAScale), b = (float)c[2];
        int64_t idx = code_pool_index(g, j, (float)c[0]);
        if (idx < 0) idx = 0;  // an encoder's code is always inside the pool
        const int x = (int)(j % g.rpw) * B, y = (int)(j / g.rpw) * B;
        const uint8_t *d = dec + (int64_t)((int)(idx / g.dpw) * g.step + ry) * g.sw + (int)(idx % g.dpw) * g.step;
        const uint8_t *s = src + (int64_t)(y + ry) * g.W + x;
#pragma unroll
        for (int ch = 0; ch < C; ch++) {
            // grey b = qb; RGB bR = qbR / 1e5f, bG = qbG / 1e5f, bB = qbB (unscaled, FC:450)
            const float bc = C == 1 ? b : (ch == 2 ? (float)c[4] : __fdiv_rn((float)c[2 + ch], kRgbBScale));
            const uint8_t *dc = d + (int64_t)ch * g.sw * g.sh, *sc = s + (int64_t)ch * g.W * g.H;
            for (int rx = 0; rx < B; rx++) {
                const int v = (int)decode_px(a, bc, dc[rx]) - (int)sc[rx];
                e += (uint32_t)(v * v);
            }
        }
    }
    for (int o = B / 2; o > 0; o >>= 1) e += __shfl_down_sync(0xffffffffu, e, o, B);
    if (j < g.NR && ry == 0) err[j] = e;
}

struct QtSplit {
    QtGeom q;
    const uint32_t *err;  // level-major collage errors
    double max_mse;
};

// Where range j of level L of the CTA's image sits in the level-major tables (BATCH: image blockIdx.y of gridDim.y).
template <bool BATCH>
__device__ __forceinline__ int64_t qt_at(const QtGeom &q, int L, int64_t j)
{
    return BATCH ? (int64_t)gridDim.y * q.first[L] + (int64_t)blockIdx.y * q.g[L].NR + j : q.first[L] + j;
}

// A block above b_min is split iff (double)E > max_mse * (double)(C * B * B).  BATCH: of the CTA's image.
template <int C, bool BATCH>
__device__ __forceinline__ bool qt_split(const QtSplit &p, int L, int64_t j)
{
    return L < p.q.nl - 1 && (double)p.err[qt_at<BATCH>(p.q, L, j)] > __dmul_rn(p.max_mse, (double)(C * p.q.g[L].n));
}

// One thread per top block (and per padding byte of the flags): its flag byte into the stream, its leaf count's
// exclusive prefix within the warp to pre[t], the warp's total to wsum[warp].  BATCH: image blockIdx.y, whose stream body
// starts at flags + blockIdx.y * qt_body_pitch and whose prefixes and warp totals are its own (the qt_err layout).
template <int C, bool BATCH>
__global__ void __launch_bounds__(256) k_qt_decide(QtSplit p, uint8_t *__restrict__ flags, uint32_t *__restrict__ pre,
                                                   uint32_t *__restrict__ wsum)
{
    if (BATCH) {
        flags += blockIdx.y * qt_body_pitch(p.q);
        pre += blockIdx.y * p.q.flag_bytes;
        wsum += blockIdx.y * qt_warps(p.q);
    }
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    uint32_t n = 0, f = 0;
    if (t < p.q.g[0].NR) {
        if (qt_split<C, BATCH>(p, 0, t)) {
            f = 1;
            for (int k = 0; k < 4; k++)
                if (qt_split<C, BATCH>(p, 1, qt_child(p.q, 0, t, k))) f |= 2u << k;
        }
        n = (uint32_t)qt_leaf_count(f);
    }
    uint32_t incl = n;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (t < p.q.flag_bytes) {
        flags[t] = (uint8_t)f;
        pre[t] = incl - n;
        if (lane == 31 || t == p.q.flag_bytes - 1) wsum[t >> 5] = incl;
    }
}

__device__ __forceinline__ uint32_t bswap32(int32_t v) { return __byte_perm((uint32_t)v, 0u, 0x0123); }

// One thread per top block: its leaves' codes (3 ints grey, 5 RGB), big endian (DataOutputStream.writeInt), at their
// place in the stream.  BATCH: image blockIdx.y, its leaves after its own flag bytes, counted from its first leaf.
template <int C, bool BATCH>
__global__ void __launch_bounds__(256) k_qt_scatter(QtGeom q, const int32_t *__restrict__ codes, const uint8_t *__restrict__ flags,
                                                    const uint32_t *__restrict__ pre, const uint32_t *__restrict__ wsum,
                                                    uint32_t *__restrict__ leaves)
{
    constexpr int S = C == 1 ? 3 : 5;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= q.g[0].NR) return;
    uint32_t first = 0;
    if (BATCH) {
        const int64_t body = blockIdx.y * qt_body_pitch(q);
        flags += body;
        leaves += body / 4;
        pre += blockIdx.y * q.flag_bytes;
        wsum += blockIdx.y * qt_warps(q);
        first = wsum[0];
    }
    uint32_t *o = leaves + S * (int64_t)(wsum[t >> 5] + pre[t] - first);
    qt_visit_leaves(q, t, flags[t], [&](int L, int64_t j) {
        const int32_t *c = codes + S * qt_at<BATCH>(q, L, j);
        o[0] = bswap32(c[0]);
        o[1] = bswap32(c[1]);
        o[2] = bswap32(c[2]);
        if (C == 3) {
            o[3] = bswap32(c[3]);
            o[4] = bswap32(c[4]);
        }
        o += S;
    });
}

template <int C, bool BATCH>
static int launch_qt_stream_c(const Work &w, const QtGeom &q, int n, double max_mse, cudaStream_t s)
{
    constexpr int S = C == 1 ? 3 : 5;
    uint32_t *total = w.qt_err, *pre = w.qt_err + 1, *wsum = pre + n * q.flag_bytes, *err = w.qt_err + qt_err_at(q, n);
    int launches = 0;
    for (int L = 0; L < q.nl; L++) {
        const Geom &g = q.g[L];
        const int64_t threads = g.NR * g.B;
        k_qt_collage_sse<C, BATCH><<<dim3((unsigned)((threads + 255) / 256), n), 256, 0, s>>>(w.src, w.dec, w.qt_codes + S * n * q.first[L],
                                                                                             err + n * q.first[L], g);
        launches++;
    }
    const QtSplit p = {q, err, max_mse};
    k_qt_decide<C, BATCH><<<dim3((unsigned)((q.flag_bytes + 255) / 256), n), 256, 0, s>>>(p, w.qt_stream, pre, wsum);
    launches += 1 + launch_scan_u32(wsum, n * qt_warps(q), total, s);
    k_qt_scatter<C, BATCH><<<dim3((unsigned)((q.g[0].NR + 255) / 256), n), 256, 0, s>>>(q, w.qt_codes, w.qt_stream, pre, wsum,
                                                                                       (uint32_t *)(w.qt_stream + q.flag_bytes));
    return launches + 1;
}

int launch_qt_stream(const Work &w, const QtGeom &q, int n, double max_mse, cudaStream_t s)
{
    if (n == 1) return q.g[0].C == 3 ? launch_qt_stream_c<3, false>(w, q, 1, max_mse, s) : launch_qt_stream_c<1, false>(w, q, 1, max_mse, s);
    return q.g[0].C == 3 ? launch_qt_stream_c<3, true>(w, q, n, max_mse, s) : launch_qt_stream_c<1, true>(w, q, n, max_mse, s);
}

size_t qt_body_bytes(const QtGeom &q) { return (size_t)qt_body_pitch(q); }

}  // namespace fic
