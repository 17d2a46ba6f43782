// fic_quadtree.cu -- the quadtree extension (FIC_MODE_GREY_QT and FIC_MODE_RGB_QT, not in the reference): the stream's
// geometry and parser, and the kernels that turn every level's codes into the stream body on the device -- the collage
// error of each range block, the split flags of each top block, the leaf scan and the big-endian leaf scatter; for an
// encode to a byte budget, the keys and the per-image radix select that choose max_mse on the device.  The
// per-level encodes are the library's ordinary grey or RGB encodes (fic_encode.cu); the decoder sweep lives with the
// other sweeps in fic_decode.cu.  The kernels take the channel count C (1 grey, 3 RGB) as a template parameter.
#include <math.h>
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

// qt_err layout for a group of n images: [0] leaf total, [1] unused, [2, 2 + 2n) the budget form's max_mse of every
// image (doubles, so that they come down in the copy of the leaf total), then the per-top-block in-warp prefixes
// (n * flag_bytes words), the per-warp totals (n * qt_warps), then the collage errors of every level (level-major, then
// image-major: level L of image i at n * QtGeom::first[L] + i * NR_L).  An image's top blocks start a new warp, so its
// prefixes and warp totals are its own; one scan over every warp total of the group gives each image's first leaf at its
// first warp.
__host__ __device__ inline int64_t qt_warps(const QtGeom &q) { return (q.flag_bytes + 31) / 32; }
size_t qt_head_words(int n) { return 2 + 2 * (size_t)n; }
size_t qt_starts_at(const QtGeom &q, int n) { return qt_head_words(n) + n * q.flag_bytes; }
static int64_t qt_err_at(const QtGeom &q, int n) { return (int64_t)qt_starts_at(q, n) + n * qt_warps(q); }
size_t qt_err_words(const QtGeom &q, int n) { return (size_t)(qt_err_at(q, n) + n * q.codes); }
int64_t qt_nodes(const QtGeom &q) { return q.nl == 1 ? 0 : q.g[0].NR * (q.nl == 3 ? 5 : 1); }
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
__device__ __forceinline__ bool qt_split(const QtSplit &p, double max_mse, int L, int64_t j)
{
    return L < p.q.nl - 1 && (double)p.err[qt_at<BATCH>(p.q, L, j)] > __dmul_rn(max_mse, (double)(C * p.q.g[L].n));
}

// One thread per top block (and per padding byte of the flags): its flag byte into the stream, its leaf count's
// exclusive prefix within the warp to pre[t], the warp's total to wsum[warp].  BATCH: image blockIdx.y, whose stream body
// starts at flags + blockIdx.y * qt_body_pitch and whose prefixes and warp totals are its own (the qt_err layout).
// BUDGET: the image's max_mse is thr[image] (k_qt_select's), not p.max_mse.
template <int C, bool BATCH, bool BUDGET>
__global__ void __launch_bounds__(256) k_qt_decide(QtSplit p, uint8_t *__restrict__ flags, uint32_t *__restrict__ pre,
                                                   uint32_t *__restrict__ wsum, const double *__restrict__ thr)
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
        const double m = BUDGET ? thr[BATCH ? blockIdx.y : 0] : p.max_mse;
        if (qt_split<C, BATCH>(p, m, 0, t)) {
            f = 1;
            for (int k = 0; k < 4; k++)
                if (qt_split<C, BATCH>(p, m, 1, qt_child(p.q, 0, t, k))) f |= 2u << k;
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

// ---- device: the budget form's threshold ---------------------------------------------------------------------------------
// With N0 = C * b_max^2 and N_L = N0 / s_L^2, s_L = b_max / B_L a power of two, fl(m * N_L) * s_L^2 == fl(m * N0) for every
// double m (the scaling is exact; where fl(m * N_L) is subnormal or infinite both sides compare alike with the integer
// keys), so a node of level L splits at m iff fl(m * N0) < E * s_L^2, its key.  A level-1 node splits only if its parent
// does: its effective key is min(parent's key, own key), and the nodes that split at m are those with effective key >
// fl(m * N0).  Keys are below 3 * 255^2 * 256 < 2^26.

// One thread per top block: the effective keys of its split-capable nodes, the top block's at t, its four children's
// (when b_min is two levels down) at NR_top + 4t + k.  Image blockIdx.y's keys at keys + blockIdx.y * qt_nodes.
__global__ void __launch_bounds__(256) k_qt_keys(QtGeom q, const uint32_t *__restrict__ err, uint32_t *__restrict__ keys)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, ntop = q.g[0].NR;
    if (t >= ntop) return;
    keys += blockIdx.y * ntop * (q.nl == 3 ? 5 : 1);
    const uint32_t k0 = err[qt_at<true>(q, 0, t)];
    keys[t] = k0;
    if (q.nl == 3)
        for (int k = 0; k < 4; k++) keys[ntop + 4 * t + k] = min(k0, 4u * err[qt_at<true>(q, 1, qt_child(q, 0, t, k))]);
}

constexpr int kSelThreads = 1024, kSelDigit = 13, kSelBins = 1 << kSelDigit;

// Of the keys whose digit above `shift` equals `prefix`: the histogram of their 13-bit digit at `shift`, then the digit d
// holding the rank-r key counting from the largest (0-based), and r less the keys above d.  r must be below their count.
__device__ void qt_select_digit(const uint32_t *__restrict__ keys, int64_t nk, int shift, uint32_t prefix, uint32_t *hist,
                                uint32_t *part, uint32_t &digit, uint32_t &r)
{
    const int tid = threadIdx.x, lane = tid & 31;
    for (int b = tid; b < kSelBins; b += kSelThreads) hist[b] = 0;
    __syncthreads();
    for (int64_t j0 = tid - lane; j0 < nk; j0 += kSelThreads) {  // warp-uniform trips
        const int64_t j = j0 + lane;
        const uint32_t k = j < nk ? keys[j] : 0u;
        const bool in = j < nk && (k >> shift >> kSelDigit) == prefix;
        const uint32_t bin = in ? (k >> shift) & (kSelBins - 1) : kSelBins;
        const uint32_t peers = __match_any_sync(0xffffffffu, bin);  // flat images: many equal keys, one atomic
        if (in && lane == __ffs(peers) - 1) atomicAdd(&hist[bin], __popc(peers));
    }
    __syncthreads();
    // Thread tid owns the 8 bins below kSelBins - 8 * tid: a suffix count over threads finds the owner of rank r.
    constexpr int per = kSelBins / kSelThreads;
    const int top = kSelBins - 1 - per * tid;
    uint32_t own = 0;
    for (int b = 0; b < per; b++) own += hist[top - b];
    uint32_t incl = own;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) part[tid >> 5] = incl;
    __syncthreads();
    uint32_t before = 0;  // keys in the bins of lower-numbered threads (larger digits)
    for (int wi = 0; wi < (tid >> 5); wi++) before += part[wi];
    before += incl - own;
    const uint32_t want = r;
    __syncthreads();
    if (want >= before && want < before + own) {
        uint32_t c = before;
        for (int b = 0; b < per; b++) {
            const uint32_t hb = hist[top - b];
            if (want < c + hb) {
                part[32] = (uint32_t)(top - b);
                part[33] = want - c;
                break;
            }
            c += hb;
        }
    }
    __syncthreads();
    digit = part[32];
    r = part[33];
    __syncthreads();
}

// One CTA per image of the group: the image's max_mse m* = the smallest double with fl(m* * N0) >= v, v the (K+1)-th
// largest effective key (K = kq[image], the splits the budget allows), by a two-digit radix select over the keys; -inf
// when there are at most K keys; +0.0 when v == 0.  Into thr[image].
__global__ void __launch_bounds__(kSelThreads) k_qt_select(const uint32_t *__restrict__ keys, int64_t nk, const int64_t *__restrict__ kq,
                                                           double N0, double *__restrict__ thr)
{
    __shared__ uint32_t hist[kSelBins], part[34];
    const int i = blockIdx.x;
    const int64_t K = kq[i];
    if (K >= nk) {
        if (threadIdx.x == 0) thr[i] = -INFINITY;
        return;
    }
    keys += i * nk;
    uint32_t hi, lo, r = (uint32_t)K;
    qt_select_digit(keys, nk, kSelDigit, 0, hist, part, hi, r);
    qt_select_digit(keys, nk, 0, hi, hist, part, lo, r);
    if (threadIdx.x) return;
    const double v = (double)(hi << kSelDigit | lo);
    double m = 0.0;
    if (v > 0) {  // v / N0 is exact for grey (N0 a power of two); RGB's N0 = 3 * 4^k may need a step of an ulp
        m = __ddiv_rn(v, N0);  // positive: an ulp step is +-1 on its bits
        while (__dmul_rn(m, N0) < v) m = __longlong_as_double(__double_as_longlong(m) + 1);
        for (double d = __longlong_as_double(__double_as_longlong(m) - 1); __dmul_rn(d, N0) >= v;
             d = __longlong_as_double(__double_as_longlong(m) - 1))
            m = d;
    }
    thr[i] = m;
}

int64_t qt_budget_splits(const QtGeom &q, size_t max_bytes)
{
    const size_t leaf = qt_leaf_bytes(q), least = kQtHeaderBytes + (size_t)q.flag_bytes + leaf * (size_t)q.g[0].NR;
    if (max_bytes < least) return -1;
    const size_t k = (max_bytes - least) / (3 * leaf);
    return k > (size_t)INT64_MAX ? INT64_MAX : (int64_t)k;
}

template <int C, bool BATCH, bool BUDGET>
static int launch_qt_stream_c(const Work &w, const QtGeom &q, int n, double max_mse, cudaStream_t s)
{
    constexpr int S = C == 1 ? 3 : 5;
    uint32_t *total = w.qt_err, *pre = w.qt_err + qt_head_words(n), *wsum = pre + n * q.flag_bytes, *err = w.qt_err + qt_err_at(q, n);
    double *thr = (double *)(w.qt_err + 2);
    int launches = 0;
    for (int L = 0; L < q.nl; L++) {
        const Geom &g = q.g[L];
        const int64_t threads = g.NR * g.B;
        k_qt_collage_sse<C, BATCH><<<dim3((unsigned)((threads + 255) / 256), n), 256, 0, s>>>(w.src, w.dec, w.qt_codes + S * n * q.first[L],
                                                                                             err + n * q.first[L], g);
        launches++;
    }
    if (BUDGET) {
        const int64_t nk = qt_nodes(q);
        uint32_t *keys = (uint32_t *)(w.qt_keys + n);
        if (nk) k_qt_keys<<<dim3((unsigned)((q.g[0].NR + 255) / 256), n), 256, 0, s>>>(q, err, keys);
        k_qt_select<<<n, kSelThreads, 0, s>>>(keys, nk, w.qt_keys, (double)(C * q.g[0].n), thr);
        launches += 1 + (nk > 0);
    }
    const QtSplit p = {q, err, max_mse};
    k_qt_decide<C, BATCH, BUDGET><<<dim3((unsigned)((q.flag_bytes + 255) / 256), n), 256, 0, s>>>(p, w.qt_stream, pre, wsum, thr);
    launches += 1 + launch_scan_u32(wsum, n * qt_warps(q), total, s);
    k_qt_scatter<C, BATCH><<<dim3((unsigned)((q.g[0].NR + 255) / 256), n), 256, 0, s>>>(q, w.qt_codes, w.qt_stream, pre, wsum,
                                                                                       (uint32_t *)(w.qt_stream + q.flag_bytes));
    return launches + 1;
}

template <bool BUDGET>
static int launch_qt_stream_b(const Work &w, const QtGeom &q, int n, double max_mse, cudaStream_t s)
{
    if (n == 1)
        return q.g[0].C == 3 ? launch_qt_stream_c<3, false, BUDGET>(w, q, 1, max_mse, s) : launch_qt_stream_c<1, false, BUDGET>(w, q, 1, max_mse, s);
    return q.g[0].C == 3 ? launch_qt_stream_c<3, true, BUDGET>(w, q, n, max_mse, s) : launch_qt_stream_c<1, true, BUDGET>(w, q, n, max_mse, s);
}

int launch_qt_stream(const Work &w, const QtGeom &q, int n, double max_mse, bool budget, cudaStream_t s)
{
    return budget ? launch_qt_stream_b<true>(w, q, n, max_mse, s) : launch_qt_stream_b<false>(w, q, n, max_mse, s);
}

size_t qt_body_bytes(const QtGeom &q) { return (size_t)qt_body_pitch(q); }

}  // namespace fic
