/*
 * fic_oracle_quadtree_rgb.c -- CPU oracle of the RGB quadtree extension (TEST INFRASTRUCTURE ONLY, see
 * fic_oracle_quadtree_rgb.h).
 *
 * NOT IN THE REFERENCE: an RGB image on a quadtree of block sizes b_max, b_max/2, ..., b_min -- the grey quadtree of
 * fic_oracle_quadtree.c with the reference's RGB codes.  Every level is the reference's RGB encode at that blockgroesse
 * (fic_oracle_encode_rgb of fic_oracle.c, which this file is linked with), quantised as writeData does (FC:250-254);
 * the collage error sums over the three channels, with the domain pixels read from the source's RGB-decimated image
 * (fic_oracle_scale_image_rgb, FC:901-962), and a block above b_min splits iff E > max_mse * 3 * B^2.  The geometry
 * helpers below restate those of fic_oracle_quadtree.c (static there).  Same build rules as fic_oracle.c:
 * gcc -O2 -ffp-contract=off -fno-fast-math (Java float semantics: binary32, no fused multiply-add).
 */
#include "fic_oracle_quadtree_rgb.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "fic_oracle.h"

/* Java (int) of a float: truncate toward zero, saturate, NaN -> 0 (JLS 5.1.3). */
static int32_t j_f2i(float f)
{
    if (f != f) return 0;
    if (f >= 2147483648.0f) return INT32_MAX;
    if (f <= -2147483648.0f) return INT32_MIN;
    return (int32_t)f;
}

static inline int ch_r(int32_t p) { return (p >> 16) & 0xff; }
static inline int32_t pack(int r, int g, int b)
{
    return (int32_t)(0xff000000u | ((uint32_t)r << 16) | ((uint32_t)g << 8) | (uint32_t)b);
}
static int thresh(int v) { return v < 0 ? 0 : (v > 255 ? 255 : v); } /* FC:743-749 */

static void put_be32(uint8_t **p, int32_t v)
{
    (*p)[0] = (uint8_t)((uint32_t)v >> 24); (*p)[1] = (uint8_t)((uint32_t)v >> 16);
    (*p)[2] = (uint8_t)((uint32_t)v >> 8);  (*p)[3] = (uint8_t)v;
    *p += 4;
}

static int32_t get_be32(const uint8_t *p)
{
    return (int32_t)(((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]);
}

/* The argument sets on which the reference would fault (as fic_oracle.c rejects them). */
static int check_args(int W, int H, int B, int wk)
{
    if (B < 4 || (B & (B - 1))) return -1;
    if (W <= 0 || H <= 0 || W % B || H % B) return -2;
    int rpw = W / B, rph = H / B;
    if (rpw < 2 || rph < 2) return -3;
    int dpw = rpw * 2 - 3, dph = rph * 2 - 3;
    if (wk < 1 || wk > dpw || wk > dph) return -4;
    return 0;
}

static int qt_levels(int W, int H, int b_max, int b_min, int wk)
{
    if (!(b_max == 8 || b_max == 16) || !(b_min == 4 || b_min == 8 || b_min == 16) || b_min > b_max) return -1;
    if (W <= 0 || H <= 0 || W % b_max || H % b_max) return -2;
    if (wk < 0 || (wk == 0 && W != H)) return -4;
    int nl = 0;
    for (int B = b_max; B >= b_min; B /= 2, nl++) {
        int rc = check_args(W, H, B, wk ? wk : 2 * (W / B) - 3);
        if (rc) return rc;
    }
    return nl;
}

typedef struct {
    int nl, W, H, B[3], wk[3], rpw[3];
    const int32_t *codes[3];  /* [NR_L][5] */
    const long long *err[3];  /* [NR_L]    */
    double max_mse;
} qt_t;

static long qt_child(const qt_t *t, int L, long j, int k)
{
    long y = 2 * (j / t->rpw[L]) + (k >> 1), x = 2 * (j % t->rpw[L]) + (k & 1);
    return y * t->rpw[L + 1] + x;
}

static inline int ch_g(int32_t p) { return (p >> 8) & 0xff; }
static inline int ch_b(int32_t p) { return p & 0xff; }

size_t fic_oracle_quadtree_rgb_bound(int W, int H, int b_max, int b_min)
{
    long top = (long)(W / b_max) * (H / b_max);
    return 32 + (size_t)((top + 3) & ~3L) + 20 * (size_t)(W / b_min) * (size_t)(H / b_min);
}

/* Range block j of level geometry (W, H, B, wk): its RGB code {c, qa, qbR, qbG, qbB} -> codebook index
 * (calculate_indices, FC:853-893, float division and remainder), a = qa / 1e6f, b[] = {qbR / 1e5f, qbG / 1e5f, qbB}
 * (FC:446-450: blue is not scaled).  Returns the index, or -1 outside the pool. */
static long qt_dequant_rgb(int W, int H, int B, int wk, long j, const int32_t *code, float *a, float b[3])
{
    float c = (float)code[0];
    int rpw = W / B, rph = H / B, dpw = rpw * 2 - 3, dph = rph * 2 - 3;
    int x = (int)(j % rpw) * B, y = (int)(j / rpw) * B;
    int di = fic_oracle_domain_block_index(x, y, rpw, rph, dpw, B);
    int dy, dx;
    fic_oracle_generate_kernel(dpw, dph, di, wk, &dy, &dx);
    int yd = j_f2i(c / (float)wk);
    int xd = j_f2i(fmodf(c, (float)wk));
    long idx = (long)xd + dx + (long)(yd + dy) * dpw;
    *a = (float)code[1] / 1000000.0f;
    b[0] = (float)code[2] / 100000.0f;
    b[1] = (float)code[3] / 100000.0f;
    b[2] = (float)code[4];
    return idx < 0 || idx >= (long)dpw * dph ? -1 : idx;
}

/* thresh((int)(a * d + b)) of each channel of the packed pixel d, packed. */
static int32_t qt_px_rgb(float a, const float b[3], int32_t d)
{
    return pack(thresh(j_f2i(a * (float)ch_r(d) + b[0])), thresh(j_f2i(a * (float)ch_g(d) + b[1])),
                thresh(j_f2i(a * (float)ch_b(d) + b[2])));
}

static long long sq_rgb(int32_t p, int32_t q)
{
    long long dr = ch_r(p) - ch_r(q), dg = ch_g(p) - ch_g(q), db = ch_b(p) - ch_b(q);
    return dr * dr + dg * dg + db * db;
}

static long long qt_block_sse_rgb(const int32_t *img, const int32_t *dec, int W, int B, int wk_l, int H, long j,
                                  const int32_t *code, int *bad)
{
    float a, b[3];
    long idx = qt_dequant_rgb(W, H, B, wk_l, j, code, &a, b);
    if (idx < 0) { *bad = 1; return 0; }
    int sw = W / 2, rpw = W / B, dpw = rpw * 2 - 3, step = B / 4;
    int drow = (int)(idx / dpw) * step, dcol = (int)(idx % dpw) * step;
    int x = (int)(j % rpw) * B, y = (int)(j / rpw) * B;
    long long e = 0;
    for (int ry = 0; ry < B; ry++)
        for (int rx = 0; rx < B; rx++)
            e += sq_rgb(qt_px_rgb(a, b, dec[dcol + rx + (drow + ry) * sw]), img[x + rx + (y + ry) * W]);
    return e;
}

static int qt_split_rgb(const qt_t *t, int L, long j)
{
    return L < t->nl - 1 && (double)t->err[L][j] > t->max_mse * (double)(3 * t->B[L] * t->B[L]);
}

static void qt_emit_rgb(const qt_t *t, int L, long j, uint8_t **p, long *n)
{
    if (qt_split_rgb(t, L, j)) {
        for (int k = 0; k < 4; k++) qt_emit_rgb(t, L + 1, qt_child(t, L, j, k), p, n);
        return;
    }
    const int32_t *c = t->codes[L] + 5 * j;
    for (int k = 0; k < 5; k++) put_be32(p, c[k]);
    (*n)++;
}

int fic_oracle_encode_quadtree_rgb(const int32_t *argb, int W, int H, int b_max, int b_min, int wk, double max_mse,
                                   int nthreads, uint8_t *out, size_t *nbytes)
{
    int nl = qt_levels(W, H, b_max, b_min, wk);
    if (nl < 0) return nl;
    if (max_mse != max_mse) return -1;
    qt_t t = {0};
    t.nl = nl; t.W = W; t.H = H; t.max_mse = max_mse;
    int32_t *dec = (int32_t *)malloc(sizeof(int32_t) * (size_t)(W / 2) * (H / 2));
    fic_oracle_scale_image_rgb(argb, W, H, dec); /* every level's codebook is cut from this image */
    int rc = 0, bad = 0;
    for (int L = 0; L < nl && !rc; L++) {
        int B = b_max >> L, wkl = wk ? wk : 2 * (W / B) - 3;
        long nr = (long)(W / B) * (H / B);
        t.B[L] = B; t.wk[L] = wkl; t.rpw[L] = W / B;
        float *info = (float *)malloc(sizeof(float) * 5 * (size_t)nr);
        int32_t *q = (int32_t *)malloc(sizeof(int32_t) * 5 * (size_t)nr);
        long long *e = (long long *)malloc(sizeof(long long) * (size_t)nr);
        rc = fic_oracle_encode_rgb(argb, W, H, B, wkl, 0, nr, nthreads, info);
        for (long j = 0; j < nr && !rc; j++) { /* FC:250-254 */
            q[5 * j] = j_f2i(info[5 * j]);
            q[5 * j + 1] = j_f2i(info[5 * j + 1] * 1000000);
            q[5 * j + 2] = j_f2i(info[5 * j + 2] * 100000);
            q[5 * j + 3] = j_f2i(info[5 * j + 3] * 100000);
            q[5 * j + 4] = j_f2i(info[5 * j + 4]);
            e[j] = qt_block_sse_rgb(argb, dec, W, B, wkl, H, j, q + 5 * j, &bad);
        }
        free(info);
        t.codes[L] = q;
        t.err[L] = e;
    }
    if (!rc && bad) rc = -8;
    if (!rc) {
        long ntop = (long)(W / b_max) * (H / b_max), pad = (ntop + 3) & ~3L, n = 0;
        uint8_t *p = out + 32 + pad;
        memset(out + 32, 0, (size_t)pad);
        for (long j = 0; j < ntop; j++) {
            uint8_t f = 0;
            if (qt_split_rgb(&t, 0, j)) {
                f = 1;
                for (int k = 0; k < 4; k++)
                    if (qt_split_rgb(&t, 1, qt_child(&t, 0, j, k))) f |= (uint8_t)(2 << k);
            }
            out[32 + j] = f;
            qt_emit_rgb(&t, 0, j, &p, &n);
        }
        uint8_t *h = out;
        put_be32(&h, 4); put_be32(&h, W); put_be32(&h, H); put_be32(&h, 0);
        put_be32(&h, wk); put_be32(&h, b_max); put_be32(&h, b_min); put_be32(&h, (int32_t)n);
        *nbytes = (size_t)(p - out);
    }
    for (int L = 0; L < nl; L++) { free((void *)t.codes[L]); free((void *)t.err[L]); }
    free(dec);
    return rc;
}

int fic_oracle_decode_quadtree_rgb(const uint8_t *s, size_t nbytes, int max_iters, int32_t *out, float *avg_error,
                                   int *iters)
{
    if (nbytes < 32 || max_iters < 1) return -7;
    int W = get_be32(s + 4), H = get_be32(s + 8), wk = get_be32(s + 16);
    int b_max = get_be32(s + 20), b_min = get_be32(s + 24), n_leaves = get_be32(s + 28);
    if (get_be32(s) != 4 || get_be32(s + 12) != 0) return -7;
    int nl = qt_levels(W, H, b_max, b_min, wk);
    if (nl < 0) return nl;
    long ntop = (long)(W / b_max) * (H / b_max), pad = (ntop + 3) & ~3L, n = 0;
    if (nbytes < 32 + (size_t)pad) return -7;
    for (long j = 0; j < ntop; j++) {
        int f = s[32 + j];
        int allowed = nl == 1 ? 0 : ((nl == 2 || !(f & 1)) ? 1 : 0x1f);
        if (f & ~allowed) return -7;
        if (!(f & 1)) n += 1;
        else for (int k = 0; k < 4; k++) n += (f >> (1 + k)) & 1 ? 4 : 1;
    }
    if (n != n_leaves || nbytes < 32 + (size_t)pad + 20 * (size_t)n) return -7;
    typedef struct { int B, x, y, drow, dcol; float a, b[3]; } leaf_t;
    leaf_t *lf = (leaf_t *)malloc(sizeof(leaf_t) * (size_t)(n ? n : 1));
    const uint8_t *p = s + 32 + pad;
    long k = 0;
    int rc = 0;
    for (long t = 0; t < ntop && !rc; t++) {
        int f = s[32 + t];
        long list_j[16];
        int list_l[16], m = 0;
        if (!(f & 1)) { list_l[m] = 0; list_j[m++] = t; }
        else {
            int rpw0 = W / b_max, rpw1 = W / (b_max / 2), rpw2 = W / (b_max / 4);
            for (int c = 0; c < 4; c++) {
                long j1 = (2 * (t / rpw0) + (c >> 1)) * rpw1 + 2 * (t % rpw0) + (c & 1);
                if (!((f >> (1 + c)) & 1)) { list_l[m] = 1; list_j[m++] = j1; continue; }
                for (int c2 = 0; c2 < 4; c2++) {
                    list_l[m] = 2;
                    list_j[m++] = (2 * (j1 / rpw1) + (c2 >> 1)) * rpw2 + 2 * (j1 % rpw1) + (c2 & 1);
                }
            }
        }
        for (int i = 0; i < m; i++, k++, p += 20) {
            int B = b_max >> list_l[i], wkl = wk ? wk : 2 * (W / B) - 3, dpw = 2 * (W / B) - 3;
            int32_t code[5] = {get_be32(p), get_be32(p + 4), get_be32(p + 8), get_be32(p + 12), get_be32(p + 16)};
            long idx = qt_dequant_rgb(W, H, B, wkl, list_j[i], code, &lf[k].a, lf[k].b);
            if (idx < 0) { rc = -2; break; }
            lf[k].B = B;
            lf[k].x = (int)(list_j[i] % (W / B)) * B;
            lf[k].y = (int)(list_j[i] / (W / B)) * B;
            lf[k].drow = (int)(idx / dpw) * (B / 4);
            lf[k].dcol = (int)(idx % dpw) * (B / 4);
        }
    }
    int32_t *dec = (int32_t *)malloc(sizeof(int32_t) * (size_t)(W / 2) * (H / 2));
    int sw = W / 2, done = 0;
    float avg = 0;
    for (long q = 0; q < (long)W * H; q++) out[q] = pack(128, 128, 128); /* FC:1142-1148 */
    for (int it = 0; it < max_iters && !rc; it++) {
        fic_oracle_scale_image_rgb(out, W, H, dec);
        unsigned long long S = 0;
        for (long i = 0; i < n; i++)
            for (int ry = 0; ry < lf[i].B; ry++)
                for (int rx = 0; rx < lf[i].B; rx++) {
                    int32_t *px = &out[lf[i].x + rx + (lf[i].y + ry) * W];
                    int32_t v = qt_px_rgb(lf[i].a, lf[i].b, dec[lf[i].dcol + rx + (lf[i].drow + ry) * sw]);
                    S += (unsigned long long)sq_rgb(*px, v);
                    *px = v;
                }
        done = it + 1;
        avg = (float)S / (float)(W * H);
        if (avg < 1) break;
    }
    free(dec);
    free(lf);
    if (rc) return rc;
    if (avg_error) *avg_error = avg;
    if (iters) *iters = done;
    return 0;
}
