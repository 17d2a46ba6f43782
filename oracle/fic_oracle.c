/*
 * fic_oracle.c -- CPU oracle (TEST INFRASTRUCTURE ONLY, see fic_oracle.h).
 *
 * Plain-C restatement of the reference's encode/decode path.  Every function names
 * the reference lines it follows (FC = src/bvk_ss19/FractalCompression.java,
 * DB = src/bvk_ss19/Domainblock.java).  The arithmetic is kept in the reference's
 * types and order: Java `float` is IEEE binary32 with no fused multiply-add and no
 * extended intermediates, so this file must be built with
 *     gcc -O2 -ffp-contract=off -fno-fast-math      (see oracle/Makefile)
 * on x86-64 (SSE arithmetic, FLT_EVAL_METHOD == 0).
 *
 * Parity status: pinned by unknown.run (RGB path, byte exact) and the Animation.gif
 * avgError labels (grey path), see tests/test_oracle_golden.py.
 */
#include "fic_oracle.h"

#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------ Java casts */

/* Java (int) of a float: truncate toward zero, saturate, NaN -> 0 (JLS 5.1.3). */
static int32_t j_f2i(float f)
{
    if (f != f) return 0;
    if (f >= 2147483648.0f) return INT32_MAX;
    if (f <= -2147483648.0f) return INT32_MIN;
    return (int32_t)f;
}

static inline int ch_r(int32_t p) { return (p >> 16) & 0xff; }
static inline int ch_g(int32_t p) { return (p >> 8) & 0xff; }
static inline int ch_b(int32_t p) { return p & 0xff; }
static inline int32_t pack(int r, int g, int b)
{
    return (int32_t)(0xff000000u | ((uint32_t)r << 16) | ((uint32_t)g << 8) | (uint32_t)b);
}

/* ------------------------------------------------------------------ domain block */

/* DB:5-20: one codebook entry. */
typedef struct {
    const int32_t *argb;            /* B*B values: grey level, or packed ARGB (RGB path) */
    float variance;                 /* DB:9   (stays 0 on the RGB path, DB:30-41)         */
    int mittelWert;                 /* DB:10  */
    int mittelWertR, mittelWertG, mittelWertB;
    float varianceR, varianceG, varianceB;
} dblock_t;

/* DB:92-98 (and FC:67-73): integer mean, truncating division. */
static int mittelwert(const int *v, int n)
{
    int sum = 0;
    for (int i = 0; i < n; i++) sum += v[i];
    return sum / n;
}

/* DB:106-115: float accumulation of (v - mean)^2 in source order. */
static float varianz(int mw, const int *v, int n)
{
    float acc = 0;
    for (int i = 0; i < n; i++) {
        float g = (float)(v[i] - mw);
        acc += g * g;
    }
    return acc;
}

/* DB:23-42. `tmp` is scratch for one channel (n ints). */
static void dblock_init(dblock_t *d, const int32_t *argb, int n, int is_rgb, int *tmp)
{
    memset(d, 0, sizeof *d);
    d->argb = argb;
    if (!is_rgb) {
        d->mittelWert = mittelwert((const int *)argb, n);
        d->variance = varianz(d->mittelWert, (const int *)argb, n);
    } else {
        /* DB:31: mean of the packed ints (int overflow wraps as in Java); never used. */
        int32_t s = 0;
        for (int i = 0; i < n; i++) s = (int32_t)((uint32_t)s + (uint32_t)argb[i]);
        d->mittelWert = s / n;
        for (int i = 0; i < n; i++) tmp[i] = ch_r(argb[i]);
        d->mittelWertR = mittelwert(tmp, n);
        d->varianceR = varianz(d->mittelWertR, tmp, n);
        for (int i = 0; i < n; i++) tmp[i] = ch_g(argb[i]);
        d->mittelWertG = mittelwert(tmp, n);
        d->varianceG = varianz(d->mittelWertG, tmp, n);
        for (int i = 0; i < n; i++) tmp[i] = ch_b(argb[i]);
        d->mittelWertB = mittelwert(tmp, n);
        d->varianceB = varianz(d->mittelWertB, tmp, n);
    }
}

/* ------------------------------------------------------------------ geometry */

/* FC:516-545 getDomainBlockIndex. */
int fic_oracle_domain_block_index(int x, int y, int rpw, int rph, int dpw, int B)
{
    int xr = x / B, yr = y / B, i = 0;
    if (yr == 0) yr = 1;
    if (xr == 0) xr = 1;
    if (yr == rph - 1) yr = yr - 1;
    if (xr == rpw - 1) xr = xr - 1;
    if (xr > 1) {
        if (yr == 0) i = xr;
        else i = (xr * 2) - 2 + (yr + yr - 1) * dpw;
    } else if (xr == 1) {
        if (yr == 0) i = xr;
        else i = xr + (yr + yr - 1) * dpw;
    }
    return i;
}

/* FC:84-100 generateKernel (duplicated at FC:868-879). */
void fic_oracle_generate_kernel(int dpw, int dph, int index, int wk, int *dy, int *dx)
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

/* ------------------------------------------------------------------ decimation */

/* FC:970-1007 scaleImage: red channel, 2x2 box, /4 truncating; border quirks kept
 * (FC:993 compares x+1 against image.height). */
void fic_oracle_scale_image(const int32_t *a, int W, int H, int32_t *dst)
{
    int i = 0;
    for (int y = 0; y < H; y += 2) {
        for (int x = 0; x < W; x += 2) {
            int m = ch_r(a[x + y * W]);
            if (x + 1 >= W) {
                m += 128;
            } else {
                m += ch_r(a[x + 1 + y * W]);
                if (y + 1 >= H) m += 128;
                else m += ch_r(a[x + (y + 1) * W]);
            }
            if (y + 1 >= H) m += 128;
            else {
                if (x + 1 >= H) m += 128;
                else m += ch_r(a[x + 1 + (y + 1) * W]);
            }
            m = m / 4;
            dst[i++] = pack(m, m, m);
        }
    }
}

/* FC:901-962 scaleImageRGB: the fourth tap re-reads (x, y+1) (FC:945-947), so the
 * average is (p00 + p10 + 2*p01)/4 per channel. */
void fic_oracle_scale_image_rgb(const int32_t *a, int W, int H, int32_t *dst)
{
    int i = 0;
    for (int y = 0; y < H; y += 2) {
        for (int x = 0; x < W; x += 2) {
            int r = ch_r(a[x + y * W]), g = ch_g(a[x + y * W]), b = ch_b(a[x + y * W]);
            if (x + 1 >= W) {
                r += 128; g += 128; b += 128;
            } else {
                int32_t p = a[x + 1 + y * W];
                r += ch_r(p); g += ch_g(p); b += ch_b(p);
                if (y + 1 >= H) {
                    r += 128; g += 128; b += 128;
                } else {
                    p = a[x + (y + 1) * W];
                    r += ch_r(p); g += ch_g(p); b += ch_b(p);
                }
            }
            if (y + 1 >= H) {
                r += 128; g += 128; b += 128;
            } else {
                if (x + 1 >= H) {
                    r += 128; g += 128; b += 128;
                } else {
                    int32_t p = a[x + (y + 1) * W];
                    r += ch_r(p); g += ch_g(p); b += ch_b(p);
                }
            }
            r /= 4; g /= 4; b /= 4;
            dst[i++] = pack(r, g, b);
        }
    }
}

/* ------------------------------------------------------------------ codebook */

typedef struct {
    long nd;
    int n;
    int32_t *pix;    /* nd * n block values */
    dblock_t *blk;   /* nd entries          */
} codebook_t;

static void codebook_free(codebook_t *cb)
{
    free(cb->pix);
    free(cb->blk);
    cb->pix = NULL;
    cb->blk = NULL;
}

/* FC:1015-1050 createCodebuch / FC:1058-1093 createCodebuchRGB. */
static int codebook_build(codebook_t *cb, const int32_t *argb, int W, int H, int B, int is_rgb)
{
    int sw = W / 2, sh = H / 2;
    int32_t *s = (int32_t *)malloc(sizeof(int32_t) * (size_t)sw * sh);
    if (!s) return -1;
    if (is_rgb) fic_oracle_scale_image_rgb(argb, W, H, s);
    else fic_oracle_scale_image(argb, W, H, s);
    int abstand = B / 4;                                           /* FC:1019 */
    long cap = (long)(sw / abstand - 3) * (long)(sh / abstand - 3); /* FC:1022 */
    int n = B * B;
    cb->n = n;
    cb->pix = (int32_t *)malloc(sizeof(int32_t) * (size_t)cap * n);
    cb->blk = (dblock_t *)malloc(sizeof(dblock_t) * (size_t)cap);
    int *tmp = (int *)malloc(sizeof(int) * n);
    if (!cb->pix || !cb->blk || !tmp) { free(s); free(tmp); codebook_free(cb); return -1; }
    long i = 0;
    for (int y = 0; y < sh; y += abstand) {
        for (int x = 0; x < sw; x += abstand) {
            if (y + B <= sh && x + B <= sw) {
                if (i >= cap) { free(s); free(tmp); codebook_free(cb); return -2; } /* AIOOBE */
                int32_t *blk = cb->pix + i * n;
                for (int ry = 0; ry < B; ry++)
                    for (int rx = 0; rx < B; rx++) {
                        int32_t p = s[x + rx + (y + ry) * sw];
                        blk[rx + ry * B] = is_rgb ? pack(ch_r(p), ch_g(p), ch_b(p)) : ch_r(p);
                    }
                dblock_init(&cb->blk[i], blk, n, is_rgb, tmp);
                i++;
            }
        }
    }
    cb->nd = i;
    free(s);
    free(tmp);
    return 0;
}

long fic_oracle_create_codebook(const int32_t *argb, int W, int H, int B, int is_rgb,
                                int32_t *pool, int32_t *mean, float *var)
{
    codebook_t cb;
    if (B < 4 || W < 2 || H < 2) return -1;
    if (codebook_build(&cb, argb, W, H, B, is_rgb)) return -1;
    if (pool) memcpy(pool, cb.pix, sizeof(int32_t) * (size_t)cb.nd * cb.n);
    for (long i = 0; i < cb.nd; i++) {
        const dblock_t *d = &cb.blk[i];
        if (!is_rgb) {
            if (mean) mean[i] = d->mittelWert;
            if (var) var[i] = d->variance;
        } else {
            if (mean) {
                mean[4 * i] = d->mittelWert; mean[4 * i + 1] = d->mittelWertR;
                mean[4 * i + 2] = d->mittelWertG; mean[4 * i + 3] = d->mittelWertB;
            }
            if (var) {
                var[3 * i] = d->varianceR; var[3 * i + 1] = d->varianceG;
                var[3 * i + 2] = d->varianceB;
            }
        }
    }
    long nd = cb.nd;
    codebook_free(&cb);
    return nd;
}

/* ------------------------------------------------------------------ grey search */

/* FC:655-687 getErrorVarianceCovariance -> {error, kov, varD, rangeM, domainM}. */
static void err_var_cov(const int *range, int rangeM, const dblock_t *db, int n, float out[5])
{
    float domainM = (float)db->mittelWert;
    float kov = 0, vR = 0;
    float varSq = db->variance;
    const int *domain = (const int *)db->argb;
    for (int i = 0; i < n; i++) {
        float gR = (float)(range[i] - rangeM);
        float gD = (float)domain[i] - domainM;
        kov += gR * gD;
        vR += gR;
    }
    float r = 0, error = 0;
    if (vR == 0 || sqrt((double)varSq) == 0)
        r = 0;
    else
        r = (float)((double)kov / ((double)vR * sqrt((double)varSq)));
    r = r * r;
    error = (vR * vR) * (1 - r);
    out[0] = error; out[1] = kov; out[2] = varSq; out[3] = (float)rangeM; out[4] = domainM;
}

/* FC:613-644 getBestDomainblock over the wk x wk window anchored at (dy, dx)
 * (window gather FC:139-150 is folded into the index expression). */
static void best_domainblock(const codebook_t *cb, int dpw, int wk, int dy, int dx,
                             const int *range, int rangeM, float res[3])
{
    float smallest = 10000000;
    float best[6] = {0, 0, 0, 0, 0, 0};
    int c = 0;
    for (int ky = 0; ky < wk; ky++) {
        for (int kx = 0; kx < wk; kx++, c++) {
            long index = dx + kx + (long)(dy + ky) * dpw;
            float ab[5];
            err_var_cov(range, rangeM, &cb->blk[index], cb->n, ab);
            if (ab[0] < smallest) {
                smallest = ab[0];
                best[0] = (float)c;
                best[1] = ab[0]; best[2] = ab[1]; best[3] = ab[2]; best[4] = ab[3]; best[5] = ab[4];
            }
        }
    }
    float a = best[2] / best[3];
    if (a < -1) a = -1;
    else if (a > 1) a = 1;
    float b = best[4] - a * best[5];
    res[0] = best[0]; res[1] = a; res[2] = b;
}

/* ------------------------------------------------------------------ isometry extension
 * NOT IN THE REFERENCE (which searches the identity only, FC:642, FC:733): the classical 8 isometries of
 * a square block.  T_k maps a range pixel (ry, rx) to the domain pixel (sy, sx) whose value it is compared
 * with / reconstructed from.  k: 0 identity, 1-3 rotations by 90/180/270 degrees, 4 mirror x, 5 mirror y,
 * 6 transpose, 7 anti-transpose.  Parity of this mode is defined by this file, not by the reference. */
void fic_oracle_iso_map(int k, int B, int ry, int rx, int *sy, int *sx)
{
    int m = B - 1;
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

/* getBestDomainblock with the candidate loop extended by an inner loop over the 8 isometries: same score
 * (err_var_cov on the permuted domain block), same strict-< rule, candidate order (c, k) lexicographic.
 * res = {c, a, b, k}. */
static void best_domainblock_iso(const codebook_t *cb, int dpw, int wk, int dy, int dx, int B,
                                 const int *range, int rangeM, float res[4])
{
    float smallest = 10000000;
    float best[7] = {0, 0, 0, 0, 0, 0, 0};
    int n = cb->n;
    int32_t *perm = (int32_t *)malloc(sizeof(int32_t) * n);
    int c = 0;
    for (int ky = 0; ky < wk; ky++) {
        for (int kx = 0; kx < wk; kx++, c++) {
            long index = dx + kx + (long)(dy + ky) * dpw;
            const dblock_t *src = &cb->blk[index];
            for (int k = 0; k < 8; k++) {
                dblock_t db = *src;  /* mean and variance are invariant under a pixel permutation */
                for (int ry = 0; ry < B; ry++)
                    for (int rx = 0; rx < B; rx++) {
                        int sy, sx;
                        fic_oracle_iso_map(k, B, ry, rx, &sy, &sx);
                        perm[rx + ry * B] = src->argb[sx + sy * B];
                    }
                db.argb = perm;
                float ab[5];
                err_var_cov(range, rangeM, &db, n, ab);
                if (ab[0] < smallest) {
                    smallest = ab[0];
                    best[0] = (float)c;
                    best[1] = ab[0]; best[2] = ab[1]; best[3] = ab[2]; best[4] = ab[3]; best[5] = ab[4];
                    best[6] = (float)k;
                }
            }
        }
    }
    free(perm);
    float a = best[2] / best[3];
    if (a < -1) a = -1;
    else if (a > 1) a = 1;
    float b = best[4] - a * best[5];
    res[0] = best[0]; res[1] = a; res[2] = b; res[3] = best[6];
}

/* ------------------------------------------------------------------ RGB search */

/* FC:760-808 getErrorVarianceCovarianceRGB ->
 * {error, kov, varSq, rangeRM, domainR, rangeGM, domainG, rangeBM, domainB}. */
static void err_var_cov_rgb(const int32_t *range, const dblock_t *db, int n, int *tmp, float out[9])
{
    const int32_t *domain = db->argb;
    float domainR = (float)db->mittelWertR, domainG = (float)db->mittelWertG,
          domainB = (float)db->mittelWertB;
    for (int i = 0; i < n; i++) tmp[i] = ch_r(range[i]);
    int rangeRM = mittelwert(tmp, n);
    for (int i = 0; i < n; i++) tmp[i] = ch_g(range[i]);
    int rangeGM = mittelwert(tmp, n);
    for (int i = 0; i < n; i++) tmp[i] = ch_b(range[i]);
    int rangeBM = mittelwert(tmp, n);

    float kov = 0;
    float varSq = (db->varianceR + db->varianceG + (float)db->mittelWertB); /* FC:776 (sic) */
    float vR = 0;
    float vD = (float)sqrt((double)db->variance);                           /* FC:778 */
    for (int i = 0; i < n; i++) {
        float gD = ((float)ch_r(domain[i]) - domainR) + ((float)ch_g(domain[i]) - domainG) +
                   ((float)ch_b(domain[i]) - domainB);
        float gR = (float)((ch_r(range[i]) - rangeRM) + (ch_g(range[i]) - rangeGM) +
                           (ch_b(range[i]) - rangeBM));
        kov += gR * gD;
        vR += gR;
        vD += gD;
    }
    float r = 0, error = 0;
    if (vR == 0 || vD == 0) r = 0;
    else r = kov / (vR * vD);
    r = r * r;
    error = (vR * vR) * (1 - r);
    out[0] = error; out[1] = kov; out[2] = varSq;
    out[3] = (float)rangeRM; out[4] = domainR;
    out[5] = (float)rangeGM; out[6] = domainG;
    out[7] = (float)rangeBM; out[8] = domainB;
}

/* FC:697-735 getBestDomainblockRGB. */
static void best_domainblock_rgb(const codebook_t *cb, int dpw, int wk, int dy, int dx,
                                 const int32_t *range, int *tmp, float res[5])
{
    float smallest = 10000000;
    float best[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    int c = 0;
    for (int ky = 0; ky < wk; ky++) {
        for (int kx = 0; kx < wk; kx++, c++) {
            long index = dx + kx + (long)(dy + ky) * dpw;
            float ab[9];
            err_var_cov_rgb(range, &cb->blk[index], cb->n, tmp, ab);
            if (ab[0] < smallest) {
                smallest = ab[0];
                best[0] = (float)c;
                for (int k = 0; k < 9; k++) best[k + 1] = ab[k];
            }
        }
    }
    float a = best[2] / best[3];
    if (a > 1) a = 1;
    if (a < -1) a = -1;
    float bR = best[4] - a * best[5];
    float bG = best[6] - a * best[7];
    float bB = best[8] - a * best[9];
    res[0] = best[0]; res[1] = a; res[2] = bR; res[3] = bG; res[4] = bB;
}

/* ------------------------------------------------------------------ encode drivers */

static int check_args(int W, int H, int B, int wk)
{
    if (B < 4 || (B & (B - 1))) return -1;        /* FC:1019: B/4 == 0 divides by zero */
    if (W <= 0 || H <= 0 || W % B || H % B) return -2; /* FC:124-126 overflow otherwise */
    int rpw = W / B, rph = H / B;
    if (rpw < 2 || rph < 2) return -3;            /* negative codebook size */
    int dpw = rpw * 2 - 3, dph = rph * 2 - 3;
    if (wk < 1 || wk > dpw || wk > dph) return -4; /* FC:93-96 -> negative index */
    return 0;
}

typedef struct {
    const int32_t *argb;
    int W, H, B, wk, is_rgb;
    const codebook_t *cb;
    long j0, j1;
    float *info;
    const long *list; /* NULL: ranges j0..j1-1; else ranges list[j0..j1-1] (any order, test spot checks) */
} job_t;

/* Body of the range loops FC:125-159 (grey) / FC:186-215 (RGB) for j in [j0, j1). */
static void *encode_job(void *arg)
{
    job_t *jb = (job_t *)arg;
    int W = jb->W, H = jb->H, B = jb->B, wk = jb->wk, n = B * B;
    int rpw = W / B, rph = H / B, dpw = rpw * 2 - 3, dph = rph * 2 - 3;
    int32_t *range = (int32_t *)malloc(sizeof(int32_t) * n);
    int *tmp = (int *)malloc(sizeof(int) * n);
    for (long jj = jb->j0; jj < jb->j1; jj++) {
        const long j = jb->list ? jb->list[jj] : jj;
        int x = (int)(j % rpw) * B, y = (int)(j / rpw) * B;
        int i = fic_oracle_domain_block_index(x, y, rpw, rph, dpw, B);
        int dy, dx;
        fic_oracle_generate_kernel(dpw, dph, i, wk, &dy, &dx);
        /* FC:588-602 getRangeblock / FC:564-577 getRangeblockRGB */
        int k = 0;
        for (int ry = 0; ry < B && y + ry < H; ry++)
            for (int rx = 0; rx < B && x + rx < W; rx++) {
                int32_t v = jb->argb[(x + rx) + (y + ry) * W];
                range[k++] = jb->is_rgb == 1 ? v : ch_r(v);
            }
        if (jb->is_rgb == 2) { /* grey + isometries (extension) */
            int rangeM = mittelwert((const int *)range, n);
            best_domainblock_iso(jb->cb, dpw, wk, dy, dx, B, (const int *)range, rangeM, jb->info + 4 * j);
        } else if (!jb->is_rgb) {
            int rangeM = mittelwert((const int *)range, n); /* FC:154 */
            best_domainblock(jb->cb, dpw, wk, dy, dx, (const int *)range, rangeM, jb->info + 3 * j);
        } else {
            best_domainblock_rgb(jb->cb, dpw, wk, dy, dx, range, tmp, jb->info + 5 * j);
        }
    }
    free(range);
    free(tmp);
    return NULL;
}

static int encode_common(const int32_t *argb, int W, int H, int B, int wk, int is_rgb,
                         long j0, long j1, int nthreads, float *info, const long *list)
{
    int rc = check_args(W, H, B, wk);
    if (rc) return rc;
    long nr = (long)(W / B) * (H / B);
    if (j0 < 0 || j0 > j1) return -5;
    if (!list && j1 > nr) return -5;
    if (list)
        for (long k = j0; k < j1; k++)
            if (list[k] < 0 || list[k] >= nr) return -5;
    codebook_t cb;
    if (codebook_build(&cb, argb, W, H, B, is_rgb == 1)) return -6;
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 256) nthreads = 256;
    if ((long)nthreads > j1 - j0) nthreads = (int)(j1 - j0 > 0 ? j1 - j0 : 1);
    job_t jobs[256];
    pthread_t th[256];
    long per = (j1 - j0 + nthreads - 1) / nthreads;
    for (int t = 0; t < nthreads; t++) {
        long a = j0 + t * per, b = a + per;
        if (a > j1) a = j1;
        if (b > j1) b = j1;
        jobs[t] = (job_t){argb, W, H, B, wk, is_rgb, &cb, a, b, info, list};
    }
    if (nthreads == 1) {
        encode_job(&jobs[0]);
    } else {
        for (int t = 0; t < nthreads; t++) pthread_create(&th[t], NULL, encode_job, &jobs[t]);
        for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
    }
    codebook_free(&cb);
    return 0;
}

int fic_oracle_encode_grey(const int32_t *argb, int W, int H, int B, int wk,
                           long range_begin, long range_end, int nthreads, float *info)
{
    return encode_common(argb, W, H, B, wk, 0, range_begin, range_end, nthreads, info, NULL);
}

int fic_oracle_encode_rgb(const int32_t *argb, int W, int H, int B, int wk,
                          long range_begin, long range_end, int nthreads, float *info)
{
    return encode_common(argb, W, H, B, wk, 1, range_begin, range_end, nthreads, info, NULL);
}

int fic_oracle_encode_grey_iso(const int32_t *argb, int W, int H, int B, int wk,
                               long range_begin, long range_end, int nthreads, float *info)
{
    return encode_common(argb, W, H, B, wk, 2, range_begin, range_end, nthreads, info, NULL);
}

/* The same range-loop body for an arbitrary list of range blocks (spot checks of images whose full encode the
 * CPU cannot finish): the codebook is built once, info[j] is written for every listed j.  mode: 0 grey, 1 RGB,
 * 2 grey + isometries (extension). */
int fic_oracle_encode_list(const int32_t *argb, int W, int H, int B, int wk, int mode,
                           const long *ranges, long count, int nthreads, float *info)
{
    if (mode < 0 || mode > 2 || count < 0 || (count && !ranges)) return -5;
    return encode_common(argb, W, H, B, wk, mode, 0, count, nthreads, info, ranges);
}

/* ------------------------------------------------------------------ stream I/O */

static void put_be32(uint8_t **p, int32_t v)
{
    if (*p) {
        (*p)[0] = (uint8_t)((uint32_t)v >> 24); (*p)[1] = (uint8_t)((uint32_t)v >> 16);
        (*p)[2] = (uint8_t)((uint32_t)v >> 8);  (*p)[3] = (uint8_t)v;
        *p += 4;
    }
}

static int32_t get_be32(const uint8_t *p)
{
    return (int32_t)(((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]);
}

/* FC:230-261 writeData. */
size_t fic_oracle_write_data(int is_rgb, int W, int H, int B, int wk, const float *info, uint8_t *out)
{
    long nr = (long)(W / B) * (H / B);
    uint8_t *p = out;
    put_be32(&p, is_rgb); put_be32(&p, W); put_be32(&p, H); put_be32(&p, B); put_be32(&p, wk);
    if (is_rgb == 0) {
        for (long r = 0; r < nr; r++) {
            put_be32(&p, j_f2i(info[3 * r + 0]));
            put_be32(&p, j_f2i(info[3 * r + 1] * 100));
            put_be32(&p, j_f2i(info[3 * r + 2]));
        }
        return 20 + 12 * (size_t)nr;
    }
    if (is_rgb == 2) { /* extension: grey codes + isometry index */
        for (long r = 0; r < nr; r++) {
            put_be32(&p, j_f2i(info[4 * r + 0]));
            put_be32(&p, j_f2i(info[4 * r + 1] * 100));
            put_be32(&p, j_f2i(info[4 * r + 2]));
            put_be32(&p, j_f2i(info[4 * r + 3]));
        }
        return 20 + 16 * (size_t)nr;
    }
    for (long r = 0; r < nr; r++) {
        put_be32(&p, j_f2i(info[5 * r + 0]));
        put_be32(&p, j_f2i(info[5 * r + 1] * 1000000));
        put_be32(&p, j_f2i(info[5 * r + 2] * 100000));
        put_be32(&p, j_f2i(info[5 * r + 3] * 100000));
        put_be32(&p, j_f2i(info[5 * r + 4]));
    }
    return 20 + 20 * (size_t)nr;
}

/* ------------------------------------------------------------------ decode */

/* FC:853-893 calculateIndices: window-local -> codebook index, in place, in float. */
static void calculate_indices(float *d, int stride, int W, int H, int B, int wk)
{
    int rpw = W / B, rph = H / B, dpw = rpw * 2 - 3, dph = rph * 2 - 3;
    long i = 0;
    for (int y = 0; y < H; y += B)
        for (int x = 0; x < W; x += B) {
            int di = fic_oracle_domain_block_index(x, y, rpw, rph, dpw, B);
            int dy, dx;
            fic_oracle_generate_kernel(dpw, dph, di, wk, &dy, &dx);
            int yd = j_f2i(d[i * stride] / (float)wk);
            int xd = j_f2i(fmodf(d[i * stride], (float)wk));
            int result = xd + dx + (yd + dy) * dpw;
            d[i * stride] = (float)result;
            i++;
        }
}

static int thresh(int v) { return v < 0 ? 0 : (v > 255 ? 255 : v); } /* FC:743-749 */

/* One sweep of FC:386-412 (grey) / FC:463-499 (RGB): snapshot codebook of `img`,
 * rewrite `img` in place, accumulate *avg in float in loop order. */
static int sweep(int32_t *img, int W, int H, int B, int is_rgb, const float *d, int stride,
                 int unquantised_collage, const int32_t *src, float *avg)
{
    codebook_t cb;
    if (codebook_build(&cb, src ? src : img, W, H, B, is_rgb == 1)) return -1;
    long i = 0;
    float acc = avg ? *avg : 0;
    (void)unquantised_collage;
    for (int y = 0; y < H; y += B)
        for (int x = 0; x < W; x += B) {
            const float *c = d + i * stride;
            long idx = (long)j_f2i(c[0]);
            if (idx < 0 || idx >= cb.nd) { codebook_free(&cb); return -2; }
            const int32_t *dom = cb.blk[idx].argb;
            for (int ry = 0; ry < B && y + ry < H; ry++)
                for (int rx = 0; rx < B && x + rx < W; rx++) {
                    int32_t old = img[x + rx + (y + ry) * W];
                    int32_t dv = dom[rx + ry * B];
                    if (is_rgb == 2) { /* extension: the domain pixel the isometry c[3] maps (ry, rx) to */
                        int sy, sx;
                        fic_oracle_iso_map(j_f2i(c[3]), B, ry, rx, &sy, &sx);
                        dv = dom[sx + sy * B];
                    }
                    if (is_rgb != 1) {
                        int range = ch_r(old);
                        int v = thresh(j_f2i(c[1] * (float)dv + c[2]));
                        img[x + rx + (y + ry) * W] = pack(v, v, v);
                        acc += (float)((range - v) * (range - v));
                    } else {
                        int vr = thresh(j_f2i(c[1] * (float)ch_r(dv) + c[2]));
                        int vg = thresh(j_f2i(c[1] * (float)ch_g(dv) + c[3]));
                        int vb = thresh(j_f2i(c[1] * (float)ch_b(dv) + c[4]));
                        int rr = ch_r(old), rg = ch_g(old), rb = ch_b(old);
                        img[x + rx + (y + ry) * W] = pack(vr, vg, vb);
                        acc += (float)((rr - vr) * (rr - vr) + (rg - vg) * (rg - vg) +
                                       (rb - vb) * (rb - vb));
                    }
                }
            i++;
        }
    if (avg) *avg = acc;
    codebook_free(&cb);
    return 0;
}

/* FC:547-553 decode -> FC:356-421 decodeGreyScale / FC:430-508 decodeRGB. */
int fic_oracle_decode(const uint8_t *s, size_t nbytes, int32_t *out, float *avg_error, int *iters)
{
    return fic_oracle_decode_iters(s, nbytes, 50, out, avg_error, iters);
}

int fic_oracle_decode_iters(const uint8_t *s, size_t nbytes, int max_iters, int32_t *out, float *avg_error, int *iters)
{
    if (nbytes < 20 || max_iters < 1) return -1;
    int is_rgb = get_be32(s) == 2 ? 2 : (get_be32(s) != 0); /* 2: isometry extension stream */
    int W = get_be32(s + 4), H = get_be32(s + 8), B = get_be32(s + 12), wk = get_be32(s + 16);
    int rc = check_args(W, H, B, wk);
    if (rc) return rc;
    long nr = (long)(W / B) * (H / B);
    int stride = is_rgb == 1 ? 5 : (is_rgb == 2 ? 4 : 3);
    if (nbytes < 20 + (size_t)nr * stride * 4) return -7;
    float *d = (float *)malloc(sizeof(float) * (size_t)nr * stride);
    const uint8_t *p = s + 20;
    for (long r = 0; r < nr; r++) {
        if (is_rgb == 2) {
            d[4 * r + 0] = (float)get_be32(p);
            d[4 * r + 1] = (float)get_be32(p + 4) / 100.0f;
            d[4 * r + 2] = (float)get_be32(p + 8);
            d[4 * r + 3] = (float)get_be32(p + 12);
            p += 16;
        } else if (!is_rgb) {
            d[3 * r + 0] = (float)get_be32(p);
            d[3 * r + 1] = (float)get_be32(p + 4) / 100.0f;
            d[3 * r + 2] = (float)get_be32(p + 8);
            p += 12;
        } else {
            d[5 * r + 0] = (float)get_be32(p);
            d[5 * r + 1] = (float)get_be32(p + 4) / 1000000.0f;
            d[5 * r + 2] = (float)get_be32(p + 8) / 100000.0f;
            d[5 * r + 3] = (float)get_be32(p + 12) / 100000.0f;
            d[5 * r + 4] = (float)get_be32(p + 16);
            p += 20;
        }
    }
    calculate_indices(d, stride, W, H, B, wk);
    for (long k = 0; k < (long)W * H; k++) out[k] = pack(128, 128, 128); /* FC:1142-1148 */
    float avg = avg_error ? *avg_error : 0;
    int counter;
    int done = 0;
    for (counter = 0; counter < max_iters; counter++) {
        rc = sweep(out, W, H, B, is_rgb, d, stride, 0, NULL, &avg);
        if (rc) { free(d); return rc; }
        done = counter + 1;
        avg = avg / (float)(W * H);
        if (avg < 1) break;
        if (counter != max_iters - 1) avg = 0;
    }
    if (avg_error) *avg_error = avg;
    if (iters) *iters = done;
    free(d);
    return 0;
}

/* FC:269-300 getBestGeneratedCollage / FC:308-347 getBestGeneratedCollageRGB. */
int fic_oracle_collage(const int32_t *argb, int W, int H, int B, int wk, int is_rgb,
                       float *info, int32_t *out)
{
    int rc = check_args(W, H, B, wk);
    if (rc) return rc;
    int stride = is_rgb == 1 ? 5 : (is_rgb == 2 ? 4 : 3);
    calculate_indices(info, stride, W, H, B, wk);                 /* FC:273 / FC:311 */
    for (long k = 0; k < (long)W * H; k++) out[k] = (int32_t)0xffa0a0a0; /* RI:19, RI:31 */
    return sweep(out, W, H, B, is_rgb, info, stride, 1, argb, NULL);
}

/* FC:32-45 isGreyScale. */
int fic_oracle_is_grey(const int32_t *a, int W, int H)
{
    for (long k = 0; k < (long)W * H; k++) {
        int r = ch_r(a[k]), g = ch_g(a[k]), b = ch_b(a[k]);
        if (r != g || g != b || b != r) return 0;
    }
    return 1;
}
