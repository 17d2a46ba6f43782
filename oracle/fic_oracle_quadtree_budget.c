/*
 * fic_oracle_quadtree_budget.c -- CPU oracle of the grey quadtree encode to a byte budget (TEST INFRASTRUCTURE ONLY, see
 * fic_oracle_quadtree_budget.h).  It includes fic_oracle_quadtree.c so that every level's codes, every block's collage
 * error and every trial tree come from the grey quadtree oracle's own static helpers (qt_block_sse, qt_split, qt_emit):
 * the tree written at m* is by construction the one fic_oracle_encode_quadtree writes at max_mse = m*.  Built as a
 * library of its own (with fic_oracle.c); same flags as fic_oracle.c.
 */
#include "fic_oracle_quadtree.c"

#include "fic_oracle_quadtree_budget_core.h"

typedef struct {
    qt_t t;
    int wk; /* as in the header: 0 = every level's whole pool */
} qt_budget_t;

/* The stream of the tree at max_mse = m (fic_oracle_encode_quadtree's flag and leaf loop); returns its size. */
static size_t qt_write_grey(void *ctx, double m, uint8_t *out)
{
    qt_budget_t *c = (qt_budget_t *)ctx;
    qt_t *t = &c->t;
    t->max_mse = m;
    long ntop = (long)(t->W / t->B[0]) * (t->H / t->B[0]), pad = (ntop + 3) & ~3L, n = 0;
    uint8_t *p = out + 32 + pad;
    memset(out + 32, 0, (size_t)pad);
    for (long j = 0; j < ntop; j++) {
        uint8_t f = 0;
        if (qt_split(t, 0, j)) {
            f = 1;
            for (int k = 0; k < 4; k++)
                if (qt_split(t, 1, qt_child(t, 0, j, k))) f |= (uint8_t)(2 << k);
        }
        out[32 + j] = f;
        qt_emit(t, 0, j, &p, &n);
    }
    uint8_t *h = out;
    put_be32(&h, 3); put_be32(&h, t->W); put_be32(&h, t->H); put_be32(&h, 0);
    put_be32(&h, c->wk); put_be32(&h, t->B[0]); put_be32(&h, t->B[t->nl - 1]); put_be32(&h, (int32_t)n);
    return (size_t)(p - out);
}

int fic_oracle_encode_quadtree_budget(const int32_t *argb, int W, int H, int b_max, int b_min, int wk, size_t max_bytes,
                                      int nthreads, uint8_t *out, size_t *nbytes, double *max_mse)
{
    int nl = qt_levels(W, H, b_max, b_min, wk);
    if (nl < 0) return nl;
    qt_budget_t c;
    memset(&c, 0, sizeof c);
    qt_t *t = &c.t;
    t->nl = nl; t->W = W; t->H = H; c.wk = wk;
    long nr[3] = {0};
    long long *err[3] = {0};
    double N[3] = {0};
    int32_t *dec = (int32_t *)malloc(sizeof(int32_t) * (size_t)(W / 2) * (H / 2));
    fic_oracle_scale_image(argb, W, H, dec); /* every level's codebook is cut from this plane */
    int rc = 0, bad = 0;
    for (int L = 0; L < nl && !rc; L++) { /* fic_oracle_encode_quadtree's levels */
        int B = b_max >> L, wkl = wk ? wk : 2 * (W / B) - 3;
        nr[L] = (long)(W / B) * (H / B);
        N[L] = (double)(B * B);
        t->B[L] = B; t->wk[L] = wkl; t->rpw[L] = W / B;
        float *info = (float *)malloc(sizeof(float) * 3 * (size_t)nr[L]);
        int32_t *q = (int32_t *)malloc(sizeof(int32_t) * 3 * (size_t)nr[L]);
        err[L] = (long long *)malloc(sizeof(long long) * (size_t)nr[L]);
        rc = fic_oracle_encode_grey(argb, W, H, B, wkl, 0, nr[L], nthreads, info);
        for (long j = 0; j < nr[L] && !rc; j++) { /* FC:242-244 */
            q[3 * j] = j_f2i(info[3 * j]);
            q[3 * j + 1] = j_f2i(info[3 * j + 1] * 100);
            q[3 * j + 2] = j_f2i(info[3 * j + 2]);
            err[L][j] = qt_block_sse(argb, dec, W, B, wkl, H, j, q + 3 * j, &bad);
        }
        free(info);
        t->codes[L] = q;
        t->err[L] = err[L];
    }
    if (!rc && bad) rc = -8;
    if (!rc) rc = qt_budget_search(&c, qt_write_grey, nl, nr, err, N, max_bytes, out, nbytes, max_mse);
    for (int L = 0; L < nl; L++) { free((void *)t->codes[L]); free(err[L]); }
    free(dec);
    return rc;
}
