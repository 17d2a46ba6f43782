/*
 * fic_oracle_quadtree_budget_core.h -- the budget search of the quadtree oracles (TEST INFRASTRUCTURE ONLY), included by
 * fic_oracle_quadtree_budget.c (grey) and fic_oracle_quadtree_rgb_budget.c (RGB).  It knows nothing of the split rule's
 * shortcut on the device: each node's threshold comes from the literal (double)E > m * (double)N, and every trial tree
 * is written by the mode's own tree rule (the `write` callback).
 */
#include <math.h>
#include <stdlib.h>

#include "fic_oracle_quadtree_budget.h"

/* Writes the stream of tree `t` at max_mse = m into out; returns its size. */
typedef size_t (*qt_write_fn)(void *t, double m, uint8_t *out);

/* The smallest double m at which (double)E > m * N no longer holds (+0.0 for E == 0). */
static double qt_stop_mse(long long E, double N)
{
    double m = (double)E / N;
    while ((double)E > m * N) m = nextafter(m, INFINITY);
    for (double d = nextafter(m, -INFINITY); !((double)E > d * N); d = nextafter(m, -INFINITY)) m = d;
    return m;
}

static int qt_cmp_double(const void *a, const void *b)
{
    double x = *(const double *)a, y = *(const double *)b;
    return x < y ? -1 : x > y;
}

/* nl levels, level L with nr[L] blocks of collage error err[L][.] and N[L] = C * B_L^2. */
static int qt_budget_search(void *t, qt_write_fn write, int nl, const long *nr, long long *const *err, const double *N,
                            size_t max_bytes, uint8_t *out, size_t *nbytes, double *max_mse)
{
    size_t least = write(t, INFINITY, out), full = write(t, -INFINITY, out);
    if (max_bytes < least) {
        *nbytes = least;
        *max_mse = INFINITY;
        return -9;
    }
    if (full <= max_bytes) {
        *nbytes = full;
        *max_mse = -INFINITY;
        return 0;
    }
    long k = 0;
    for (int L = 0; L + 1 < nl; L++) k += nr[L];
    double *c = (double *)malloc(sizeof(double) * (size_t)k);
    k = 0;
    for (int L = 0; L + 1 < nl; L++)
        for (long j = 0; j < nr[L]; j++) c[k++] = qt_stop_mse(err[L][j], N[L]);
    qsort(c, (size_t)k, sizeof(double), qt_cmp_double);
    /* size is constant between consecutive thresholds and fits at the largest (every node stops: the unsplit tree) */
    long lo = 0, hi = k - 1;
    while (lo < hi) {
        long mid = (lo + hi) / 2;
        if (write(t, c[mid], out) <= max_bytes) hi = mid;
        else lo = mid + 1;
    }
    *max_mse = c[lo];
    *nbytes = write(t, c[lo], out);
    free(c);
    return 0;
}
