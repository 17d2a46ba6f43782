/*
 * fic_oracle_quadtree.h -- CPU oracle of the quadtree extension FIC_MODE_GREY_QT (include/fic_b200.h).
 *
 * TEST INFRASTRUCTURE ONLY, like fic_oracle.h, on which it builds: only tests/ and tools/ load it (through
 * oracle/quadtree.py); the product never links, loads or calls it.  Not in the reference, so it is pinned by the numpy
 * restatement of its rule in tests/test_oracle_quadtree.py and by the degenerate trees, which must reproduce the
 * reference-shaped fixed-block encode and decode of fic_oracle.c.
 */
#ifndef FIC_ORACLE_QUADTREE_H
#define FIC_ORACLE_QUADTREE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* encode: levels b_max .. b_min, each fic_oracle_encode_grey at that B (wk == 0: each level's whole pool, W == H);
 * a block above b_min is split iff (double)E > max_mse * (double)(B*B), E = sum over its pixels of
 * (thresh((int)(a * d + b)) - s)^2 with its quantised code {c, qa, qb}, a = qa / 100f, b = qb, d from the source's
 * decimated plane at the code's codebook block.  out must hold fic_oracle_quadtree_bound bytes; *nbytes gets the size.
 * decode: the constant-128 image, then sweeps that decimate the last image and let every leaf write
 * thresh((int)(a * d + b)); S = exact u64 sum of squared changes, avgError = (float)S / (float)(W*H); stops below 1 or
 * after max_iters sweeps.  argb_out: W*H ints.  Returns 0, or a negative code (-7 malformed stream, -2 a leaf outside
 * its pool, -1..-4 bad geometry). */
size_t fic_oracle_quadtree_bound(int W, int H, int b_max, int b_min);
int fic_oracle_encode_quadtree(const int32_t *argb, int W, int H, int b_max, int b_min, int wk, double max_mse,
                               int nthreads, uint8_t *out, size_t *nbytes);
int fic_oracle_decode_quadtree(const uint8_t *stream, size_t nbytes, int max_iters, int32_t *argb_out,
                               float *avg_error, int *iters);

#ifdef __cplusplus
}
#endif
#endif
