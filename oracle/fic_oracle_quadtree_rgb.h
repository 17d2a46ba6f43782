/*
 * fic_oracle_quadtree_rgb.h -- CPU oracle of the RGB quadtree extension FIC_MODE_RGB_QT (include/fic_b200.h).
 *
 * TEST INFRASTRUCTURE ONLY, like fic_oracle.h, on which it builds: only tests/ and tools/ load it (through
 * oracle/quadtree_rgb.py); the product never links, loads or calls it.  Not in the reference, so it is pinned by the
 * numpy restatement of its rule in tests/test_oracle_quadtree_rgb.py, by the degenerate trees, which must reproduce the
 * fixed-block RGB encode and decode of fic_oracle.c, and by the reference's own stream unknown.run, whose codes a tree
 * that never splits at b_max = 8, wk = 2 on LenaColored must carry.
 */
#ifndef FIC_ORACLE_QUADTREE_RGB_H
#define FIC_ORACLE_QUADTREE_RGB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* The grey quadtree rule of fic_oracle_quadtree.h with the reference's RGB codes.  encode: levels b_max .. b_min, each
 * fic_oracle_encode_rgb at that B (wk == 0: each level's whole pool, W == H), its codes quantised as writeData does
 * {c, qa, qbR, qbG, qbB}; a block above b_min is split iff (double)E > max_mse * (double)(3*B*B), E = sum over its pixels
 * and the three channels of (thresh((int)(a * d_c + b_c)) - s_c)^2, the code dequantised as the RGB decoder does
 * (a = qa / 1e6f, bR = qbR / 1e5f, bG = qbG / 1e5f, bB = qbB), d_c from the source's RGB decimation
 * (fic_oracle_scale_image_rgb) at the code's codebook block.  Header 4, W, H, 0, wk, b_max, b_min, n_leaves, the flag
 * bytes, 20 bytes per leaf.  out must hold fic_oracle_quadtree_rgb_bound bytes; *nbytes gets the size.
 * decode: the constant-128 image, then sweeps that RGB-decimate the last image and let every leaf write each channel's
 * thresh((int)(a * d_c + b_c)); S = exact u64 sum of squared changes over pixels and channels,
 * avgError = (float)S / (float)(W*H); stops below 1 or after max_iters sweeps.  argb_out: W*H ints.  Returns 0, or a
 * negative code (-7 malformed stream, among them a grey quadtree stream; -2 a leaf outside its pool; -1..-4 bad
 * geometry). */
size_t fic_oracle_quadtree_rgb_bound(int W, int H, int b_max, int b_min);
int fic_oracle_encode_quadtree_rgb(const int32_t *argb, int W, int H, int b_max, int b_min, int wk, double max_mse,
                                   int nthreads, uint8_t *out, size_t *nbytes);
int fic_oracle_decode_quadtree_rgb(const uint8_t *stream, size_t nbytes, int max_iters, int32_t *argb_out,
                                   float *avg_error, int *iters);

#ifdef __cplusplus
}
#endif
#endif
