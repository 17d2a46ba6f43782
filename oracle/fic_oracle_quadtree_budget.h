/*
 * fic_oracle_quadtree_budget.h -- CPU oracle of the quadtree encode to a byte budget (TEST INFRASTRUCTURE ONLY).
 *
 * NOT IN THE REFERENCE.  size(m) is the size of the stream fic_oracle_encode_quadtree[_rgb] writes at max_mse = m; these
 * entries write the stream at m* and report m*, the smallest double with size(m*) <= max_bytes (-inf when the fully split
 * tree fits).  Stated plainly: every split-capable node's own threshold (the smallest m at which (double)E > m * (double)N
 * no longer holds, N = C * B^2, found by nextafter steps), sorted, bisected with the oracle's own tree rule.
 * max_bytes below the unsplit tree's size: -9, with that size in *nbytes and +inf in *max_mse.  `out` must hold
 * fic_oracle_quadtree[_rgb]_bound bytes.  Other return codes as fic_oracle_encode_quadtree[_rgb].
 */
#ifndef FIC_ORACLE_QUADTREE_BUDGET_H
#define FIC_ORACLE_QUADTREE_BUDGET_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

int fic_oracle_encode_quadtree_budget(const int32_t *argb, int W, int H, int b_max, int b_min, int wk, size_t max_bytes,
                                      int nthreads, uint8_t *out, size_t *nbytes, double *max_mse);
int fic_oracle_encode_quadtree_rgb_budget(const int32_t *argb, int W, int H, int b_max, int b_min, int wk,
                                          size_t max_bytes, int nthreads, uint8_t *out, size_t *nbytes, double *max_mse);

#ifdef __cplusplus
}
#endif
#endif
