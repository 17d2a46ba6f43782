/*
 * fic_oracle.h -- CPU oracle for the fractal encode/decode hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  This is a plain-C restatement of the reference
 * algorithm (LariWa/Fractal-Image-Compression, src/bvk_ss19/FractalCompression.java
 * = "FC", src/bvk_ss19/Domainblock.java = "DB").  Only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs may load it; the product
 * (libfic_b200.so) never links, loads or calls anything in oracle/.
 *
 * Parity pinning: the reference ships no tests and cannot run here (no JVM), so the
 * oracle is pinned by the two artefacts the reference does ship (see
 * tests/test_oracle_golden.py): the bundled stream `unknown.run` (RGB encode of
 * LenaColored.jpg, B=8, wk=2 -- reproduced byte for byte) and the five "MSE" labels
 * visible in Animation.gif (grey encode -> quantise -> decode of LenaGrey.png).
 * Everything beyond those (full-pool search, synthetic images) rests on the oracle
 * being a literal restatement that passes both.
 */
#ifndef FIC_ORACLE_H
#define FIC_ORACLE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Geometry helpers (FC:516-545, FC:84-100). */
int fic_oracle_domain_block_index(int x, int y, int rpw, int rph, int dpw, int B);
void fic_oracle_generate_kernel(int dpw, int dph, int index, int wk, int *dy, int *dx);

/* 2x decimation (FC:970-1007 grey, FC:901-962 RGB).  dst holds (W/2)*(H/2) ARGB ints. */
void fic_oracle_scale_image(const int32_t *argb, int W, int H, int32_t *dst);
void fic_oracle_scale_image_rgb(const int32_t *argb, int W, int H, int32_t *dst);

/* Codebook (FC:1015-1050 / FC:1058-1093 + DB:23-42).  Returns the number of domain
 * blocks; pool gets ND*B*B ints (grey value, or packed ARGB when is_rgb), mean gets
 * ND (grey) or 4*ND (RGB: mittelWert-of-argb, R, G, B) ints, var gets ND (grey) or
 * 3*ND (RGB: R, G, B) floats.  Any output pointer may be NULL. */
long fic_oracle_create_codebook(const int32_t *argb, int W, int H, int B, int is_rgb,
                                int32_t *pool, int32_t *mean, float *var);

/* Encoders (FC:109-162 grey -> info[NR][3]; FC:171-219 RGB -> info[NR][5]).
 * Ranges j in [range_begin, range_end) are computed (raster order, as FC:123-158);
 * pass 0, NR for a full encode.  info is indexed by absolute j.  nthreads > 1 splits
 * the range loop over threads (ranges are independent; results are identical).
 * Returns 0, or a negative code when the reference would fault on the arguments. */
int fic_oracle_encode_grey(const int32_t *argb, int W, int H, int B, int wk,
                           long range_begin, long range_end, int nthreads, float *info);
int fic_oracle_encode_rgb(const int32_t *argb, int W, int H, int B, int wk,
                          long range_begin, long range_end, int nthreads, float *info);

/* The same loop body for a list of range blocks (count entries of `ranges`, any order): info[j] is written for
 * every listed j only.  mode: 0 grey, 1 RGB, 2 grey + isometries.  Used by the spot checks of the 4096^2 / 8192^2
 * configurations, whose full encode takes the CPU hours. */
int fic_oracle_encode_list(const int32_t *argb, int W, int H, int B, int wk, int mode,
                           const long *ranges, long count, int nthreads, float *info);

/* EXTENSION (not in the reference, which has no isometries): grey encode whose candidate loop has an inner
 * loop over the 8 isometries of the domain block (order (c, k) lexicographic, same score, same strict-<
 * rule) -> info[NR][4] = {c, a, b, k}.  is_rgb == 2 selects this mode in write_data / collage, and a stream
 * whose first header int is 2 decodes with it.  fic_oracle_iso_map: range pixel (ry, rx) -> domain pixel. */
void fic_oracle_iso_map(int k, int B, int ry, int rx, int *sy, int *sx);
int fic_oracle_encode_grey_iso(const int32_t *argb, int W, int H, int B, int wk,
                               long range_begin, long range_end, int nthreads, float *info);

/* writeData (FC:230-261): serialises header + quantised codes, big endian.
 * Returns the byte count (20 + 12*NR grey, 20 + 20*NR RGB); out may be NULL. */
size_t fic_oracle_write_data(int is_rgb, int W, int H, int B, int wk, const float *info,
                             uint8_t *out);

/* decode (FC:547-553, FC:356-421, FC:430-508).  avg_error is the reference's static
 * FractalCompression.avgError: read on entry (it is never reset between decodes)
 * and written on exit.  iters receives the number of sweeps executed.
 * fic_oracle_decode_iters: the same loop with the limit max_iters (>= 1) in place of the
 * reference's 50 (FC:381), as fic_decode's max_iters; an unconverged value is kept after
 * the last allowed sweep (FC:416-417). */
int fic_oracle_decode(const uint8_t *stream, size_t nbytes, int32_t *argb_out,
                      float *avg_error, int *iters);
int fic_oracle_decode_iters(const uint8_t *stream, size_t nbytes, int max_iters,
                            int32_t *argb_out, float *avg_error, int *iters);

/* getBestGeneratedCollage[RGB] (FC:269-347): one decode step from the source image
 * with the unquantised codes.  Like the reference it rewrites info[.][0] in place
 * from window-local to codebook index (FC:273). */
int fic_oracle_collage(const int32_t *argb, int W, int H, int B, int wk, int is_rgb,
                       float *info, int32_t *argb_out);

/* isGreyScale (FC:32-45). */
int fic_oracle_is_grey(const int32_t *argb, int W, int H);

#ifdef __cplusplus
}
#endif
#endif
