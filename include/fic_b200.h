/*
 * fic_b200.h -- C ABI of libfic_b200.so, the B200-native (sm_100a) drop-in for the
 * encode / decode hot path of LariWa/Fractal-Image-Compression.
 *
 * The reference (Java, src/bvk_ss19/FractalCompression.java = "FC") has no FFI seam of
 * its own; this header is the seam SURVEY.md section 8(b) cuts: the bodies of the two
 * range-block driver loops and of the decoder sweep move behind these calls, while
 * image loading (RasterImage.java), grey/RGB dispatch (FC:54-59) and the stream
 * writer stay on the host side (Java through Panama FFM / JNI, see INTEGRATION.md;
 * C++ and Python mirrors live in fractal-image-compression_b200/host/).
 *
 * Conventions
 *   - Plain pointers and sizes only.  The caller owns every host buffer; the library
 *     owns device memory, streams and events inside the opaque handle.
 *   - `argb` is the reference's pixel format: int32 0xAARRGGBB, scanline order,
 *     W*H entries (RasterImage.java:22).
 *   - Codes are returned in the reference's own layout: `info` is
 *     FractalCompression.imageInfo (float[NR][3] = {window-local index, a, b}, FC:124,
 *     FC:642) or imageInfoRGB (float[NR][5] = {index, a, bR, bG, bB}, FC:185, FC:733);
 *     `qcodes` (optional, may be NULL) holds the ints writeData would emit for the same
 *     rows (FC:242-244 / FC:250-254), so the Java side needs no float work.
 *   - Range blocks j are in raster order (FC:123-158); every encode entry takes a
 *     half-open range-block interval [range_begin, range_end) so that one image can be
 *     sharded over GPUs / processes by range rows.  Outputs are indexed by absolute j;
 *     rows outside the interval are left untouched.
 *   - Every entry returns FIC_OK (0) or a negative FIC_E_* code; fic_last_error()
 *     gives the message.  The reference signals all failures as `throws Exception`
 *     (FC:54, FC:109, FC:171, FC:230, FC:356, FC:547); argument sets on which the
 *     reference would throw (ArithmeticException for B < 4 at FC:1019,
 *     ArrayIndexOutOfBounds for W % B != 0 at FC:124-126 or widthKernel > pool width at
 *     FC:93-96) are rejected with FIC_E_ARG, not "fixed".
 *   - One in-flight call per handle; distinct handles are independent.
 *   - There is no CPU fallback: without a CUDA device every compute entry fails with
 *     FIC_E_CUDA.
 */
#ifndef FIC_B200_H
#define FIC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FIC_OK 0
#define FIC_E_ARG (-1)     /* arguments the reference would throw on              */
#define FIC_E_CUDA (-2)    /* CUDA runtime / launch failure, or no device         */
#define FIC_E_NOMEM (-3)   /* device or host allocation failed                    */
#define FIC_E_STREAM (-4)  /* malformed .run stream                               */
#define FIC_E_INTERNAL (-5)

/* Code layout / colour mode (the `is_rgb` argument of the entries below; 0 and 1 are the reference's isRGB
 * header flag, FC:234-238).  FIC_MODE_GREY_ISO is an EXTENSION the reference does not have: every candidate
 * domain block is tried under the 8 isometries of the square; codes carry a 4th value, the isometry index. */
#define FIC_MODE_GREY 0     /* {c, a, b} per range                       */
#define FIC_MODE_RGB 1      /* {c, a, bR, bG, bB} per range              */
#define FIC_MODE_GREY_ISO 2 /* {c, a, b, k} per range; k = isometry 0..7 */

/* Search engine selection (fic_set_option(FIC_OPT_ENGINE, ...)). */
#define FIC_ENGINE_AUTO 0   /* tcgen05 search when the window is the whole pool; the fused one-launch encode for the
                             * reference's GUI windows (widthKernel <= 16) on images of up to 16 K range blocks; else direct */
#define FIC_ENGINE_DIRECT 1 /* multi-kernel direct (CUDA-core) windowed search for every window */
#define FIC_ENGINE_UMMA 2   /* force the tcgen05 search; FIC_E_ARG if not applicable  */
#define FIC_ENGINE_FUSED 3  /* force the fused windowed encode (decimate + stats + search + solve in one launch);
                             * FIC_E_ARG unless widthKernel <= 16 and no isometries  */

/* Tensor-core instruction kind of the tcgen05 search (fic_set_option(FIC_OPT_UMMA_KIND, ...)).
 * Both produce the exact integer covariances, hence the same codes.  RGB images have a kind::f16 path only
 * (blockgroesse 4, 8 and 16): this option does not apply to them. */
#define FIC_UMMA_KIND_AUTO 0 /* kind::f16 for B = 4, 8; kind::i8 for B = 16               */
#define FIC_UMMA_KIND_I8 1   /* u8 x s8 -> s32, two s8 digits per centred domain pixel    */
#define FIC_UMMA_KIND_F16 2  /* binary16 x binary16 -> binary32 (B = 16 still runs i8)    */

/* CTA pairs of the tcgen05 search (fic_set_option(FIC_OPT_UMMA_PAIR, ...)): two CTAs of one TPC share every
 * tcgen05.mma (cta_group::2, M = 256), each supplying half of every domain tile.  Same codes either way.  The
 * pair kernel exists for kind::f16 (grey, RGB, isometry extension) and for kind::i8 at blockgroesse 16; elsewhere
 * (kind::i8 at blockgroesse 4, 8), and on a device partition that cannot co-schedule a 2-CTA cluster, the option is
 * ignored. */
#define FIC_UMMA_PAIR_AUTO 0 /* pairs where measured faster: blockgroesse 8 and 16 */
#define FIC_UMMA_PAIR_OFF 1
#define FIC_UMMA_PAIR_ON 2

#define FIC_OPT_ENGINE 1
#define FIC_OPT_UMMA_KIND 2
/* Read-only (fic_get_option): 1 if this device's kind::f16 tensor path reproduced the exact integer
 * covariances in the library's self-test (run once per handle, before the first kind::f16 search);
 * 0 means the handle silently runs kind::i8 (RGB: the CUDA-core search) instead. */
#define FIC_OPT_F16_EXACT 3
#define FIC_OPT_UMMA_PAIR 4
/* Read-only: 1 if the handle's last tcgen05 search ran the CTA-pair kernel. */
#define FIC_OPT_UMMA_PAIR_USED 5

typedef struct fic_handle fic_handle;
typedef struct fic_multi fic_multi; /* one context over several GPUs of the node, see "multi-GPU" below */

/* Per-call device timings in milliseconds (CUDA events on the handle's stream). */
typedef struct fic_timings {
    float h2d_ms;     /* host -> device copies                                   */
    float pool_ms;    /* unpack + 2x decimation + per-domain / per-range stats   */
    float search_ms;  /* range x domain search (direct or tcgen05) incl. operand packing */
    float kernel_ms;  /* the dominant search kernel alone (k_umma_search or k_search_direct_*) */
    float solve_ms;   /* winner -> (a, b) solve + quantisation                   */
    float d2h_ms;     /* device -> host copies                                   */
    float total_ms;
    int engine;       /* FIC_ENGINE_DIRECT, _UMMA or _FUSED actually used        */
    int launches;     /* kernels launched by this call                           */
    double search_evals; /* range x candidate evaluations done by the search     */
} fic_timings;

/* ---- lifetime ---------------------------------------------------------------- */

/* Creates a context on CUDA device `device` (cudaSetDevice ordinal). */
int fic_create(int device, fic_handle **out);
void fic_destroy(fic_handle *h);
const char *fic_last_error(const fic_handle *h); /* h may be NULL: last create error */
const char *fic_version(void);
int fic_set_option(fic_handle *h, int option, int value);
int fic_get_option(fic_handle *h, int option, int *value);
/* Run subsequent calls on a caller-provided CUDA stream (cudaStream_t), or NULL for
 * the handle's own stream (pass cudaStreamLegacy, 0x1, to mean the legacy default stream).  Used by the torch.distributed host so that library work
 * orders after the NCCL broadcast without a device-wide sync. */
int fic_set_stream(fic_handle *h, void *cuda_stream);
int fic_get_timings(const fic_handle *h, fic_timings *out);

/* ---- geometry (pure host helpers, no device needed) -------------------------- */

/* NR = (W/B)*(H/B), pool size ND = (2W/B-3)*(2H/B-3) (FC:111-116, FC:1022); returns
 * FIC_E_ARG on argument sets the reference would throw on. */
int fic_geometry(int W, int H, int B, int wk, int64_t *n_ranges, int64_t *n_domains);

/* ---- encode: replaces FC:119 + FC:125-159 (grey) and FC:181 + FC:186-215 (RGB) */

int fic_encode_grey(fic_handle *h, const int32_t *argb, int W, int H, int B, int wk,
                    int64_t range_begin, int64_t range_end, float *info, int32_t *qcodes);
int fic_encode_rgb(fic_handle *h, const int32_t *argb, int W, int H, int B, int wk,
                   int64_t range_begin, int64_t range_end, float *info, int32_t *qcodes);

/* The same calls for hosts that already hold 8-bit pixels (SURVEY 8b allows `const uint8_t*`): `plane` is the red
 * channel of a grey image (W*H bytes -- what FC:596 / FC:977 read from the ARGB ints), `planes` the R, G, B planes of
 * an RGB image (3*W*H bytes).  A quarter of the upload of the ARGB entries; results are identical. */
int fic_encode_grey_u8(fic_handle *h, const uint8_t *plane, int W, int H, int B, int wk,
                       int64_t range_begin, int64_t range_end, float *info, int32_t *qcodes);
int fic_encode_rgb_planes(fic_handle *h, const uint8_t *planes, int W, int H, int B, int wk,
                          int64_t range_begin, int64_t range_end, float *info, int32_t *qcodes);

/* EXTENSION (the reference searches the identity only, FC:642): grey encode whose candidate loop has an
 * inner loop over the 8 isometries of the domain block -- order (c, k) lexicographic, the reference's score
 * (FC:655-687) and strict-< rule.  info / qcodes are [NR][4] = {c, a, b, k} / {(int)c, (int)(a*100), (int)b, k};
 * k: 0 identity, 1-3 rotations by 90/180/270 degrees, 4 mirror x, 5 mirror y, 6 transpose, 7 anti-transpose
 * (the range pixel (ry, rx) takes the domain pixel T_k(ry, rx)).  Every
 * entry that takes `is_rgb` accepts FIC_MODE_GREY_ISO for these codes; the stream header then carries 2. */
int fic_encode_grey_iso(fic_handle *h, const int32_t *argb, int W, int H, int B, int wk,
                        int64_t range_begin, int64_t range_end, float *info, int32_t *qcodes);

/* Same, with the image already resident in device memory as 8-bit planes
 * (grey: red channel, W*H bytes; RGB: R, G, B planes, 3*W*H bytes; 16-byte aligned) and device output
 * buffers (float[NR][3|5], int32[NR][3|5]; either may be NULL).  Asynchronous on the
 * handle's stream; fic_sync() waits.  This is the entry the multi-GPU host uses after
 * the NCCL image broadcast. */
int fic_encode_planes_dev(fic_handle *h, const uint8_t *d_planes, int is_rgb, int W, int H,
                          int B, int wk, int64_t range_begin, int64_t range_end,
                          float *d_info, int32_t *d_qcodes);
int fic_sync(fic_handle *h);

/* Page-locks (and later releases) a caller-owned host buffer -- the ARGB array, the code arrays -- so that the
 * copies of fic_encode_* / fic_decode run at full PCIe rate instead of through the driver's staging buffer.
 * Optional: every entry accepts pageable memory.  A Java host calls it once per off-heap MemorySegment it
 * reuses (INTEGRATION.md); heap arrays handed over by JNI cannot be pinned this way. */
int fic_pin_host_buffer(fic_handle *h, void *ptr, size_t bytes);
int fic_unpin_host_buffer(fic_handle *h, void *ptr);

/* ---- decode: replaces FC:378-418 / FC:455-505 (after header + code parsing) --- */

/* `qcodes` are the ints read from the stream after the 5-int header (FC:370-376 /
 * FC:444-453), NR*3 (grey) or NR*5 (RGB).  *avg_error is FractalCompression.avgError:
 * read on entry (the reference never resets it between decodes, FC:20) and written on
 * exit; *iterations receives the sweep count (<= max_iters; the reference uses 50). */
int fic_decode(fic_handle *h, int is_rgb, int W, int H, int B, int wk, const int32_t *qcodes,
               int max_iters, int32_t *argb_out, float *avg_error, int *iterations);

/* The same decoder with the image returned as 8-bit planes (grey: W*H bytes; RGB: R, G, B planes) instead of ARGB
 * ints: to host memory, or (fic_decode_planes_dev) from device-resident codes -- as fic_encode_planes_dev leaves
 * them -- to a 16-byte-aligned device buffer.  Both synchronise before they return (avg_error / iterations are host
 * scalars). */
int fic_decode_u8(fic_handle *h, int is_rgb, int W, int H, int B, int wk, const int32_t *qcodes,
                  int max_iters, uint8_t *planes_out, float *avg_error, int *iterations);
int fic_decode_planes_dev(fic_handle *h, int is_rgb, int W, int H, int B, int wk,
                          const int32_t *d_qcodes, int max_iters, uint8_t *d_planes_out,
                          float *avg_error, int *iterations);

/* ---- batches: n_images same-size images per call ------------------------------- */

/* n_images images of W x H, back to back: argb [n][H][W]; codes [n][NR][S], S = 3 / 5 / 4 by mode
 * (FIC_MODE_GREY / FIC_MODE_RGB / FIC_MODE_GREY_ISO).  Every image's codes, decoded pixels, avgError bits and
 * iteration count equal what the single entries give for that image alone, bit for bit.
 *
 * Encode: where the single encode would run the fused one-launch kernel (widthKernel <= 16, no isometries, up to 16 K
 * range blocks per image, FIC_ENGINE_AUTO or _FUSED) the whole batch is one launch per group of images.  With the full
 * domain pool (widthKernel == domain blocks per width == per height; RGB without isometries) a group of images is ONE
 * tcgen05 tensor-core search: one pool build, sort, operand pack, search kernel, refine and solve for the whole group.
 * FIC_ENGINE_UMMA always runs it; FIC_ENGINE_AUTO runs it where the single encode would, and instead of the CUDA-core
 * search for groups of 4 images or more (full pools of up to 16 x 16 domains keep the fused kernel, which is faster
 * there).  A tensor-core group holds at most 256 images and about 1 GB of operand workspace.  Every other case (forced
 * DIRECT, windows between 17 and the full pool, the isometry extension below the full pool) runs the single-image
 * engine once per image inside the call: the images still go up and their codes come down in one copy per group, but
 * there is no launch saving.  planes (the _u8 form): [n][C][H][W], C = 3 for RGB, else 1 (the red channel).
 *
 * Decode: where the single decode would run its one-launch decoder (blockgroesse >= 8, W % 16 == 0, no isometries, up to
 * 2^20 pixels) a group of images decodes in one cooperative launch; every other image decodes as fic_decode would.
 * The reference's avgError is a never-reset static (FC:20), so a chain of single decodes carries each image's value
 * into the next image; a batch cannot reproduce that chain without running the images one after another, so it takes
 * one carry-in per image: avg_error[i] is read on entry and written on exit, exactly like the scalar of fic_decode,
 * and NULL means 0 for every image.  iterations: [n] or NULL.  planes_out: [n][C][H][W].
 *
 * FIC_E_ARG for n_images < 1, NULL images or codes, or a batch whose byte count overflows, besides the single entries'
 * rejections; FIC_E_STREAM when some image's codes index outside the domain pool (fic_last_error names the lowest
 * such image).  fic_get_timings then reports the whole call: total_ms, launches, engine (encode) and search_evals
 * (n * NR * widthKernel^2 * isometries); on the tensor-core engine also pool_ms, search_ms, kernel_ms and solve_ms,
 * summed over the groups. */
int fic_encode_batch(fic_handle *h, int mode, const int32_t *argb, int n_images, int W, int H, int B, int wk,
                     float *info, int32_t *qcodes);
int fic_encode_batch_u8(fic_handle *h, int mode, const uint8_t *planes, int n_images, int W, int H, int B, int wk,
                        float *info, int32_t *qcodes);
int fic_decode_batch(fic_handle *h, int mode, int n_images, int W, int H, int B, int wk, const int32_t *qcodes,
                     int max_iters, int32_t *argb_out, float *avg_error, int *iterations);
int fic_decode_batch_u8(fic_handle *h, int mode, int n_images, int W, int H, int B, int wk, const int32_t *qcodes,
                        int max_iters, uint8_t *planes_out, float *avg_error, int *iterations);

/* getBestGeneratedCollage[RGB] (FC:269-347): one decode step from the source image
 * with the unquantised codes.  Like the reference it rewrites info[.][0] in place from
 * window-local to codebook index (FC:273). */
int fic_collage(fic_handle *h, int is_rgb, const int32_t *argb, int W, int H, int B, int wk,
                float *info, int32_t *argb_out);

/* ---- multi-GPU: the same encode over several GPUs of one node (SURVEY 8b, 8e) --- */

/* Replaces the same reference loops (FC:119 + FC:125-159, FC:181 + FC:186-215) with the range-block rows sharded
 * over `n_devices` GPUs of this process: the image is uploaded once, broadcast to the other devices with
 * ncclBroadcast over NVLink (NCCL is loaded at run time; n_devices == 1 needs none), every device builds the whole
 * domain pool and searches a contiguous slice of range rows, and each device copies its code rows straight into the
 * caller's arrays.  Results are byte-identical to the single-device entries for every device count.
 * `devices` are CUDA ordinals (distinct).  One in-flight call per multi handle. */
int fic_create_multi(const int *devices, int n_devices, fic_multi **out);
void fic_destroy_multi(fic_multi *m);
const char *fic_multi_last_error(const fic_multi *m); /* m may be NULL: last create error */
int fic_multi_device_count(const fic_multi *m);
/* The per-device context of `rank` (0 .. n-1), owned by the multi handle: for fic_decode / fic_collage (replicas
 * only: the decoder does not shard), fic_pin_host_buffer, per-device timings.  Do not fic_destroy it. */
fic_handle *fic_multi_handle(fic_multi *m, int rank);
int fic_multi_set_option(fic_multi *m, int option, int value); /* fic_set_option on every device */
/* rank < 0: the slowest device per stage (total_ms: the longest device timeline); else that device's timings */
int fic_multi_get_timings(const fic_multi *m, int rank, fic_timings *out);
/* the range-block interval [begin, end) device `rank` encoded in the last call */
int fic_multi_range_slice(const fic_multi *m, int rank, int64_t *range_begin, int64_t *range_end);

int fic_multi_encode_grey(fic_multi *m, const int32_t *argb, int W, int H, int B, int wk, float *info, int32_t *qcodes);
int fic_multi_encode_rgb(fic_multi *m, const int32_t *argb, int W, int H, int B, int wk, float *info, int32_t *qcodes);
int fic_multi_encode_grey_iso(fic_multi *m, const int32_t *argb, int W, int H, int B, int wk, float *info, int32_t *qcodes);
int fic_multi_encode_grey_u8(fic_multi *m, const uint8_t *plane, int W, int H, int B, int wk, float *info, int32_t *qcodes);
int fic_multi_encode_rgb_planes(fic_multi *m, const uint8_t *planes, int W, int H, int B, int wk, float *info, int32_t *qcodes);

/* ---- diagnostics -------------------------------------------------------------- */

/* Measures the dense int8 tensor-pipe rate of the handle's GPU with a bare tcgen05.mma.kind::i8
 * loop (no epilogue, operands resident in shared memory): *tops receives TOP/s (2 ops per MAC).
 * bench.py uses it as the measured roofline denominator of the search kernel. */
int fic_measure_int8_peak(fic_handle *h, double *tops);

/* The same loop for either instruction kind (FIC_UMMA_KIND_I8 / FIC_UMMA_KIND_F16) and MMA shape
 * M = 128 x N = n_cols (128: the shape the search issues; 256: the widest single-CTA shape). */
int fic_measure_mma_peak(fic_handle *h, int kind, int n_cols, double *tops);

/* The loop issued by CTA pairs (tcgen05.mma.cta_group::2, M = 256, N = 128: the shape the pair form of the
 * search kernel issues, FIC_OPT_UMMA_PAIR). */
int fic_measure_mma_peak_pair(fic_handle *h, int kind, double *tops);

/* The decoder's avgError arithmetic on its own (test hook): the reference adds every squared pixel change to a
 * binary32 running sum in loop order (FractalCompression.java:407), so the value depends on the order once it passes
 * 2^24.  *sum receives carry + terms[0] + terms[1] + ... accumulated exactly that way, computed as fic_decode folds a
 * sweep: a one-warp replay for count < 2^22, the chunked transducer replay above.  terms: `count` integers in
 * [0, 3 * 255^2] (host memory). */
int fic_debug_float_sum(fic_handle *h, const int32_t *terms, int64_t count, float carry, float *sum);

/* ---- domain pool inspection (tests / debugging; not on the hot path) ---------- */

/* Runs the pool builder only and returns the 2x-decimated plane(s) (W/2*H/2 bytes per
 * channel), per-domain integer sums (ND per channel) and sums of squares. Any output
 * may be NULL. */
int fic_build_pool(fic_handle *h, const int32_t *argb, int is_rgb, int W, int H, int B,
                   uint8_t *decimated, int32_t *dom_sum, int32_t *dom_sumsq);

/* ---- .run stream (writeData FC:230-261, header parse FC:357-363, FC:548) ------ */

size_t fic_stream_size(int is_rgb, int W, int H, int B);
/* Serialises header + qcodes big-endian exactly as DataOutputStream.writeInt does. */
int fic_stream_write(int is_rgb, int W, int H, int B, int wk, const int32_t *qcodes,
                     uint8_t *out, size_t out_bytes);
/* Parses the header; *qcodes_off is the byte offset of the first code. */
int fic_stream_read_header(const uint8_t *stream, size_t nbytes, int *is_rgb, int *W, int *H,
                           int *B, int *wk, size_t *qcodes_off);
/* Copies the big-endian codes of a stream into host-endian ints (NR*3 or NR*5). */
int fic_stream_read_codes(const uint8_t *stream, size_t nbytes, int32_t *qcodes);

#ifdef __cplusplus
}
#endif
#endif /* FIC_B200_H */
