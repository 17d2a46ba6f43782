// fic_internal.h -- shared host/device declarations of libfic_b200 (not part of the ABI).
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/fic_b200.h"

namespace fic {

// Block / pool geometry of one encode or decode call (FC:111-116, FC:1019-1022).
struct Geom {
    int W, H, B, n;       // image size, block size, n = B*B
    int wk;               // widthKernel: search window edge in domain-grid cells
    int rpw, rph;         // range blocks per width / height
    int dpw, dph;         // domain blocks per width / height (= 2*rp - 3)
    int sw, sh;           // decimated image size (W/2, H/2)
    int step;             // domain grid stride in decimated pixels (B/4, FC:1019)
    int C;                // channels: 1 grey, 3 RGB
    int n_iso;            // isometries searched per candidate: 1 (the reference), 8 (extension, grey only)
    int64_t NR, ND;
};

// Floats / ints per range in the code tables: {c, a, b} grey, {c, a, bR, bG, bB} RGB, {c, a, b, k} grey + isometry.
__host__ __device__ inline int code_stride(const Geom &g) { return g.C == 3 ? 5 : (g.n_iso > 1 ? 4 : 3); }

// mode: FIC_MODE_GREY / FIC_MODE_RGB / FIC_MODE_GREY_ISO.  Returns FIC_OK or FIC_E_ARG (same rejections as the
// reference's exceptions).
int make_geom(int W, int H, int B, int wk, int mode, Geom *g, const char **why);

// State block of a decode (device memory), shared by its kernels and read back by the host: the running sweep's exact
// sum of squared pixel changes, a "code indexes outside the pool" flag, the ticket of the sweep's CTAs, the done flag
// (converged, FC:414), the sweeps run, avgError's bits, and the grid barrier and bail word of the one-launch decoder.
// 8-byte aligned for the u64 atomics.  The one-launch decoder of a batch keeps one block per image; the first block's
// barrier is the launch's grid barrier and its ticket the launch's "some image is still sweeping" word.
struct DecodeState {
    unsigned long long sq_sum, bad_index;
    uint32_t ticket, done, iters, avg_bits, barrier, bail;
};
static_assert(sizeof(DecodeState) == 40 && offsetof(DecodeState, bad_index) == 8 && offsetof(DecodeState, ticket) == 16 &&
              offsetof(DecodeState, avg_bits) == 28 && offsetof(DecodeState, bail) == 36, "u64 words 0-1, u32 words 4-9");

// Device workspace owned by a handle (grow-only).
struct Work {
    int32_t *argb = nullptr;    // W*H staging of the caller's ARGB ints
    uint8_t *src = nullptr;     // C planes W*H (grey: red channel)
    uint8_t *dec = nullptr;     // C planes sw*sh, 2x decimated
    int32_t *dsum = nullptr;    // [C][ND] sum of domain pixels
    int32_t *dsq = nullptr;     // [C][ND] sum of squares of domain pixels
    int32_t *rsum = nullptr;    // [C][NR] sum of range pixels
    int32_t *best = nullptr;    // [NR] winning window-local candidate index
    float *info = nullptr;      // [NR][3|5] unquantised codes
    int32_t *q = nullptr;       // [NR][3|5] quantised codes
    // tcgen05 search operands (see fic_search_umma.cu)
    uint8_t *opA = nullptr;     // range operand blobs
    uint8_t *opB = nullptr;     // domain operand blobs
    // decoder
    uint8_t *img = nullptr;     // C planes W*H: the image being reconstructed (updated in place)
    uint8_t *dec2 = nullptr;    // second decimated buffer (Jacobi ping-pong with `dec`)
    float *dcode = nullptr;     // [NR][3|5] dequantised codes with codebook indices, then s32 doff[NR] (domain byte offsets)
    int32_t *perr = nullptr;    // per-pixel squared change in reference loop order (exact avgError path)
    DecodeState *state = nullptr;  // the decoder's state block
    uint16_t *dec3 = nullptr;   // RGB: R + G + B of the decimated planes (CUDA-core search)
    uint8_t *replay = nullptr;  // decoder, large images: per-chunk records of the exact avgError replay
    size_t cap[20] = {0};
};

// ---- kernel launchers (each returns the number of kernels it launched) -----------
// The pool builders take n_images same-size images back to back, one launch for all: ARGB [n][H][W] -> planes
// [n][C][H][W] -> decimated planes [n][C][sh][sw], dsum / dsq [n][C][ND], rsum [n][C][NR], dec3 [n][sh][sw].
int launch_unpack(const int32_t *d_argb, uint8_t *d_planes, int W, int H, int C, cudaStream_t s, int n_images = 1);
int launch_decimate(const uint8_t *d_src, uint8_t *d_dec, const Geom &g, cudaStream_t s, int n_images = 1);
int launch_domain_stats(const uint8_t *d_dec, int32_t *d_dsum, int32_t *d_dsq, const Geom &g,
                        cudaStream_t s, int n_images = 1);
int launch_range_stats(const uint8_t *d_src, int32_t *d_rsum, const Geom &g, cudaStream_t s, int n_images = 1);
int launch_sum_planes(const uint8_t *d_dec, uint16_t *d_dec3, const Geom &g, cudaStream_t s, int n_images = 1);  // RGB only
int launch_search_direct(const Work &w, const Geom &g, int64_t j0, int64_t j1, cudaStream_t s);
// Fused windowed encode (widthKernel <= 16, no isometries): decimation, stats, search, solve and quantisation in one
// launch, straight from the caller's pixels (ARGB ints or 8-bit planes); no intermediate arrays.  n_images > 1: that
// many images back to back at d_src, every range of each (j0 = 0, j1 = NR), codes in [n][NR] tables.
bool fused_encode_applicable(const Geom &g);
int launch_encode_fused(const void *d_src, int src_is_argb, const Geom &g, int64_t j0, int64_t j1, float *d_info,
                        int32_t *d_q, cudaStream_t s, int n_images = 1);
// Solve of ranges [j0, j1); a group of images (after the pool builders and launch_search_umma with n_images) passes
// the flat range [0, n * NR): best, info and q are [n][NR] tables.
int launch_solve(const Work &w, const Geom &g, int64_t j0, int64_t j1, float *d_info, int32_t *d_q,
                 cudaStream_t s);

// tcgen05 fused full-pool search (grey, window == whole pool).
// bare tcgen05.mma loop (M = 128, N = n_cols in {128, 256}): measured dense rate of kind::i8 (f16 = 0) or
// kind::f16 on this GPU in TOP/s (< 0 on error)
double measure_mma_peak(int num_sms, cudaStream_t s, int reps, int f16, int n_cols, const char **err);
double measure_mma_peak_pair(int num_sms, cudaStream_t s, int reps, int f16, uint32_t *tmem_bases, const char **err);
// 1: kind::f16 accumulators are the exact integer covariances on this device; 0: not; < 0: CUDA error
int umma_f16_selftest(int num_sms, cudaStream_t s, const char **err);
bool umma_applicable(const Geom &g);
// in-tree stable radix sort on 24-bit keys (probe / tests): result in the *_out arrays; 0 or a CUDA error code
int umma_debug_sort(uint32_t *d_keys, int32_t *d_vals, uint32_t *d_keys_out, int32_t *d_vals_out, int64_t n, cudaStream_t s);
// `kind`: FIC_UMMA_KIND_AUTO / _I8 / _F16 (B = 16 always runs kind::i8); umma_default_kind = what AUTO picks
int umma_default_kind(const Geom &g);
size_t umma_opA_bytes(const Geom &g, int64_t j0, int64_t j1, int num_sms, int kind, int n_images = 1);
size_t umma_opB_bytes(const Geom &g, int kind, int n_images = 1);
// device table: sweep position -> domain index (-1: padding), valid after a launch; probe only
void umma_debug_positions(const Work &w, const Geom &g, int64_t rows, int num_sms, int kind,
                          const int32_t **d_pos_dom, int64_t *npos);
// k0 / k1 (optional): events recorded around the search kernel.  pair: FIC_UMMA_PAIR_AUTO / _ON / _OFF; *pair_used
// (optional) = 1 if the CTA-pair kernel ran.  dump (optional, probe / self-test): every accumulator (kov) of every
// (operand row, sweep position) pair, row stride dump_ld; status_dev (optional, mapped host memory): the code of a
// pipeline wait that timed out.  n_images (1 to 256): a group of same-size images searched as one block-diagonal
// problem -- ranges [j0, j1) of every image, each against its own pool, in one pool sort, one pack of either operand,
// one search kernel and one refine; workspace (w.src, w.dec, w.dsum, w.dsq, w.rsum, w.dec3) holds the group back to
// back as the pool builders write it, w.best is [n][NR], opA / opB are sized with the same n_images.
int launch_search_umma(const Work &w, const Geom &g, int64_t j0, int64_t j1, int num_sms,
                       cudaStream_t s, const char **err, int kind, cudaEvent_t k0 = nullptr,
                       cudaEvent_t k1 = nullptr, int pair = FIC_UMMA_PAIR_AUTO, int *pair_used = nullptr,
                       int32_t *dump = nullptr, int64_t dump_ld = 0, int *status_dev = nullptr, int n_images = 1);

// ---- decoder (fic_decode.cu) -----------------------------------------------------------------------------------------
// Outcome of a decoder entry.  rc: FIC_OK; FIC_E_STREAM when a code indexes outside the domain pool (the reference
// throws ArrayIndexOutOfBounds); FIC_E_CUDA when `call` (file:line) returned `cuda`.
struct DecodeStatus {
    int rc = FIC_OK;
    cudaError_t cuda = cudaSuccess;
    const char *call = nullptr, *file = nullptr;
    int line = 0;
};

// Iterative decode (FC:355-420) of the codes at d_q into the device planes d_img, also copied to argb_out (host ARGB) or
// planes_out (host planes) when given.  avg_error (optional): in, the avgError the last decode left (FC:20); out, this
// decode's.  tm: total_ms from ev0 (recorded by the caller) to end, and launches.  h_scratch: pinned, sizeof(DecodeState).
// Workspace: dcode, dec, dec2, state, perr (W*H ints), replay (decode_replay_bytes(W*H)) and, with argb_out, argb.
DecodeStatus decode_run(const Work &w, const Geom &g, const int32_t *d_q, uint8_t *d_img, int32_t *argb_out,
                        uint8_t *planes_out, int max_iters, float *avg_error, int *iterations, void *h_scratch,
                        cudaEvent_t ev0, cudaEvent_t end, fic_timings *tm, cudaStream_t s);
// One collage step (FC:268-280): the float codes in w.info applied once to the source's codebook w.dec over an image of
// 0xa0 pixels; the image to argb_out, the codes with codebook indices (FC:888) to info_out.  Also uses dcode, img, argb.
DecodeStatus collage_run(const Work &w, const Geom &g, int32_t *argb_out, float *info_out, void *h_scratch, cudaStream_t s);
// *sum = carry + terms[0] + ... + terms[count - 1] in binary32, in order, as the last sweep of a decode over `count`
// pixels folds it (terms in [0, 3 * 255^2]).  Workspace: perr (count ints), state, replay (decode_replay_bytes(count)).
DecodeStatus decode_float_sum(const Work &w, const int32_t *terms, int64_t count, float carry, void *h_scratch, float *sum,
                              cudaStream_t s);
// Device workspace of the chunked replay of a sweep over `pixels` pixels (0: the one-warp replay needs none).
size_t decode_replay_bytes(int64_t pixels);

// Batch decode (fic_decode_batch): images per cooperative launch of the one-launch decoder for geometry g, 0 when g
// decodes image by image (decode_run).  At most kDecodeBatchMax.
constexpr int kDecodeBatchMax = 2048;
int decode_batch_group(const Geom &g);
// n images, codes [n][NR][S] at host `qcodes`, the decoded images to argb_out [n][H][W] or planes_out [n][C][H][W]; avg_error
// (optional) [n]: in, each image's carry; out, each image's avgError; iterations (optional) [n].  group =
// decode_batch_group(g).  Workspace: q, dcode, img, dec, dec2, argb (with argb_out) for `group` images (1 if 0),
// state for group (DecodeState + float carry), and what decode_run needs for one image.  h_stage: pinned, >= group *
// sizeof(DecodeState); h_scratch as decode_run's.  On FIC_E_STREAM *bad_image is the lowest image whose codes index
// outside the pool.
DecodeStatus decode_batch_run(const Work &w, const Geom &g, int n, int group, const int32_t *qcodes, int32_t *argb_out,
                              uint8_t *planes_out, int max_iters, float *avg_error, int *iterations, void *h_stage,
                              void *h_scratch, cudaEvent_t ev0, cudaEvent_t end, fic_timings *tm, int *bad_image, cudaStream_t s);

}  // namespace fic
