// fic_internal.h -- shared host/device declarations of libfic_b200 (not part of the ABI).
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/fic_b200.h"

namespace fic {

// Outcome of an encoder (fic_encode.cu) or decoder (fic_decode.cu) entry.  rc: FIC_OK or a FIC_E_* code; msg: the
// message for fic_last_error, or "" where the caller words it (a decoder's FIC_E_STREAM: a code indexes outside the
// domain pool).
struct Status {
    int rc;
    char msg[512];
    explicit Status(int code = FIC_OK) : rc(code) { msg[0] = 0; }
};
// A Status with code rc and a printf-style message (fic_api.cu).
Status fail(int rc, const char *fmt, ...) __attribute__((format(printf, 2, 3)));

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
    // quadtree extension (fic_quadtree.cu)
    uint8_t *qt_stream = nullptr;  // stream body: encode, written by k_qt_decide / k_qt_scatter; decode, the caller's stream
    int32_t *qt_codes = nullptr;   // encode: every level's quantised codes [NR_L][3|5], level after level (QtGeom::first)
    uint32_t *qt_err = nullptr;    // encode: leaf total, per-top-block leaf prefixes, per-warp totals, collage errors
    int4 *qt_leaf = nullptr;       // decode, per leaf: grey {a, b, domain byte offset, log2 blockgroesse}; RGB two records,
                                   // {a, bR, bG, bB} and {domain byte offset, log2 blockgroesse, 0, 0}
    int32_t *qt_map = nullptr;     // decode: leaf of every b_min x b_min cell, then the first leaf of every top block
    int64_t *qt_keys = nullptr;    // budget encode: every image's allowed splits K, then its effective keys (qt_nodes each)
    size_t cap[24] = {0};
};

enum Slot { S_ARGB, S_SRC, S_DEC, S_DSUM, S_DSQ, S_RSUM, S_BEST, S_INFO, S_Q, S_OPA, S_OPB, S_IMG, S_DEC2, S_DCODE, S_PERR, S_STATE, S_DEC3, S_REPLAY, S_QT_STREAM, S_QT_CODES,
            S_QT_ERR, S_QT_LEAF, S_QT_MAP, S_QT_KEYS };

// Grows workspace buffer p (its capacity is w.cap[slot]) to at least `bytes`; never shrinks it.
template <typename T>
Status ensure(Work &w, T *&p, int slot, size_t bytes)
{
    if (bytes == 0) bytes = 16;
    if (w.cap[slot] >= bytes && p) return Status();
    if (p) cudaFree(p);
    p = nullptr;
    w.cap[slot] = 0;
    size_t want = (bytes + 255) & ~(size_t)255;
    cudaError_t e = cudaMalloc((void **)&p, want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(FIC_E_NOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
    }
    w.cap[slot] = want;
    return Status();
}

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

// ---- encoder host side (fic_encode.cu) --------------------------------------------------------------------------------
// Per-handle encoder state: the options that choose an engine, what the last tcgen05 search did, and the events a run
// records around its stages (created and destroyed with the handle).
struct Encoder {
    int engine_opt = FIC_ENGINE_AUTO;    // FIC_OPT_ENGINE
    int umma_kind = FIC_UMMA_KIND_AUTO;  // FIC_OPT_UMMA_KIND
    int umma_pair = FIC_UMMA_PAIR_AUTO;  // FIC_OPT_UMMA_PAIR
    int pair_used = 0;                   // did the last tcgen05 search run the CTA-pair kernel
    int f16_state = 0;  // kind::f16 self-test: 0 not run yet, 1 exact, -1 not exact on this device (use kind::i8)
    int num_sms = 0;
    int run_engine = FIC_ENGINE_DIRECT;  // engine of the last run: which of the stage events it recorded
    cudaEvent_t ev[6] = {nullptr};
};

// What an encode call runs: the engine (FIC_ENGINE_DIRECT / _UMMA / _FUSED), the tcgen05 instruction kind, and the most
// images one run takes (1 unless a batch).
struct EncodePlan {
    int engine, kind, group;
};

// The plan for ranges [j0, j1) of n_images images of geometry g whose pixels arrive as ARGB ints (argb) or 8-bit planes;
// n_images = 1 is a single image or range slice, more is a batch (j0 = 0, j1 = NR).  FIC_E_ARG when the forced engine
// does not apply.  Runs the kind::f16 self-test on stream s the first time a plan would use kind::f16.
Status plan_encode(Encoder &e, const Geom &g, int64_t j0, int64_t j1, int n_images, bool argb, cudaStream_t s,
                   EncodePlan *plan);
// Runs plan p on device-resident pixels (ARGB ints or 8-bit planes, n_images <= p.group images back to back): ranges
// [j0, j1) of one image, or every range of a group (codes in [n][NR] tables).  Sizes its workspace in w, records the stage
// events, and adds engine, launches and search_evals to *tm.
Status run_encode(Encoder &e, Work &w, const Geom &g, const EncodePlan &p, const void *d_pixels, bool argb, int64_t j0,
                  int64_t j1, int n_images, float *d_info, int32_t *d_q, fic_timings *tm, cudaStream_t s);
// Whether the last run's events have completed.
bool run_done(const Encoder &e);
// Adds the last run's stage times (its events must have completed) to pool_ms, search_ms, kernel_ms and solve_ms of
// *acc, and sets total_ms = begin -> end.  begin: the call's start event (then h2d_ms = begin -> the run's start), or null
// for the run's start; end: the call's end event (then d2h_ms = the run's end -> end), or null for the run's end.
void read_stages(const Encoder &e, fic_timings *acc, cudaEvent_t begin, cudaEvent_t end);
// The kind::f16 self-test of the handle's device, run once per handle (Encoder::f16_state); FIC_E_CUDA if it cannot run.
Status f16_selftest(Encoder &e, cudaStream_t s);

// ---- decoder (fic_decode.cu) -----------------------------------------------------------------------------------------
// Decoder entries return FIC_E_STREAM with no message when a code indexes outside the domain pool (the reference throws
// ArrayIndexOutOfBounds).

// Iterative decode (FC:355-420) of the codes at d_q into the device planes d_img, also copied to argb_out (host ARGB) or
// planes_out (host planes) when given.  avg_error (optional): in, the avgError the last decode left (FC:20); out, this
// decode's.  tm: total_ms from ev0 (recorded by the caller) to end, and launches.  h_scratch: pinned, sizeof(DecodeState).
// Workspace: dcode, dec, dec2, state, perr (W*H ints), replay (decode_replay_bytes(W*H)) and, with argb_out, argb.
Status decode_run(const Work &w, const Geom &g, const int32_t *d_q, uint8_t *d_img, int32_t *argb_out,
                        uint8_t *planes_out, int max_iters, float *avg_error, int *iterations, void *h_scratch,
                        cudaEvent_t ev0, cudaEvent_t end, fic_timings *tm, cudaStream_t s);
// One collage step (FC:268-280): the float codes in w.info applied once to the source's codebook w.dec over an image of
// 0xa0 pixels; the image to argb_out, the codes with codebook indices (FC:888) to info_out.  Also uses dcode, img, argb.
Status collage_run(const Work &w, const Geom &g, int32_t *argb_out, float *info_out, void *h_scratch, cudaStream_t s);
// *sum = carry + terms[0] + ... + terms[count - 1] in binary32, in order, as the last sweep of a decode over `count`
// pixels folds it (terms in [0, 3 * 255^2]).  Workspace: perr (count ints), state, replay (decode_replay_bytes(count)).
Status decode_float_sum(const Work &w, const int32_t *terms, int64_t count, float carry, void *h_scratch, float *sum,
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
Status decode_batch_run(const Work &w, const Geom &g, int n, int group, const int32_t *qcodes, int32_t *argb_out,
                              uint8_t *planes_out, int max_iters, float *avg_error, int *iterations, void *h_stage,
                              void *h_scratch, cudaEvent_t ev0, cudaEvent_t end, fic_timings *tm, int *bad_image, cudaStream_t s);

// ---- quadtree extension (FIC_MODE_GREY_QT, FIC_MODE_RGB_QT; fic_quadtree.cu) ----------------------------------------
// Levels L = 0 .. nl - 1 of blockgroesse b_max >> L over one grey or RGB image, each with its own Geom (widthKernel wk,
// or the level's whole pool when wk == 0); the Geoms carry the channel count (Geom::C: 1 grey, 3 RGB).  Top blocks are
// the level-0 range blocks; every per-level table is level-major with level L starting at first[L].
constexpr int kQtMaxLevels = 3;
struct QtGeom {
    int nl;
    int wk;                      // as in the stream header: 0 = every level's whole pool
    Geom g[kQtMaxLevels];
    int64_t first[kQtMaxLevels];
    int64_t codes;               // sum of NR_L
    int64_t flag_bytes;          // NR_top padded to a multiple of 4
    int64_t leaves;              // n_leaves (decode: from the header)
};
constexpr size_t kQtHeaderBytes = 32;
// mode: FIC_MODE_GREY_QT or FIC_MODE_RGB_QT.  FIC_E_ARG (with *why) unless b_max in {8, 16}, b_min in {4, 8, 16},
// b_min <= b_max, wk >= 0 (0: W == H) and every level passes make_geom.
int qt_geom(int mode, int W, int H, int b_max, int b_min, int wk, QtGeom *q, const char **why);
// Bytes per leaf in the stream: 12 ({c, qa, qb}) grey, 20 ({c, qa, qbR, qbG, qbB}) RGB.
size_t qt_leaf_bytes(const QtGeom &q);
// Largest stream of the mode and geometry (every block split to b_min); 0 for non-positive arguments.
size_t qt_stream_bound(int mode, int W, int H, int b_max, int b_min);
// Header (its first int must be `mode`), flags and size of a stream (FIC_E_STREAM with *why otherwise); base (optional,
// NR_top entries): the first leaf of every top block.  check_leaves: also every leaf's domain index against its level's
// pool.
int qt_parse(int mode, const uint8_t *stream, size_t nbytes, QtGeom *q, int32_t *base, bool check_leaves, const char **why);
// Words of Work::qt_err an encode of a group of n images needs; its first qt_head_words(n): [0] the group's leaf total,
// [2, 2 + 2n) every image's max_mse as a double (budget form); image i's first leaf sits at
// w.qt_err[qt_starts_at(q, n) + i * ceil(flag_bytes / 32)].
size_t qt_err_words(const QtGeom &q, int n);
size_t qt_head_words(int n);
size_t qt_starts_at(const QtGeom &q, int n);
// Split-capable nodes of one image (blocks above b_min): NR_top, 5 NR_top when b_min is two levels down, 0 for one level.
int64_t qt_nodes(const QtGeom &q);
// Splits a stream of at most max_bytes can hold, K = (max_bytes - 32 - flag_bytes - leaf_bytes * NR_top) / (3 * leaf_bytes)
// (capped at INT64_MAX), or -1 when max_bytes is below the unsplit tree's size.
int64_t qt_budget_splits(const QtGeom &q, size_t max_bytes);
// Bytes of one image's stream body on the device (flags and the most leaves it can have): the stream bound less the header.
size_t qt_body_bytes(const QtGeom &q);
// A group of n images (planes [n][C][H][W] in w.src, decimated planes [n][C][sh][sw] in w.dec, every level's codes in
// w.qt_codes level-major and image-major: level L of image i at first[L] * n + i * NR_L): collage errors, split flags,
// leaf scan and leaf scatter into image i's body at w.qt_stream + i * qt_body_bytes (flags at 0, leaves at flag_bytes).
// The group's leaf total lands in w.qt_err[0] and image i's first leaf (counted over the group) as qt_err_words says.
// n = 1 runs the single-image kernels.  budget: max_mse is ignored; image i's is the smallest double whose tree needs at
// most w.qt_keys[i] splits (qt_budget_splits), found on the device from the collage errors (the keys after the n counts
// in w.qt_keys, n * qt_nodes words) and left in the qt_err head.
int launch_qt_stream(const Work &w, const QtGeom &q, int n, double max_mse, bool budget, cudaStream_t s);
// Iterative decode of n streams of one geometry into w.img (C planes per image), copied to planes_out [n][C][H][W].
// w.qt_stream holds the n images' flag bytes back to back and then every leaf of the group, image after image; w.qt_map
// holds n cell maps and then n first-leaf tables (NR_top entries each, counted over the group).  Each image's avgError =
// (float)S / (float)(W*H) of the exact sum S of its squared changes over pixels and channels; an image stops below 1 and
// stays frozen while the others sweep, all stop after max_iters sweeps.  avg_error and iterations ([n]) may be NULL.
// h_stage: pinned, n * sizeof(DecodeState).  Workspace: img, dec, dec2 (C planes per image), state (n blocks), qt_leaf
// (the group's leaves, two int4 each for RGB), qt_map.  On FIC_E_STREAM *bad_image is the lowest image with a leaf
// outside its level's pool.  Adds its launches to tm; total_ms runs from ev0 to end.
Status decode_quadtree_run(const Work &w, const QtGeom &q, int n, int max_iters, uint8_t *planes_out, float *avg_error,
                           int *iterations, void *h_stage, cudaEvent_t ev0, cudaEvent_t end, fic_timings *tm,
                           int *bad_image, cudaStream_t s);
// Exclusive prefix sums of n counters in place (one block, the radix sort's row scan); *total = their sum.
int launch_scan_u32(uint32_t *d, int64_t n, uint32_t *total, cudaStream_t s);

}  // namespace fic
