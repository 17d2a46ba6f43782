// fic_internal.h -- shared host/device declarations of libfic_b200 (not part of the ABI).
#pragma once

#include <cuda_runtime.h>
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
    float *avgf = nullptr;      // 1 float: running avgError for the exact replay kernel
    float *dcode = nullptr;     // [NR][3|5] dequantised codes with codebook indices, then s32 doff[NR] (domain byte offsets)
    int32_t *perr = nullptr;    // per-pixel squared change in reference loop order (exact avgError path)
    unsigned long long *acc = nullptr;  // [64] integer accumulators / flags
    uint16_t *dec3 = nullptr;   // RGB: R + G + B of the decimated planes (CUDA-core search)
    uint8_t *replay = nullptr;  // decoder, large images: per-chunk records of the exact avgError replay
    size_t cap[20] = {0};
};

// ---- kernel launchers (each returns the number of kernels it launched) -----------
int launch_unpack(const int32_t *d_argb, uint8_t *d_planes, int W, int H, int C, cudaStream_t s);
int launch_pack_argb(const uint8_t *d_planes, int32_t *d_argb, int W, int H, int C, cudaStream_t s);
int launch_decimate(const uint8_t *d_src, uint8_t *d_dec, const Geom &g, cudaStream_t s);
int launch_domain_stats(const uint8_t *d_dec, int32_t *d_dsum, int32_t *d_dsq, const Geom &g,
                        cudaStream_t s);
int launch_range_stats(const uint8_t *d_src, int32_t *d_rsum, const Geom &g, cudaStream_t s);
int launch_sum_planes(const uint8_t *d_dec, uint16_t *d_dec3, const Geom &g, cudaStream_t s);  // RGB only
int launch_search_direct(const Work &w, const Geom &g, int64_t j0, int64_t j1, cudaStream_t s);
// Fused windowed encode (widthKernel <= 16, no isometries): decimation, stats, search, solve and quantisation in one
// launch, straight from the caller's pixels (ARGB ints or 8-bit planes); no intermediate arrays.
bool fused_encode_applicable(const Geom &g);
int launch_encode_fused(const void *d_src, int src_is_argb, const Geom &g, int64_t j0, int64_t j1, float *d_info,
                        int32_t *d_q, cudaStream_t s);
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
size_t umma_opA_bytes(const Geom &g, int64_t j0, int64_t j1, int num_sms, int kind);
size_t umma_opB_bytes(const Geom &g, int kind);
// device table: sweep position -> domain index (-1: padding), valid after a launch; probe only
void umma_debug_positions(const Work &w, const Geom &g, int64_t rows, int num_sms, int kind,
                          const int32_t **d_pos_dom, int64_t *npos);
// k0 / k1 (optional): events recorded around the search kernel.  pair: FIC_UMMA_PAIR_AUTO / _ON / _OFF; *pair_used
// (optional) = 1 if the CTA-pair kernel ran.  dump (optional, probe / self-test): every accumulator (kov) of every
// (operand row, sweep position) pair, row stride dump_ld; status_dev (optional, mapped host memory): the code of a
// pipeline wait that timed out.
int launch_search_umma(const Work &w, const Geom &g, int64_t j0, int64_t j1, int num_sms,
                       cudaStream_t s, const char **err, int kind, cudaEvent_t k0 = nullptr,
                       cudaEvent_t k1 = nullptr, int pair = FIC_UMMA_PAIR_AUTO, int *pair_used = nullptr,
                       int32_t *dump = nullptr, int64_t dump_ld = 0, int *status_dev = nullptr);

// decoder
int launch_dequant(const int32_t *d_q, float *d_code, int32_t *d_off, const Geom &g, int unquantised,
                   const float *d_info, unsigned long long *d_acc, int packed, cudaStream_t s);
int launch_fill(uint8_t *d_planes, size_t bytes, int value, cudaStream_t s);
// Control block of one decoder sweep.  st == nullptr: a plain sweep (the one-shot collage).  Otherwise st points at
// the decoder state (fic_kernels.cu, "Decoder state block"): the sweep returns at once when the done flag is set,
// adds its squared pixel changes to st[0] and, with finish != 0, its last CTA folds the sweep into the state
// (avgError, iteration count, done flag; FC:413-417) so that the host need not look at every sweep.
struct SweepCtl {
    unsigned long long *st;
    int it;      // sweep index (FC:381 counter)
    int finish;  // 1: fold inside the sweep kernel -- only when the float sum needs no replay (see k_sweep_finish)
    float fwh;   // (float)(W*H), FC:413
};
// first (only where decode_sweep_has_first(g)): the sweep starts from the constant-128 image (FC:360) and reads nothing
// interleaved (only where decode_sweep_interleaved(g)): decoder loop over the row-pair interleaved decimated plane
// (k_decode_sweep_il); d_off then holds packed positions (launch_dequant with packed = 1)
int launch_decode_sweep(const uint8_t *d_dec_in, uint8_t *d_img, uint8_t *d_dec_out,
                        const float *d_code, const int32_t *d_off, const Geom &g,
                        const SweepCtl &ctl, int32_t *d_perr, int first, int interleaved, cudaStream_t s);
bool decode_sweep_has_first(const Geom &g);
// Small images (<= 2^20 pixels, interleaved-plane geometry): dequantisation, every sweep, the convergence rule and the
// ARGB conversion (d_argb may be null) in ONE cooperative launch.  Returns 1 if launched: the state block (zero on
// entry) then holds done / sweeps / avgError as after the per-sweep kernels, or word 9 != 0 = "bailed: repeat through the
// per-sweep kernels" (a float avgError sum that would need a replay).  0: not taken (geometry, device).
int launch_decode_small(const int32_t *d_q, float *d_code, int32_t *d_pos, uint8_t *d_img, uint8_t *d_dec_a, uint8_t *d_dec_b,
                        int32_t *d_argb, const Geom &g, unsigned long long *d_state, int max_iters, float carry, float fwh,
                        cudaStream_t s);
bool decode_sweep_interleaved(const Geom &g);
// folds a sweep whose float running sum may have to be replayed in loop order (see k_sweep_finish)
// d_workspace: sweep_finish_workspace(count) bytes (0 for small images: one warp replays the sum literally)
int launch_sweep_finish(const int32_t *d_perr, int64_t count, unsigned long long *d_state, int it, int last,
                        float carry, float fwh, void *d_workspace, cudaStream_t s);
size_t sweep_finish_workspace(int64_t count);

}  // namespace fic
