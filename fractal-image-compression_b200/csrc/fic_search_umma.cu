// fic_search_umma.cu -- K2+K3: the full-pool range x domain search as an exact integer
// contraction on the 5th-generation tensor cores (tcgen05, accumulators in TMEM), with the
// scoring / argmin filter fused into the epilogue so that no score matrix is ever written to
// HBM.  sm_100a only.
//
// What is computed.  For range block i and domain block j the reference scores
//     error = vR^2 * (1 - (kov / (vR * sqrt(varD)))^2)          (FC:677-683)
// with the exact integers kov = sum (r - rmean)(d - dmean), vR = sum (r - rmean) and
// varD = sum (d - dmean)^2, and keeps the first index with the smallest float error
// (strict <, ascending loop, FC:619-632).  Every rounding step of that expression is
// monotone, so error is a non-increasing function of x = |kov| / sqrt(varD), and the set T
// of candidates that reach the minimal float error is { j : x_j >= x_lo } for some x_lo
// within a relative 2^-20 (and an absolute 2^-21 in (x/vR)^2, the resolution of 1 - r^2)
// of the row maximum.  The reference's answer is the lowest index in T.
//
//   1. The tensor cores produce kov[i][j] exactly (two instruction kinds, below).
//   2. The fused epilogue needs no per-candidate floating point: domains are swept in
//      order of increasing varD, so every 32-column chunk of an accumulator shares the
//      scale 1/sqrt(varD) up to a tiny spread [rlo, rhi].  A thread takes the exact
//      max |kov| of its row over the chunk, and with M = max |kov|:
//      M*rhi bounds every x of the chunk from above, M*rlo bounds the row maximum from
//      below.  A chunk is flagged when M*rhi exceeds the row's threshold
//      thresh^2 = lb_max^2 * (1 - 2^-19) - vR^2 * 2^-21  (lb_max = running max of M*rlo),
//      i.e. whenever it could contain a member of T.  Flags are rare (O(log N) per row).
//   3. A refine kernel evaluates every candidate of every flagged chunk with the
//      reference's own float/double expression and takes the lexicographic (error, index)
//      minimum -- over a superset of T that is exactly the reference's winner.
// Result: the same winner index as the reference for every row, bit for bit, in any sweep
// order.
//
// kov on the tensor cores, kind::f16 (B = 4, 8).  A row = (r - rmean), B row = (d - dmean), both as
// binary16: integers of magnitude <= 255 are exact, every product and every partial sum is an integer
// below n * 127.5^2 = 1.04e6 (Cauchy-Schwarz; n = 64) << 2^24, so the binary32 accumulator holds kov
// exactly whatever the summation order (the probe dumps and checks every accumulator).  K = n.
// The epilogue takes max |kov| with FMNMX3 |a|, |b|, |c|: 16 instructions per 32 values.
//
// RGB (kind::f16 only).  The reference's RGB score has the same shape with the channel-summed centred
// values gR, gD in [-765, 765] as operands and the integer vD = sum gD in the place of sqrt(varD); its covariance
// is provably an exact integer below 2^24 for B <= 8, and at B = 16 the chunk bounds are widened by the worst-case
// rounding of the float sums.  Same kernel, RGB packers and refine: see "RGB operands".
//
// kov on the tensor cores, kind::i8 (B = 16; selectable for B = 4, 8).  With dt = d - dmean_j
// (|dt| <= 255; +255 only occurs in a block of mean 0, whose row is stored negated -- only |kov| is used),
// split dt = h + l, h = clamp(dt, -128, 127), l = dt - h (both fit s8; l is zero unless a
// pixel is more than 127 grey levels from its block mean, so the MMA issuer skips the l
// K-slices of every domain tile whose `l` digits are all zero -- most tiles).  Then
//     kov = sum_k r_k * h_k + sum_k r_k * l_k + rmean_i * (-alpha_j),   alpha_j = sum d - n*dmean_j
// i.e. A row = [ r | r | rmean x3 0.. ] (u8) and B row = [ h | l | -alpha in three parts 0.. ] (s8), K
// padded to a multiple of 32 (one kind::i8 MMA consumes K = 32).  The duplicated `r`
// half of A is not stored twice: the MMA issuer points the A descriptor of the `l` K-slices
// back at the `r` slices.  The s32 accumulator IS kov; max |kov| needs a max and a min chain
// (32 VIMNMX3 per 32 values), which is why kind::f16 wins where the epilogue is the bottleneck.
//
// Data movement.  Operands are packed once per encode by two HBM-bound kernels into
// "blobs" that are already in the canonical no-swizzle K-major UMMA shared-memory
// layout (8x16-byte core matrices, LBO = 128 B between K-adjacent core matrices,
// SBO = KS*256 B between 8-row groups).  A blob is moved with ONE 1-D TMA bulk copy
// (cp.async.bulk, SASS UBLKCP) that completes on an mbarrier; a domain tile blob also
// carries the (rhi, rlo) pair of each of its four 32-column chunks.  (B = 16: a tile is two
// blobs, high digits + bounds and low digits, see Cfg<16, false>.)
//
// Sweep order.  Sorted position sp holds domain perm[sp] (perm = domains by increasing
// varD, k_umma_sortkeys + the in-tree radix sort).  Sorted chunks (32 positions) are visited in
// a fixed pseudo-random order (sweep chunk P holds sorted chunk (P * mult) mod NCH), so
// the chunk maxima a row sees behave like an i.i.d. sequence: O(log N) records.
//
// CTA organisation (1 CTA / SM, 640 threads, persistent over work units):
//   warp 0      TMA producer: A super-block (512 range rows, resident for the whole
//               unit) + a ring of domain tiles (128 domains each)
//   warp 1      MMA issuer (warp-uniform loop, one elected lane issues): per domain tile
//               4 accumulators (128 rows x 128 domains = all 512 TMEM columns) x NS
//               K-slices of tcgen05.mma, tcgen05.commit -> t_full[q]; a second commit hands
//               the ring slot back to the producer (the epilogue never touches the ring)
//   warp 2      TMEM allocator
//   warps 4-19  epilogue: warp e owns TMEM lane quarter e % 4 of accumulator e / 4; one thread = one
//               range row, all 128 domains of a tile: per tile one t_full wait, four
//               tcgen05.ld.32x32b.x32, one hand-back (t_empty[q]); the tile's bounds come from
//               the blob in global memory at the top of each tile.  Rare paths (flag recording,
//               mbarrier polling) are out of line.  kind::f16, B <= 8: the four loads are software-pipelined
//               (epilogue loop epi_of<B, F16, PAIR>).
// A work unit is (super-block of 512 rows) x (1/n_chunks of the domain tiles); units are
// ordered chunk-major and a row's lower bound is carried from unit to unit (row_lb).  (RGB at B = 16:
// 256-row super-blocks, two of the four accumulators, Cfg<16, true>.)
//
// CTA pairs (kind::f16 at B = 8 by default; FIC_OPT_UMMA_PAIR): the kernel runs as clusters of two CTAs -- the two SMs
// of a TPC -- that share every tcgen05.mma (cta_group::2, M = 256, N = 128).  Each CTA keeps its own super-block
// (its 4 accumulators of 128 rows in its own TMEM) and supplies HALF of every domain tile, so the tensor pipe reads
// 96 instead of 128 bytes of operands per clock from an SM's shared memory (the single-CTA shape M = N = 128 asks for
// exactly the 128 B/clock an SM has, and the ring's TMA writes come on top), and the ring's L2 traffic halves.  A unit
// is (two adjacent super-blocks) x (1/n_chunks of the tiles).  CTA 0 issues -- from TWO warps (1 and 3: accumulators
// 0, 2 and 1, 3): the serial chain of one issuing thread (barrier wait, descriptor moves, four MMAs, commit: 250-300
// clocks per accumulator on a sub-partition it shares with four busy epilogue warps) was what kept the pair kernel at
// 1190 clocks per tile; with two issuers it runs at 1046 of an ideal 1024.  Commits are multicast to both CTAs'
// barriers; CTA 1's warp 1 relays "my half has landed" to CTA 0's full barriers, and CTA 1's epilogue warps hand
// accumulators back on CTA 0's t_empty barriers (remote mbarrier arrives).  The epilogue code is the same in both CTAs.
#include <cuda_fp16.h>

#include <cmath>
#include <mutex>
#include <tuple>
#include <vector>

#include "fic_device.cuh"

namespace fic {

namespace {

constexpr int kTileN = 128;        // domains per B tile == MMA N
constexpr int kBlockM = 128;       // rows per accumulator == MMA M
constexpr int kAccs = 4;           // accumulators per tile (TMEM: 4 x 128 columns)
constexpr int kRowsPerSB = kBlockM * kAccs;
constexpr int kEpiWarps = 16;
constexpr int kThreads = (4 + kEpiWarps) * 32;
constexpr int kChunksPerTile = kTileN / 32;
// per tile, behind the operand: (rhi, rlo) f32 per 32-column chunk, tile flags (u32 + pad), and per chunk an upper bound of
// the operand rows' Euclidean norms (RGB at blockgroesse 16 only: bounds the rounding of the float covariances)
constexpr int kBoundBytes = kChunksPerTile * 2 * 4 + 16 + kChunksPerTile * 4;
constexpr int kNormOff = kChunksPerTile * 2 * 4 + 16;     // offset of the norms inside the bounds area
// Flag lists of a (row, unit): two lists (column halves of the tiles, a historical split) of 32 entries each.
constexpr int kFlagLists = 2;
constexpr int kFlagCap = 32;
constexpr float kOneMinusEps = 1.0f - 1.9073486328125e-06f;  // 1 - 2^-19 (applied to the squared score)

// Operand geometry of one (block size, MMA kind) pair.  F16 = false: kind::i8, two s8 digits per
// centred domain pixel.  F16 = true: kind::f16, both operands centred and stored as binary16.
// A "K-slice" is the 32 bytes of K one tcgen05.mma consumes (32 i8 or 16 f16 elements).
template <int B, bool F16>
struct Cfg;
template <>
struct Cfg<8, false> {
    static constexpr int n = 64;
    static constexpr int NB = 4;     // 128-row accumulator blocks per super-block (A operand resident in shared memory)
    static constexpr bool KSPLIT = false;
    static constexpr int KS_A = 3;   // physical A K-slices: r[0:32] r[32:64] [rmean rmean 0..]
    static constexpr int KS_B = 5;   // h[0:32] h[32:64] l[0:32] l[32:64] [-alpha 0..]
    static constexpr int NS = 5;     // MMA K-slices
    static constexpr int NSTAGE = 7;
    __host__ __device__ static constexpr int amap(int s) { return s < 4 ? (s & 1) : 2; }
    __host__ __device__ static constexpr bool is_l_slice(int s) { return s == 2 || s == 3; }
};
template <>
struct Cfg<4, false> {
    static constexpr int n = 16;
    static constexpr int NB = 4;     // 128-row accumulator blocks per super-block (A operand resident in shared memory)
    static constexpr bool KSPLIT = false;
    static constexpr int KS_A = 2;   // [r r] [rmean 0..]
    static constexpr int KS_B = 2;   // [h l] [-alpha 0..]
    static constexpr int NS = 2;
    static constexpr int NSTAGE = 8;
    __host__ __device__ static constexpr int amap(int s) { return s; }
    __host__ __device__ static constexpr bool is_l_slice(int) { return false; }  // h and l share slice 0
};
template <>
struct Cfg<16, false> {
    static constexpr int n = 256;
    static constexpr int NB = 4;     // 128-row accumulator blocks per super-block (A operand resident in shared memory)
    // The A super-block (144 KB) leaves room for 72 KB of domain operands, not for two whole 68 KB tiles.  A tile
    // therefore travels as two parts, P0 = [h (8 slices) | -alpha (1 slice)] + the tile's bounds and P1 = [l (8
    // slices)], through a ring of two 36 KB slots: the copy of one part overlaps the MMAs on the other, and P1 is
    // neither copied nor multiplied when the tile's low digits are all zero.
    static constexpr bool KSPLIT = true;
    static constexpr int KS_P0 = 9, KS_P1 = 8;
    static constexpr int KS_A = 9;   // r[0:256] (8 slices) [rmean 0..]
    static constexpr int KS_B = 17;  // h (8 slices) l (8 slices) [-alpha 0..] (K-slices per tile, both parts)
    static constexpr int NS = 17;
    static constexpr int NSTAGE = 2; // part slots
    __host__ __device__ static constexpr int amap(int s) { return s < 16 ? (s & 7) : 8; }
    __host__ __device__ static constexpr bool is_l_slice(int s) { return s >= 8 && s < 16; }
};
template <>
struct Cfg<8, true> {
    static constexpr int n = 64;
    static constexpr int NB = 4;     // 128-row accumulator blocks per super-block (A operand resident in shared memory)
    static constexpr bool KSPLIT = false;
    static constexpr int KS_A = 4;   // (r - rmean)[0:64] as binary16: 4 slices of 16 elements
    static constexpr int KS_B = 4;   // (d - dmean)[0:64] as binary16
    static constexpr int NS = 4;
    static constexpr int NSTAGE = 8;
    __host__ __device__ static constexpr int amap(int s) { return s; }
    __host__ __device__ static constexpr bool is_l_slice(int) { return false; }
};
template <>
struct Cfg<4, true> {
    static constexpr int n = 16;
    static constexpr int NB = 4;     // 128-row accumulator blocks per super-block (A operand resident in shared memory)
    static constexpr bool KSPLIT = false;
    static constexpr int KS_A = 1;
    static constexpr int KS_B = 1;
    static constexpr int NS = 1;
    static constexpr int NSTAGE = 8;
    __host__ __device__ static constexpr int amap(int s) { return s; }
    __host__ __device__ static constexpr bool is_l_slice(int) { return false; }
};

template <>
struct Cfg<16, true> {
    // RGB at blockgroesse 16 (see "RGB operands"): K = 256 binary16 = 16 K-slices.  The A operand of 128 rows is 64 KB,
    // so a super-block holds TWO accumulator blocks (256 rows, 128 KB) and only two of the four TMEM accumulators are
    // used -- with 16 K-slices per accumulator (1024 clocks) a ring of two hides the hand-over.  The domain tile
    // (64 KB) travels as two parts of 8 K-slices through two 32 KB slots, like Cfg<16, false>; both parts always exist.
    static constexpr int n = 256;
    static constexpr int NB = 2;
    static constexpr bool KSPLIT = true;
    static constexpr int KS_P0 = 8, KS_P1 = 8;
    static constexpr int KS_A = 16;
    static constexpr int KS_B = 16;
    static constexpr int NS = 16;
    static constexpr int NSTAGE = 2;
    __host__ __device__ static constexpr int amap(int s) { return s; }
    __host__ __device__ static constexpr bool is_l_slice(int) { return false; }
};

template <class C>
constexpr int ksplit_p0()
{
    if constexpr (C::KSPLIT) return C::KS_P0;
    else return C::KS_B;
}

template <int B, bool F16>
struct Lay {
    using C = Cfg<B, F16>;
    static constexpr int SBO_A = C::KS_A * 256;
    static constexpr int A_BLOCK_BYTES = (kBlockM / 8) * SBO_A;
    static constexpr int ROWS_SB = C::NB * kBlockM;            // range rows of one super-block
    static constexpr int A_SB_BYTES = C::NB * A_BLOCK_BYTES;
    // Domain tile blob in global memory.  Unsplit: [operand, SBO_B between 8-row groups][bounds + flag].
    // Split (Cfg::KSPLIT): [part P0, SBO_B][bounds + flag][part P1, SBO_P1].  B_OP_BYTES is the offset of the bounds.
    static constexpr int KS0 = ksplit_p0<C>();
    static constexpr int SBO_B = KS0 * 256;
    static constexpr int SBO_P1 = (C::KS_B - KS0) * 256;
    static constexpr int B_OP_BYTES = (kTileN / 8) * SBO_B;
    static constexpr int P0_BYTES = B_OP_BYTES + kBoundBytes;
    static constexpr int P1_BYTES = (kTileN / 8) * SBO_P1;
    static constexpr int B_TILE_BYTES = P0_BYTES + P1_BYTES;
    static constexpr int SLOT_BYTES = C::KSPLIT ? ((P0_BYTES + 127) / 128) * 128 : B_TILE_BYTES;  // one ring entry in shared memory
    // CTA pairs (tcgen05 cta_group::2, see k_umma_search<..., PAIR>): each CTA of the pair holds HALF of every domain
    // tile (64 operand rows = the first / second 8 row groups of the blob), so the ring has twice the depth in the
    // same shared memory (capped: the barrier area holds 2 * 12 + 10 mbarriers).
    // K-split configurations: a slot takes half of either part (P0: 8 row groups x SBO_B, P1: 8 x SBO_P1).
    static constexpr int PAIR_P0_BYTES = B_OP_BYTES / 2, PAIR_P1_BYTES = P1_BYTES / 2;
    static constexpr int PAIR_SLOT_BYTES = PAIR_P0_BYTES > PAIR_P1_BYTES ? PAIR_P0_BYTES : PAIR_P1_BYTES;
    static constexpr int PAIR_STAGES = (C::NSTAGE * SLOT_BYTES) / PAIR_SLOT_BYTES < 12 ? (C::NSTAGE * SLOT_BYTES) / PAIR_SLOT_BYTES : 12;
    static constexpr int BAR_BYTES = 512;
    static constexpr int SMEM_BYTES = A_SB_BYTES + C::NSTAGE * SLOT_BYTES + 1024 /*alignment slack*/ + BAR_BYTES /*barriers*/ +
                                      kRowsPerSB * 4 /*per-row lower bound shared by the rows of a range block (isometry extension)*/;
};

// Flag threshold from the best lower bound lb of the row's max x = |kov| / sqrt(varD): candidates with
// x^2 <= lb^2 * (1 - 2^-19) - vR^2 * 2^-21 cannot reach the minimal float error.  A non-positive right-hand
// side means even x = 0 (kov == 0, flat domains) may tie with the best -> -1: everything is a candidate.
__device__ __noinline__ float flag_threshold(float lb, float tie_abs)  // rare path: kept out of the hot loops
{
    const float rad = lb * lb * kOneMinusEps - tie_abs;
    return rad > 0.0f ? sqrtf(rad) : -1.0f;
}

// Rare path of the search epilogue, out of line so that the hot loop stays short: record a flagged chunk -- its id
// and the upper bound ub of its scores, which lets the refine step drop the chunk once the row's final bound is
// known -- and, if it raises the row's lower bound, publish the bound (shared-memory slot `sh_lb`) and recompute the
// threshold.
// share != 0: publish a raised bound to `sh_lb` (isometry rows share one bound).
struct RowFilter { float thresh, lbmax; int cnt; };
__device__ __noinline__ RowFilter flag_chunk(RowFilter st, float lb, float ub, float tie_abs, int2 *list, int chunk_id,
                                             uint32_t sh_lb, int share)
{
    if (st.cnt < kFlagCap) list[st.cnt] = make_int2(chunk_id, __float_as_int(ub));
    st.cnt++;
    if (lb > st.lbmax) {
        st.lbmax = lb;
        if (share)  // positive floats order like their bits
            asm volatile("red.shared.max.u32 [%0], %1;" ::"r"(sh_lb), "r"(__float_as_uint(lb)) : "memory");
        const float rad = lb * lb * kOneMinusEps - tie_abs;
        st.thresh = rad > 0.0f ? sqrtf(rad) : -1.0f;
    }
    return st;
}

// ---------------------------------------------------------------- sweep order --------

// Sweep chunk P (32 positions) holds sorted chunk (P * mult) mod nch (mult coprime to nch).
__host__ __device__ __forceinline__ int64_t sweep_to_sorted(int64_t pos, uint32_t mult, int64_t nch)
{
    const uint64_t chunk = (uint64_t)pos >> 5;
    return (int64_t)(((chunk * (uint64_t)mult) % (uint64_t)nch) * 32 + ((uint64_t)pos & 31));
}

// Sort keys: varD of every domain (DB:106-115), payload: the domain index.  A group of n_img images ([n_img][ND]
// stats) keys domain j of image i as i << 24 | varD and carries the group-global index i * ND + j: a stable sort on
// four digits leaves every image's domains contiguous and in the order a single image's three-digit sort gives them.
__global__ void k_umma_sortkeys(const int32_t *__restrict__ dsum, const int32_t *__restrict__ dsq, int n,
                                int64_t ND, int64_t count, uint32_t *__restrict__ keys, int32_t *__restrict__ vals)
{
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    int dmean;
    keys[j] = (uint32_t)(j >= ND ? j / ND : 0) << 24 | (uint32_t)dom_var(dsum[j], dsq[j], n, &dmean);
    vals[j] = (int32_t)j;
}


// ---------------------------------------------------------------- radix sort ----------
//
// Stable LSD radix sort of (key, value) pairs on 24-bit keys, three passes of 8 bits, in-tree (no library kernel on
// the path).  The unit of work is a WARP owning kSortSub consecutive elements.  Per pass: k_sort_hist counts the
// warp's digits into the digit-major table hist[digit][warp]; k_sort_scan_rows (one block per digit) turns every row
// into exclusive prefixes and leaves the row total; k_sort_scatter adds the scan of the 256 totals and lets every
// warp walk its elements 32 at a time, ranking equal digits by lane order (__match_any_sync), so the order inside a
// digit is the input order.  About 0.1 ms for the 10^6 domains of a 4096^2 image.
constexpr int kSortSub = 512;  // elements per warp

__global__ void __launch_bounds__(256) k_sort_hist(const uint32_t *__restrict__ keys, int64_t n, int shift, int64_t nwarps,
                                                   uint32_t *__restrict__ hist)
{
    __shared__ uint32_t s_h[8][256];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t gw = (int64_t)blockIdx.x * 8 + warp;
    for (int d = lane; d < 256; d += 32) s_h[warp][d] = 0;
    __syncwarp();
    if (gw < nwarps) {
        const int64_t a = gw * kSortSub, b = a + kSortSub < n ? a + kSortSub : n;
        for (int64_t i = a + lane; i < b; i += 32) atomicAdd(&s_h[warp][(keys[i] >> shift) & 255u], 1u);
        __syncwarp();
        for (int d = lane; d < 256; d += 32) hist[(int64_t)d * nwarps + gw] = s_h[warp][d];
    }
}

// Block d: exclusive prefix sums along row d of the table (nwarps counters), in place; totals[d] = the row's sum.
__global__ void __launch_bounds__(256) k_sort_scan_rows(uint32_t *__restrict__ hist, int64_t nwarps, uint32_t *__restrict__ totals)
{
    __shared__ uint32_t s_warp[8];
    __shared__ uint32_t s_carry;
    uint32_t *row = hist + (int64_t)blockIdx.x * nwarps;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int64_t base = 0; base < nwarps; base += 256) {
        const int64_t i = base + threadIdx.x;
        const uint32_t c = i < nwarps ? row[i] : 0u;
        uint32_t incl = c;  // inclusive scan inside the warp
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        uint32_t before = s_carry;
        for (int w = 0; w < warp; w++) before += s_warp[w];
        if (i < nwarps) row[i] = before + incl - c;
        __syncthreads();
        if (threadIdx.x == 255) s_carry = before + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) totals[blockIdx.x] = s_carry;
}

__global__ void __launch_bounds__(256) k_sort_scatter(const uint32_t *__restrict__ keys, const int32_t *__restrict__ vals,
                                                      uint32_t *__restrict__ keys_out, int32_t *__restrict__ vals_out, int64_t n,
                                                      int shift, int64_t nwarps, const uint32_t *__restrict__ hist,
                                                      const uint32_t *__restrict__ totals)
{
    __shared__ uint32_t s_digit[256];    // first output slot of each digit (exclusive scan of the row totals)
    __shared__ uint32_t s_base[8][256];  // next output slot of each digit for this warp's elements
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t gw = (int64_t)blockIdx.x * 8 + warp;
    {
        const uint32_t c = totals[threadIdx.x];
        uint32_t incl = c;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        s_digit[threadIdx.x] = incl - c;
        if (lane == 31) s_base[0][warp] = incl;  // warp totals, parked in a row that is rewritten below
        __syncthreads();
        uint32_t before = 0;
        for (int w = 0; w < warp; w++) before += s_base[0][w];
        __syncthreads();
        s_digit[threadIdx.x] += before;
        __syncthreads();
    }
    if (gw >= nwarps) return;
    for (int d = lane; d < 256; d += 32) s_base[warp][d] = s_digit[d] + hist[(int64_t)d * nwarps + gw];
    __syncwarp();
    const int64_t a = gw * kSortSub, b = a + kSortSub < n ? a + kSortSub : n;
    for (int64_t i0 = a; i0 < b; i0 += 32) {
        const int64_t i = i0 + lane;
        const bool live = i < b;
        const uint32_t k = live ? keys[i] : 0u;
        const int32_t v = live ? vals[i] : 0;
        const uint32_t d = live ? ((k >> shift) & 255u) : 256u + lane;  // dead lanes match nobody
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const int rank = __popc(peers & ((1u << lane) - 1u));
        uint32_t base = 0;
        if (live) base = s_base[warp][d];
        __syncwarp();
        if (live) {
            keys_out[base + rank] = k;
            vals_out[base + rank] = v;
            if (rank == 0) s_base[warp][d] = base + __popc(peers);  // lowest lane of the digit group advances the slot
        }
        __syncwarp();
    }
}

// Sorts n pairs (keys0, vals0) by the low 8 * passes bits of the key; the result is in (keys1, vals1) for an odd
// number of passes, in (keys0, vals0) for an even one.  `hist` holds 256 * (ceil(n / kSortSub) + 1) counters (the
// table and the 256 row totals).  Returns the number of launches.
inline size_t sort_hist_bytes(int64_t n) { return (size_t)256 * (size_t)((n + kSortSub - 1) / kSortSub + 1) * 4; }

inline int launch_sort_pairs(uint32_t *keys0, int32_t *vals0, uint32_t *keys1, int32_t *vals1, uint32_t *hist, int64_t n,
                             int passes, cudaStream_t s)
{
    const int64_t nwarps = (n + kSortSub - 1) / kSortSub;
    const unsigned blocks = (unsigned)((nwarps + 7) / 8);
    uint32_t *totals = hist + 256 * nwarps;
    uint32_t *kin = keys0, *kout = keys1;
    int32_t *vin = vals0, *vout = vals1;
    for (int pass = 0; pass < passes; pass++) {
        k_sort_hist<<<blocks, 256, 0, s>>>(kin, n, 8 * pass, nwarps, hist);
        k_sort_scan_rows<<<256, 256, 0, s>>>(hist, nwarps, totals);
        k_sort_scatter<<<blocks, 256, 0, s>>>(kin, vin, kout, vout, n, 8 * pass, nwarps, hist, totals);
        uint32_t *tk = kin; kin = kout; kout = tk;
        int32_t *tv = vin; vin = vout; vout = tv;
    }
    return 3 * passes;
}

// ---------------------------------------------------------------- operand packing ----

__device__ __forceinline__ uint32_t pack4(int a, int b, int c, int d)
{
    return (uint32_t)(a & 0xff) | ((uint32_t)(b & 0xff) << 8) | ((uint32_t)(c & 0xff) << 16) | ((uint32_t)(d & 0xff) << 24);
}

// A group of images keeps one OpBLayout region per image, `stride` bytes apart: a pointer into image 0's region, moved
// to image i's.
template <class T>
__host__ __device__ __forceinline__ T *image_region(T *p, int64_t image, size_t stride)
{
    return (T *)((uint8_t *)const_cast<void *>((const void *)p) + (size_t)image * stride);
}

// Raw domain pixels for the refine step: per 32-position chunk, 16-byte piece c of position p sits at
// [chunk][c][p % 32], so a warp that evaluates one chunk reads 512 contiguous bytes per load.
template <int n>
__host__ __device__ __forceinline__ int64_t raw_offset(int64_t pos, int c)
{
    return (pos >> 5) * (32 * n) + c * 512 + (pos & 31) * 16;
}

// Two integers in [-255, 255] as a packed pair of binary16 (exact: |v| < 2048).
__device__ __forceinline__ uint32_t pack_h2(int lo, int hi)
{
    const __half2 v = __halves2half2(__int2half_rn(lo), __int2half_rn(hi));
    return *(const uint32_t *)&v;
}

// One thread per sweep position (a warp = one 32-position chunk): centre the domain by its
// integer mean, write the tile-blob row (kind::i8: two s8 digits + the -alpha columns; kind::f16:
// binary16), the position tables and the raw pixels used by the refine step, and the chunk's scale
// bounds.  A group of images: the grid covers npos positions per image (a block = one tile, inside one image); image i
// reads its planes / stats / slice of the group's sort and writes its own OpBLayout region, opb_stride bytes on.
template <int B, bool F16>
__global__ void __launch_bounds__(128)
k_umma_pack_domains(const uint8_t *__restrict__ dec, const int32_t *__restrict__ dsum,
                    const int32_t *__restrict__ dsq, const int32_t *__restrict__ perm, uint8_t *__restrict__ opB,
                    int32_t *__restrict__ pos_dom, int4 *__restrict__ pos_info,
                    uint8_t *__restrict__ pos_raw, int64_t *__restrict__ dom0_pos,
                    Geom g, int64_t ntiles, uint32_t mult, int64_t npos, size_t opb_stride)
{
    using L = Lay<B, F16>;
    constexpr int n = Cfg<B, F16>::n;
    const int64_t p0 = (int64_t)blockIdx.x * blockDim.x;  // (a single image divides nothing)
    const int64_t image = p0 >= npos ? p0 / npos : 0;
    const int64_t pos = p0 + threadIdx.x - image * npos;
    dec += image * g.sw * g.sh;
    dsum += image * g.ND;
    dsq += image * g.ND;
    perm += image * g.ND;
    opB = image_region(opB, image, opb_stride);
    pos_dom = image_region(pos_dom, image, opb_stride);
    pos_info = image_region(pos_info, image, opb_stride);
    pos_raw = image_region(pos_raw, image, opb_stride);
    dom0_pos = image_region(dom0_pos, image, opb_stride);
    const int64_t tile = pos / kTileN;
    const int row = (int)(pos % kTileN);
    const int64_t sp = sweep_to_sorted(pos, mult, ntiles * kChunksPerTile);
    constexpr bool KSPLIT = Cfg<B, F16>::KSPLIT;
    uint8_t *blob = opB + tile * L::B_TILE_BYTES;
    uint8_t *rowp = blob + (row >> 3) * L::SBO_B + (row & 7) * 16;
    // K-split tiles keep the low digits in a second part behind the bounds (see Lay)
    uint8_t *rowp1 = blob + L::P0_BYTES + (row >> 3) * L::SBO_P1 + (row & 7) * 16;
    constexpr int NCH = L::KS0 * 2;                              // 16-byte chunks per row (of part P0)
    constexpr int NCH1 = (Cfg<B, F16>::KS_B - L::KS0) * 2;      // ... of part P1
    float rsd_hi = 0.0f, rsd_lo = __int_as_float(0x7f800000);
    int any_l = 0;
    if (sp >= g.ND) {
#pragma unroll
        for (int c = 0; c < NCH; c++) *(uint4 *)(rowp + c * 128) = make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int c = 0; c < NCH1; c++) *(uint4 *)(rowp1 + c * 128) = make_uint4(0, 0, 0, 0);
        pos_dom[pos] = -1;
        pos_info[pos] = make_int4(-1, 0, 0, 0);
    } else {
        const int64_t j = perm[sp] - image * g.ND;  // the sort carries group-global indices
        const int gx = (int)(j % g.dpw), gy = (int)(j / g.dpw);
        const uint8_t *p = dec + (int64_t)(gy * g.step) * g.sw + gx * g.step;
        int dmean;
        const int varD = dom_var(dsum[j], dsq[j], n, &dmean);
        constexpr int PCH = n / 16;  // 16-pixel groups
        // kind::i8: dt = d - dmean reaches +255 only in a block of mean 0 (B = 16), one more than the two s8 digits
        // 127 + 127 hold, while -255 = -128 - 127 fits.  Such a row is stored negated: the accumulator becomes
        // -kov, and only |kov| is ever used (the refine step recomputes kov from the raw pixels).
        const int sgn = (!F16 && dmean == 0) ? -1 : 1;
        // B = 8, decimated rows of a multiple of 8 bytes: a block row is 8 bytes at an even column -- the aligned 8-byte
        // word that holds its start and, unless the column is a multiple of 8, the next one (inside the row: see below),
        // instead of four 2-byte loads.  The gather is what this kernel pays for: every lane reads another domain.
        const bool wide8 = B == 8 && (g.sw & 7) == 0;
        const int col8 = (gx * g.step) & 7;  // the next aligned word ends at most at the row's end when col8 != 0
#pragma unroll
        for (int c = 0; c < PCH; c++) {
            int dv[16];
            uint32_t raw[4];
            if (wide8) {
#pragma unroll
                for (int r2 = 0; r2 < 2; r2++) {  // 16 pixels = two block rows
                    const uint8_t *q = p + (int64_t)(c * 2 + r2) * g.sw - col8;
                    const uint2 lo = __ldg((const uint2 *)q);
                    uint2 hi = lo;
                    if (col8) hi = __ldg((const uint2 *)(q + 8));
                    const uint32_t sh = (uint32_t)(col8 & 3) * 8u;
                    const bool up = col8 >= 4;
                    raw[2 * r2] = __funnelshift_r(up ? lo.y : lo.x, up ? hi.x : lo.y, sh);
                    raw[2 * r2 + 1] = __funnelshift_r(up ? hi.x : lo.y, up ? hi.y : hi.x, sh);
                }
            }
#pragma unroll
            for (int w = 0; w < 4; w++) {
                // pixels k .. k + 3 of the block share a row; a block row starts at a multiple of B / 4 bytes of the
                // decimated plane: one 4-byte load for B = 16, two 2-byte loads for B = 8, bytes for B = 4
                const int k = c * 16 + w * 4;
                const uint8_t *q = p + (int64_t)(k / B) * g.sw + (k % B);
                if (B == 16) raw[w] = __ldg((const uint32_t *)q);
                else if (B == 8) {
                    if (!wide8) raw[w] = (uint32_t)__ldg((const uint16_t *)q) | ((uint32_t)__ldg((const uint16_t *)(q + 2)) << 16);
                } else raw[w] = (uint32_t)__ldg(q) | ((uint32_t)__ldg(q + 1) << 8) | ((uint32_t)__ldg(q + 2) << 16) | ((uint32_t)__ldg(q + 3) << 24);
#pragma unroll
                for (int e = 0; e < 4; e++) dv[w * 4 + e] = sgn * ((int)((raw[w] >> (8 * e)) & 0xffu) - dmean);
            }
            *(uint4 *)(pos_raw + raw_offset<n>(pos, c)) = make_uint4(raw[0], raw[1], raw[2], raw[3]);
            if (F16) {
                *(uint4 *)(rowp + (2 * c) * 128) =
                    make_uint4(pack_h2(dv[0], dv[1]), pack_h2(dv[2], dv[3]), pack_h2(dv[4], dv[5]), pack_h2(dv[6], dv[7]));
                *(uint4 *)(rowp + (2 * c + 1) * 128) = make_uint4(pack_h2(dv[8], dv[9]), pack_h2(dv[10], dv[11]),
                                                                  pack_h2(dv[12], dv[13]), pack_h2(dv[14], dv[15]));
            } else {
                uint32_t hw[4], lw[4];
#pragma unroll
                for (int w = 0; w < 4; w++) {
                    int hv[4], lv[4];
#pragma unroll
                    for (int e = 0; e < 4; e++) {
                        hv[e] = max(-128, min(127, dv[w * 4 + e]));  // the low digit is zero unless |dt| > 127
                        lv[e] = dv[w * 4 + e] - hv[e];
                        any_l |= lv[e];
                    }
                    hw[w] = pack4(hv[0], hv[1], hv[2], hv[3]);
                    lw[w] = pack4(lv[0], lv[1], lv[2], lv[3]);
                }
                *(uint4 *)(rowp + c * 128) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
                if (KSPLIT) *(uint4 *)(rowp1 + c * 128) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
                else *(uint4 *)(rowp + (PCH + c) * 128) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
            }
        }
        if (!F16) {
            // -alpha (times the row's sign) in three s8 columns (alpha <= n - 1 = 255 at B = 16: thirds fit either
            // sign); A carries rmean in all three
            const int alpha = sgn * (dsum[j] - n * dmean);
            const int a1 = alpha / 3, a2 = (alpha - a1) / 2, a3 = alpha - a1 - a2;
            constexpr int ACH = KSPLIT ? PCH : 2 * PCH;  // first 16-byte chunk of the alpha K-slice
            *(uint4 *)(rowp + ACH * 128) = make_uint4(
                (uint32_t)((-a1) & 0xff) | ((uint32_t)((-a2) & 0xff) << 8) | ((uint32_t)((-a3) & 0xff) << 16), 0, 0, 0);
            *(uint4 *)(rowp + (ACH + 1) * 128) = make_uint4(0, 0, 0, 0);
        }
        pos_dom[pos] = (int32_t)j;
        pos_info[pos] = make_int4((int32_t)j, varD, dsum[j], 0);  // what the refine step needs, in one 16-byte load
        if (j == 0) *dom0_pos = pos;  // the refine step always evaluates domain 0
        if (varD > 0) {  // flat domains have kov == 0: they never set a chunk's max |kov|
            float r = __double2float_rn(__ddiv_rn(1.0, __dsqrt_rn((double)varD)));
            rsd_hi = r * (1.0f + 4.76837158203125e-07f);  // >= 1/sqrt(varD) * (1 + 2^-22): covers r's and M*rhi's rounding
            rsd_lo = r * (1.0f - 4.76837158203125e-07f);  // <= 1/sqrt(varD) * (1 - 2^-22)
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        rsd_hi = fmaxf(rsd_hi, __shfl_xor_sync(0xffffffffu, rsd_hi, o));
        rsd_lo = fminf(rsd_lo, __shfl_xor_sync(0xffffffffu, rsd_lo, o));
    }
    if ((threadIdx.x & 31) == 0) {
        if (rsd_hi == 0.0f) rsd_lo = 0.0f;  // chunk of flat / padding columns only
        *(float2 *)(blob + L::B_OP_BYTES + (row >> 5) * 8) = make_float2(rsd_hi, rsd_lo);
    }
    // One block == one tile (blockDim == kTileN): does any column of the tile need its low digit?
    const int tile_has_l = __syncthreads_or(any_l != 0);
    if (threadIdx.x == 0) *(uint4 *)(blob + L::B_OP_BYTES + kChunksPerTile * 8) = make_uint4((uint32_t)tile_has_l, 0, 0, 0);
}

// One thread per (padded) operand row of the slice [j0, j1).  kind::i8: raw pixels + the integer mean
// columns; kind::f16: pixels centred by the integer mean, as binary16.  With the isometry extension
// (g.n_iso = 8) a range block owns 8 adjacent rows: row v = (j - j0) * 8 + k holds the block permuted so that
// its dot product with an unpermuted domain block is kov(r, T_k d) -- column p carries the range pixel that
// T_k maps onto domain pixel p.  Means and sums do not depend on k.  A group of images: image i owns the rows_padded
// operand rows (whole super-blocks) from i * rows_padded on, and reads its own planes and range sums.
template <int B, bool F16>
__global__ void __launch_bounds__(128)
k_umma_pack_ranges(const uint8_t *__restrict__ src, const int32_t *__restrict__ rsum, uint8_t *__restrict__ opA,
                   int32_t *__restrict__ vRout, Geom g, int64_t j0, int64_t j1, int64_t rows_padded, int n_img)
{
    using L = Lay<B, F16>;
    constexpr int n = Cfg<B, F16>::n;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows_padded * n_img) return;
    int64_t sb = i / L::ROWS_SB;
    int rr = (int)(i % L::ROWS_SB);
    int blk = rr / kBlockM, row = rr % kBlockM;
    uint8_t *rowp = opA + sb * L::A_SB_BYTES + blk * L::A_BLOCK_BYTES + (row >> 3) * L::SBO_A + (row & 7) * 16;
    constexpr int NCH = Cfg<B, F16>::KS_A * 2;
    const int64_t image = i >= rows_padded ? i / rows_padded : 0, il = i - image * rows_padded;
    src += image * g.W * g.H;
    rsum += image * g.NR;
    const int64_t j = j0 + il / g.n_iso;
    const int kiso = (int)(il % g.n_iso);
    if (j >= j1) {
#pragma unroll
        for (int c = 0; c < NCH; c++) *(uint4 *)(rowp + c * 128) = make_uint4(0, 0, 0, 0);
        vRout[i] = 0;
        return;
    }
    int xr = (int)(j % g.rpw), yr = (int)(j / g.rpw);
    const uint8_t *p = src + (int64_t)(yr * B) * g.W + xr * B;
    int rmean;
    vRout[i] = centred_sum(rsum[j], n, &rmean);
    constexpr int PCH = n / 16;
#pragma unroll
    for (int c = 0; c < PCH; c++) {
        uint32_t w4[4];
#pragma unroll
        for (int w = 0; w < 4; w++) {
            int k = c * 16 + w * 4;
            if (kiso == 0) {
                // 4 consecutive k share a pixel row for B >= 4; 4-byte aligned since xr*B, k%B are multiples of 4
                w4[w] = *(const uint32_t *)(p + (int64_t)(k / B) * g.W + (k % B));
            } else {
                w4[w] = 0;
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    int ry, rx;  // the range pixel that T_kiso sends to domain pixel k + e
                    iso_map(iso_inverse(kiso), B, (k + e) / B, (k + e) % B, &ry, &rx);
                    w4[w] |= (uint32_t)p[(int64_t)ry * g.W + rx] << (8 * e);
                }
            }
        }
        if (F16) {
            uint32_t hw[8];
#pragma unroll
            for (int w = 0; w < 4; w++) {
                hw[2 * w] = pack_h2((int)(w4[w] & 0xff) - rmean, (int)((w4[w] >> 8) & 0xff) - rmean);
                hw[2 * w + 1] = pack_h2((int)((w4[w] >> 16) & 0xff) - rmean, (int)(w4[w] >> 24) - rmean);
            }
            *(uint4 *)(rowp + (2 * c) * 128) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
            *(uint4 *)(rowp + (2 * c + 1) * 128) = make_uint4(hw[4], hw[5], hw[6], hw[7]);
        } else {
            uint4 v = make_uint4(w4[0], w4[1], w4[2], w4[3]);
            *(uint4 *)(rowp + c * 128) = v;
            if (B == 4) *(uint4 *)(rowp + (PCH + c) * 128) = v;  // [r r] shares one 32-byte slice
        }
    }
    if (!F16) {
        constexpr int XCH = (B == 4) ? 2 * PCH : PCH;
        *(uint4 *)(rowp + XCH * 128) = make_uint4((uint32_t)rmean | ((uint32_t)rmean << 8) | ((uint32_t)rmean << 16), 0, 0, 0);
        *(uint4 *)(rowp + (XCH + 1) * 128) = make_uint4(0, 0, 0, 0);
    }
}

// ---------------------------------------------------------------- RGB operands --------
//
// The reference's RGB score (FC:760-808) uses ONE covariance for the three channels,
//     kov = sum gR_i * gD_i,   gR_i = sum_c (r_ci - rmean_c),   gD_i = sum_c (d_ci - dmean_c),
// accumulated sequentially in binary32, and  r = kov / (vR * vD)  with the small integers vR = sum gR_i and
// vD = sum gD_i (FC:790-791; the domain's `variance` is never set on this path).  error = vR^2 (1 - r^2) is again a
// non-increasing function of x = |kov| / vD, so the grey machinery applies with sqrt(varD) := vD:
//   * operands gR, gD are integers in [-765, 765]: exact in binary16, kind::f16 only;
//   * a domain with vD == 0 has r = 0 whatever its kov (FC:797): its operand row is zeroed so that it scores x = 0;
//   * exactness for B <= 8.  A channel of a block, centred by its integer mean m = floor(mu), has
//     sum (v - m)^2 = sum (v - mu)^2 + n (mu - m)^2 <= n (127.5^2 + 1)   (values in [0, 255]: variance <= 127.5^2),
//     so ||gR||_2, ||gD||_2 <= 3 sqrt(n (127.5^2 + 1)) (triangle inequality over the channels), and by Cauchy-Schwarz
//     every partial sum of |gR_i gD_i| over any subset of the pixels is <= 9 n (127.5^2 + 1) = 9 364 176 < 2^24 at
//     n = 64.  Every partial sum of every summation order is therefore an integer below 2^24: the reference's
//     sequential float kov, the tensor-core accumulator and the refine step's FMA chain are the same exact integer
//     for every block (the bound 64 * 765^2 of a term-by-term estimate is not attained);
//   * B = 16: the same bound is 3.7e7 > 2^24.  On extreme-contrast content the reference's sequential float sum ROUNDS,
//     and what it ranks by is the rounded value kov_ref.  The tensor cores then act as a filter with honest bounds
//     (Cfg<16, true>, SLACK in the search epilogue): |accumulator - kov_ref| < 4.6e-5 ||gR|| ||gD|| wherever
//     ||gR|| ||gD|| >= 2^24 and 0 below; the packers store upper bounds of ||gR|| per range row and of max ||gD|| per
//     32-domain chunk.  k_umma_refine_rgb replays the float sum in pixel order, i.e. ranks by kov_ref itself.

// Sort keys of the RGB pool: vD^2 (plays the role of varD), payload: the domain index (a group of images: see
// k_umma_sortkeys; the stats are [n_img][3][ND]).
__global__ void k_umma_sortkeys_rgb(const int32_t *__restrict__ dsum, int n, int64_t ND, int64_t count, uint32_t *__restrict__ keys,
                                    int32_t *__restrict__ vals)
{
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    const int64_t image = j >= ND ? j / ND : 0;
    int dm[3];
    const int vd = centred_sum_rgb(dsum + image * 3 * ND, ND, j - image * ND, n, dm);
    keys[j] = (uint32_t)image << 24 | (uint32_t)(vd * vd);
    vals[j] = (int32_t)j;
}

// RGB twin of k_umma_pack_domains<B, true>: the operand row holds gD as binary16 (zeros when vD == 0), pos_info =
// {domain, vD, 0, 0}; the refine step re-reads the operand row itself, so no raw copy is kept.  B = 16: the row's 32
// 16-byte pieces are split over the tile's two parts (Cfg<16, true>), and every chunk also records an upper bound of
// its rows' Euclidean norms ||gD||, from which the search kernel bounds the rounding of the float covariances.
template <int B>
__device__ __forceinline__ uint8_t *rgb_dom_piece(uint8_t *blob, int row, int c)
{
    using L = Lay<B, true>;
    constexpr int NCH0 = L::KS0 * 2;  // 16-byte pieces of a row in part P0 (all of them unless the tile is K-split)
    if (!Cfg<B, true>::KSPLIT || c < NCH0) return blob + (row >> 3) * L::SBO_B + (row & 7) * 16 + c * 128;
    return blob + L::P0_BYTES + (row >> 3) * L::SBO_P1 + (row & 7) * 16 + (c - NCH0) * 128;
}

template <int B>
__global__ void __launch_bounds__(128)
k_umma_pack_domains_rgb(const uint16_t *__restrict__ dec3, const int32_t *__restrict__ dsum,
                        const int32_t *__restrict__ perm, uint8_t *__restrict__ opB, int32_t *__restrict__ pos_dom,
                        int4 *__restrict__ pos_info, int64_t *__restrict__ dom0_pos, Geom g, int64_t ntiles, uint32_t mult,
                        int64_t npos, size_t opb_stride)
{
    using L = Lay<B, true>;
    constexpr int n = B * B;
    const int64_t p0 = (int64_t)blockIdx.x * blockDim.x;  // see k_umma_pack_domains
    const int64_t image = p0 >= npos ? p0 / npos : 0;
    const int64_t pos = p0 + threadIdx.x - image * npos;
    dec3 += image * g.sw * g.sh;
    dsum += image * 3 * g.ND;
    perm += image * g.ND;
    opB = image_region(opB, image, opb_stride);
    pos_dom = image_region(pos_dom, image, opb_stride);
    pos_info = image_region(pos_info, image, opb_stride);
    dom0_pos = image_region(dom0_pos, image, opb_stride);
    const int64_t tile = pos / kTileN;
    const int row = (int)(pos % kTileN);
    const int64_t sp = sweep_to_sorted(pos, mult, ntiles * kChunksPerTile);
    uint8_t *blob = opB + tile * L::B_TILE_BYTES;
    constexpr int NCH = n / 8;  // 16-byte pieces (8 binary16) per row
    float rsd_hi = 0.0f, rsd_lo = __int_as_float(0x7f800000), norm = 0.0f;
    if (sp >= g.ND) {
#pragma unroll
        for (int c = 0; c < NCH; c++) *(uint4 *)rgb_dom_piece<B>(blob, row, c) = make_uint4(0, 0, 0, 0);
        pos_dom[pos] = -1;
        pos_info[pos] = make_int4(-1, 0, 0, 0);
    } else {
        const int64_t j = perm[sp] - image * g.ND;
        const int gx = (int)(j % g.dpw), gy = (int)(j / g.dpw);
        // dec3 = R + G + B of the decimated planes (k_sum_planes); a block row starts at a multiple of B / 4
        // pixels: B = 8 reads pixel pairs (4-byte loads), B = 16 groups of four (8-byte loads)
        const uint16_t *p = dec3 + (int64_t)(gy * g.step) * g.sw + gx * g.step;
        int dm[3];
        const int vd = centred_sum_rgb(dsum, g.ND, j, n, dm);
        const int dmsum = dm[0] + dm[1] + dm[2];
        uint32_t sumsq = 0;  // sum gD^2 <= 256 * 765^2 = 1.5e8: exact in u32
#pragma unroll
        for (int c = 0; c < NCH; c++) {
            int dv[8];
            const int k0 = c * 8;  // first pixel of the piece: row k0 / B of the block, column k0 % B
            const uint16_t *q = p + (int64_t)(k0 / B) * g.sw + (k0 % B);
            if (B == 16) {
#pragma unroll
                for (int e = 0; e < 8; e += 4) {
                    const uint2 w = __ldg((const uint2 *)(q + e));
                    dv[e] = (int)(w.x & 0xffffu); dv[e + 1] = (int)(w.x >> 16);
                    dv[e + 2] = (int)(w.y & 0xffffu); dv[e + 3] = (int)(w.y >> 16);
                }
            } else if (B == 8) {
#pragma unroll
                for (int e = 0; e < 8; e += 2) {
                    const uint32_t w = __ldg((const uint32_t *)(q + e));
                    dv[e] = (int)(w & 0xffffu);
                    dv[e + 1] = (int)(w >> 16);
                }
            } else {
#pragma unroll
                for (int e = 0; e < 8; e++) {
                    const int k = k0 + e;
                    dv[e] = (int)__ldg(p + (int64_t)(k / B) * g.sw + (k % B));
                }
            }
#pragma unroll
            for (int e = 0; e < 8; e++) {
                dv[e] = vd != 0 ? dv[e] - dmsum : 0;
                sumsq += (uint32_t)(dv[e] * dv[e]);
            }
            *(uint4 *)rgb_dom_piece<B>(blob, row, c) =
                make_uint4(pack_h2(dv[0], dv[1]), pack_h2(dv[2], dv[3]), pack_h2(dv[4], dv[5]), pack_h2(dv[6], dv[7]));
        }
        pos_dom[pos] = (int32_t)j;
        pos_info[pos] = make_int4((int32_t)j, vd, 0, 0);
        if (j == 0) *dom0_pos = pos;
        if (vd > 0) {
            float r = __double2float_rn(__ddiv_rn(1.0, (double)vd));
            rsd_hi = r * (1.0f + 4.76837158203125e-07f);  // >= (1 / vD) * (1 + 2^-22), see k_umma_pack_domains
            rsd_lo = r * (1.0f - 4.76837158203125e-07f);
        }
        norm = __fsqrt_ru((float)sumsq) * (1.0f + 2.384185791015625e-07f);  // >= ||gD||_2
    }
    for (int o = 16; o > 0; o >>= 1) {
        rsd_hi = fmaxf(rsd_hi, __shfl_xor_sync(0xffffffffu, rsd_hi, o));
        rsd_lo = fminf(rsd_lo, __shfl_xor_sync(0xffffffffu, rsd_lo, o));
        norm = fmaxf(norm, __shfl_xor_sync(0xffffffffu, norm, o));
    }
    if ((threadIdx.x & 31) == 0) {
        if (rsd_hi == 0.0f) rsd_lo = 0.0f;
        *(float2 *)(blob + L::B_OP_BYTES + (row >> 5) * 8) = make_float2(rsd_hi, rsd_lo);
        *(float *)(blob + L::B_OP_BYTES + kNormOff + (row >> 5) * 4) = norm;
    }
    // tile flag: a K-split tile always has its second part (there is no "all low digits zero" case for binary16)
    if (threadIdx.x == 0) *(uint4 *)(blob + L::B_OP_BYTES + kChunksPerTile * 8) = make_uint4(Cfg<B, true>::KSPLIT ? 1u : 0u, 0, 0, 0);
}

// RGB twin of k_umma_pack_ranges<B, true>: gR as binary16; nRout (optional) receives an upper bound of ||gR||_2.
template <int B>
__global__ void __launch_bounds__(128)
k_umma_pack_ranges_rgb(const uint8_t *__restrict__ src, const int32_t *__restrict__ rsum, uint8_t *__restrict__ opA,
                       int32_t *__restrict__ vRout, float *__restrict__ nRout, Geom g, int64_t j0, int64_t j1, int64_t rows_padded,
                       int n_img)
{
    using L = Lay<B, true>;
    constexpr int n = B * B;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows_padded * n_img) return;
    int64_t sb = i / L::ROWS_SB;
    int rr = (int)(i % L::ROWS_SB);
    int blk = rr / kBlockM, row = rr % kBlockM;
    uint8_t *rowp = opA + sb * L::A_SB_BYTES + blk * L::A_BLOCK_BYTES + (row >> 3) * L::SBO_A + (row & 7) * 16;
    constexpr int NCH = n / 8;
    const int64_t image = i >= rows_padded ? i / rows_padded : 0;  // see k_umma_pack_ranges
    src += image * 3 * g.W * g.H;
    rsum += image * 3 * g.NR;
    const int64_t j = j0 + (i - image * rows_padded);
    if (j >= j1) {
#pragma unroll
        for (int c = 0; c < NCH; c++) *(uint4 *)(rowp + c * 128) = make_uint4(0, 0, 0, 0);
        vRout[i] = 0;
        if (nRout) nRout[i] = 0.0f;
        return;
    }
    const int xr = (int)(j % g.rpw), yr = (int)(j / g.rpw);
    const int64_t plane = (int64_t)g.W * g.H;
    const uint8_t *p = src + (int64_t)(yr * B) * g.W + xr * B;
    int rm[3];
    const int vR = centred_sum_rgb(rsum, g.NR, j, n, rm);
    const int rmsum = rm[0] + rm[1] + rm[2];
    uint32_t sumsq = 0;
#pragma unroll
    for (int c = 0; c < NCH; c++) {
        int rv[8];
#pragma unroll
        for (int e = 0; e < 8; e++) {
            const int k = c * 8 + e;
            const uint8_t *q = p + (int64_t)(k / B) * g.W + (k % B);
            rv[e] = (int)q[0] + (int)q[plane] + (int)q[2 * plane] - rmsum;
            sumsq += (uint32_t)(rv[e] * rv[e]);
        }
        *(uint4 *)(rowp + c * 128) =
            make_uint4(pack_h2(rv[0], rv[1]), pack_h2(rv[2], rv[3]), pack_h2(rv[4], rv[5]), pack_h2(rv[6], rv[7]));
    }
    vRout[i] = vR;
    if (nRout) nRout[i] = __fsqrt_ru((float)sumsq) * (1.0f + 2.384185791015625e-07f);
}

// ---------------------------------------------------------------- PTX wrappers -------

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok;
}
// Bounded wait: a pipeline bug must end in an error, never in a hung GPU.  status is
// pinned host memory (mapped), so the code survives the trap.
__device__ __noinline__ void mbar_timeout(volatile int *status, int code)
{
    if (status) {
        *status = code;
        __threadfence_system();
    }
    __trap();
}
// The polling loop lives out of line: the hot loops only carry the first try.
__device__ __noinline__ void mbar_wait_slow(uint32_t bar, uint32_t parity, volatile int *status, int code)
{
    long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 2000000000ll) mbar_timeout(status, code);
    }
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, volatile int *status, int code)
{
    if (mbar_try_wait(bar, parity)) return;
    mbar_wait_slow(bar, parity, status, code);
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ uint32_t elect_one()
{
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b32 r;\n\t"
        "elect.sync r|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_i8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
// ---- CTA pairs (cta_group::2): the two CTAs of a cluster of 2 share one tcgen05.mma of M = 256 ----
__device__ __forceinline__ uint32_t cluster_ctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> shared::cluster address of the same offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t rank)
{
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
// Remote arrive.  Default semantics (release at CTA scope), as for the local arrives: these barriers order tcgen05 /
// TMA (async proxy) work through tcgen05.fence and complete_tx, no generic-proxy data crosses the pair -- a
// .release.cluster here costs a MEMBAR.GPU per hand-back and the matching .acquire.cluster wait an L1 invalidation.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr)
{
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// commit of the pair's MMAs: arrives on the barrier at this offset in every CTA of `mask`
__device__ __forceinline__ void tc_commit2(uint32_t bar, uint32_t mask)
{
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
                 "h"((uint16_t)mask)
                 : "memory");
}
__device__ __forceinline__ void tc_mma2_i8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void tc_mma2_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void sts_u32(uint32_t saddr, uint32_t v)
{
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(saddr), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t lds_volatile_u32(uint32_t saddr)
{
    uint32_t v;
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr) : "memory");
    return v;
}
// Zero-instruction scheduling fence on 32 registers: code that consumes v[] stays behind everything issued before.
__device__ __forceinline__ void pin_order(uint32_t (&v)[32])
{
    asm volatile(""
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]),
                   "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]), "+r"(v[16]),
                   "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]), "+r"(v[24]),
                   "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
                 :
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ int dp4a_uu(uint32_t a_u8x4, uint32_t b_u8x4, int c)
{
    int d;
    asm("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a_u8x4), "r"(b_u8x4), "r"(c));
    return d;
}

// K-major, no-swizzle shared-memory matrix descriptor (PTX "matrix descriptor";
// cute::UMMA::SmemDescriptor): start address, leading (K) and stride (M/N) byte offsets
// in 16-byte units, descriptor version 1 (Blackwell) in bits 46-47, layout type 0.
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    return (uint64_t)((saddr >> 4) & 0x3fff) | ((uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32) | ((uint64_t)1 << 46);
}

// kind::i8 instruction descriptor (cute::UMMA::InstrDescriptor): D = s32 (c_format 2 at
// bit 4), A = u8 (0 at bit 7), B = s8 (1 at bit 10), both K-major, N>>3 at bit 17, M>>4
// at bit 24.
constexpr uint32_t kIdesc = (2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(kTileN >> 3) << 17) |
                            ((uint32_t)(kBlockM >> 4) << 24);
// kind::f16: D = f32 (c_format 1), A = B = binary16 (format 0), both K-major.
constexpr uint32_t kIdescF16 = (1u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(kTileN >> 3) << 17) |
                               ((uint32_t)(kBlockM >> 4) << 24);
// cta_group::2: M = 256 (128 rows in each CTA of the pair), N = 128 (64 operand rows from each CTA)
constexpr uint32_t kIdescPair = (2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(kTileN >> 3) << 17) |
                                ((uint32_t)((2 * kBlockM) >> 4) << 24);
constexpr uint32_t kIdescF16Pair = (1u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(kTileN >> 3) << 17) |
                                   ((uint32_t)((2 * kBlockM) >> 4) << 24);

// ---------------------------------------------------------------- the search kernel --

// How an epilogue warp walks its accumulator (warp e owns lane quarter e % 4 of accumulator e / 4 in every loop).
// 0: load a 32-column chunk, evaluate it, load the next.  2 (kind::f16): software-pipelined -- the load of the next
// chunk is issued behind the first level of the current chunk's max tree.  3 (kind::f16): as 2, and the four flag
// tests wait until the accumulator has been handed back.  Each configuration runs the loop measured fastest for it
// (profiles/README.md): kind::f16 B = 8 gains 1.5-5 % from the pipelined loads, B = 4 (epilogue bound) 10 % from
// deferring the flag tests as well, and the pairs at B <= 8 (the tensor pipe at its full rate) 10 % from the earlier
// hand-back.  (A fourth mapping -- every warp takes one chunk of EVERY accumulator, so that the oldest accumulator is
// drained by four warps at once -- handed accumulators back soonest and still lost on every configuration to its four
// waits per tile.)
template <int B, bool F16, bool PAIR>
__host__ __device__ constexpr int epi_of() { return (!F16 || B == 16) ? 0 : ((B == 4 || PAIR) ? 3 : 2); }

// DUMP: write every accumulator to `dump` (the probe's and the self-test's exactness check); runs the plain loop.
// status: where a bounded mbarrier wait that timed out leaves its code before the trap (null: nowhere).
//
// PAIR: the kernel runs as clusters of two CTAs (one TPC) sharing every tcgen05.mma (cta_group::2, M = 256, N = 128):
// each CTA keeps its own super-block (its 4 x 128 accumulator rows in its own TMEM) and supplies HALF of every domain
// tile (64 operand rows), so a unit is (two adjacent super-blocks) x (1/n_chunks of the tiles), the ring's TMA traffic
// and the tensor pipe's shared-memory reads of the domain operand halve.  CTA 0 of the pair issues; its commits are
// multicast to both CTAs' barriers; CTA 1's warp 1 relays "my half has landed" to CTA 0's full barriers and CTA 1's
// epilogue warps hand accumulators back on CTA 0's t_empty barriers (remote mbarrier arrives).  The epilogue is
// the same code in both CTAs.  n_sb must be even.
//
// GROUP: a group of images (block-diagonal search): super-block sb belongs to image sb / n_sb_img, whose domain tiles
// start opb_stride bytes after the previous image's; n_sb_img is even, so a CTA pair never straddles two images.  Only
// the unit's opB base depends on the image -- ntiles is per image, and row-indexed arrays use the group-global row.
// A single image runs the GROUP = false instantiation, whose code does not see the image arithmetic at all.
template <int B, bool F16, bool PAIR, bool DUMP, bool GROUP = false>
__global__ void __launch_bounds__(kThreads, 1)
k_umma_search(const uint8_t *__restrict__ opA, const uint8_t *__restrict__ opB, const int32_t *__restrict__ vRarr,
              const float *__restrict__ nRarr, int2 *__restrict__ flag_list, int32_t *__restrict__ flag_cnt, uint32_t *__restrict__ row_lb, int n_sb,
              int n_chunks, int ntiles, int iso_shift, int64_t rows_padded, int32_t *__restrict__ dump, int64_t dump_ld, volatile int *status,
              int n_sb_img, int64_t opb_stride)
{
    using C = Cfg<B, F16>;
    using L = Lay<B, F16>;
    static_assert(!PAIR || F16 || C::KSPLIT, "CTA pairs: kind::f16, or the K-split configurations (B = 16)");
    constexpr int EPI = DUMP ? 0 : epi_of<B, F16, PAIR>();
    // issuing warps of a pair: two for the whole-tile kernels (see below); one where a tile is 9-17 K-slices per
    // accumulator (K-split: the issuing thread is not the bottleneck there)
    constexpr int NISS = (PAIR && !C::KSPLIT) ? 2 : 1;
    constexpr int NSTAGE = PAIR ? L::PAIR_STAGES : C::NSTAGE;
    constexpr int SLOT = PAIR ? L::PAIR_SLOT_BYTES : L::SLOT_BYTES;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // carve: [A super-block][NSTAGE domain tiles (PAIR: half tiles)][barriers]
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t *sA = smem;
    uint8_t *sB = smem + L::A_SB_BYTES;
    uint64_t *bars = (uint64_t *)(sB + C::NSTAGE * L::SLOT_BYTES);
    uint32_t bar0 = smem_u32(bars);
    asm volatile("" : "+r"(bar0));  // opaque: keep the barrier base in a register instead of rematerialising it at every use
    auto BAR_B_FULL = [&](int s) { return bar0 + 8u * s; };
    auto BAR_B_EMPTY = [&](int s) { return bar0 + 8u * (NSTAGE + s); };
    auto BAR_T_FULL = [&](int q) { return bar0 + 8u * (2 * NSTAGE + q); };
    auto BAR_T_EMPTY = [&](int q) { return bar0 + 8u * (2 * NSTAGE + kAccs + q); };
    const uint32_t BAR_A_FULL = bar0 + 8u * (2 * NSTAGE + 2 * kAccs);
    const uint32_t BAR_A_EMPTY = BAR_A_FULL + 8u;
    uint32_t *tmem_slot = (uint32_t *)(bars + 2 * NSTAGE + 2 * kAccs + 2);
    // K-split pairs: "this tile has a second part" per ring stage, written by the producer ahead of the stage's
    // expect_tx arrive and read by the issuer / the relay behind their wait on the stage's full barrier
    const uint32_t s_has_l = bar0 + 400u;
    uint32_t *s_lb = (uint32_t *)((uint8_t *)bars + L::BAR_BYTES);  // [kRowsPerSB] binary32 bits of the row's lower bound

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // PAIR: rank of this CTA in its pair; units are walked per pair (cluster), super-block 2 * (pair index) + rank
    const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
    const int u_first = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x, u_step = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int n_sbu = PAIR ? (n_sb >> 1) : n_sb;  // super-blocks (PAIR: pairs of them) per domain chunk

    if (warp == 1 && lane == 0) {
        // PAIR, CTA 0: the full barriers also collect CTA 1's relayed arrival, t_empty the hand-backs of both CTAs
        const uint32_t both = (PAIR && rank == 0) ? 2u : 1u;
        for (int s = 0; s < NSTAGE; s++) {
            mbar_init(BAR_B_FULL(s), both);
            mbar_init(BAR_B_EMPTY(s), NISS);  // released by the MMA issuers' commits alone: the epilogue never touches the ring
        }
        for (int q = 0; q < kAccs; q++) {
            mbar_init(BAR_T_FULL(q), 1);
            mbar_init(BAR_T_EMPTY(q), both * (kEpiWarps / kAccs));  // the 4 lane quarters of the accumulator (PAIR: of both CTAs)
        }
        mbar_init(BAR_A_FULL, both);
        mbar_init(BAR_A_EMPTY, NISS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        if (PAIR) {  // one warp of EACH CTA of the pair
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    if (PAIR) cluster_sync_all();  // the peer's barriers are initialised and its TMEM allocated before anything remote
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int n_units = n_sbu * n_chunks;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            uint32_t stage = 0, phase = 0, a_phase = 0;
            for (int u = u_first; u < n_units; u += u_step) {
                int sb = PAIR ? 2 * (u % n_sbu) + (int)rank : u % n_sbu, ch = u / n_sbu;  // chunk-major: see the epilogue (bounds carried between units)
                int t0 = (int)((int64_t)ch * ntiles / n_chunks), t1 = (int)((int64_t)(ch + 1) * ntiles / n_chunks);
                const uint8_t *const opB_img = GROUP ? opB + (int64_t)(sb / n_sb_img) * opb_stride : opB;
                mbar_wait(BAR_A_EMPTY, a_phase ^ 1, status, 1);
                mbar_expect_tx(BAR_A_FULL, L::A_SB_BYTES);
                bulk_g2s(smem_u32(sA), opA + (int64_t)sb * L::A_SB_BYTES, L::A_SB_BYTES, BAR_A_FULL);
                for (int t = t0; t < t1; t++) {
                    const uint8_t *blob = opB_img + (int64_t)t * L::B_TILE_BYTES;
                    if (C::KSPLIT && PAIR) {
                        // this CTA's half (operand rows 64 * rank ..) of part P0, then of part P1 unless its digits are all zero
                        const uint32_t has_l = __ldg((const uint32_t *)(blob + L::B_OP_BYTES + kChunksPerTile * 8));
                        mbar_wait(BAR_B_EMPTY(stage), phase ^ 1, status, 2);
                        sts_u32(s_has_l + 4u * stage, has_l);
                        mbar_expect_tx(BAR_B_FULL(stage), L::PAIR_P0_BYTES);
                        bulk_g2s(smem_u32(sB + stage * SLOT), blob + rank * L::PAIR_P0_BYTES, L::PAIR_P0_BYTES, BAR_B_FULL(stage));
                        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                        if (has_l) {
                            mbar_wait(BAR_B_EMPTY(stage), phase ^ 1, status, 2);
                            mbar_expect_tx(BAR_B_FULL(stage), L::PAIR_P1_BYTES);
                            bulk_g2s(smem_u32(sB + stage * SLOT), blob + L::P0_BYTES + rank * L::PAIR_P1_BYTES, L::PAIR_P1_BYTES, BAR_B_FULL(stage));
                            if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                        }
                    } else if (C::KSPLIT) {
                        // part P0 (high digits, -alpha, bounds), then part P1 (low digits) unless they are all zero
                        mbar_wait(BAR_B_EMPTY(stage), phase ^ 1, status, 2);
                        mbar_expect_tx(BAR_B_FULL(stage), L::P0_BYTES);
                        bulk_g2s(smem_u32(sB + stage * L::SLOT_BYTES), blob, L::P0_BYTES, BAR_B_FULL(stage));
                        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                        const uint32_t has_l = __ldg((const uint32_t *)(blob + L::B_OP_BYTES + kChunksPerTile * 8));
                        if (has_l) {
                            mbar_wait(BAR_B_EMPTY(stage), phase ^ 1, status, 2);
                            mbar_expect_tx(BAR_B_FULL(stage), L::P1_BYTES);
                            bulk_g2s(smem_u32(sB + stage * L::SLOT_BYTES), blob + L::P0_BYTES, L::P1_BYTES, BAR_B_FULL(stage));
                            if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                        }
                    } else if (PAIR) {
                        // this CTA's half of the tile: operand rows 64 * rank .. 64 * rank + 63 (8 row groups, contiguous)
                        mbar_wait(BAR_B_EMPTY(stage), phase ^ 1, status, 2);
                        mbar_expect_tx(BAR_B_FULL(stage), SLOT);
                        bulk_g2s(smem_u32(sB + stage * SLOT), blob + rank * SLOT, SLOT, BAR_B_FULL(stage));
                        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                    } else {
                        mbar_wait(BAR_B_EMPTY(stage), phase ^ 1, status, 2);
                        mbar_expect_tx(BAR_B_FULL(stage), L::B_TILE_BYTES);
                        bulk_g2s(smem_u32(sB + stage * L::SLOT_BYTES), blob, L::B_TILE_BYTES, BAR_B_FULL(stage));
                        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                    }
                }
                a_phase ^= 1;
            }
        }
        __syncwarp();
    } else if (PAIR && (warp == 1 || (warp == 3 && !C::KSPLIT))) {
        // ===================== MMA issuers of a pair (CTA 0) =====================
        // What bounds the pair kernel once the operands stream at full rate is the issuing thread itself: per
        // accumulator one barrier wait, the descriptor moves into uniform registers, four tcgen05.mma and a commit
        // -- a serial chain of 250-300 clocks on a sub-partition it shares with four busy epilogue warps, against
        // 256 clocks of tensor work.  Two warps on different sub-partitions therefore issue side by side: warp 1
        // owns accumulators 0 and 2, warp 3 accumulators 1 and 3.  MMAs of different accumulators need no mutual
        // order; a ring slot (and the A super-block) is free once BOTH issuers' commits have arrived.
        if constexpr (PAIR && C::KSPLIT) {
            if (rank == 0) {
                // ===================== MMA issuer of a K-split pair (CTA 0, one warp) =====================
                uint32_t stage = 0, phase = 0, a_phase = 0, t_phase = 0;
                const uint32_t elected = elect_one();
                const uint64_t a_desc0 = make_desc(smem_u32(sA), 128, L::SBO_A);
                for (int u = u_first; u < n_units; u += u_step) {
                    int ch = u / n_sbu;
                    int t0 = (int)((int64_t)ch * ntiles / n_chunks), t1 = (int)((int64_t)(ch + 1) * ntiles / n_chunks);
                    mbar_wait(BAR_A_FULL, a_phase, status, 3);
                    for (int t = t0; t < t1; t++) {
                        mbar_wait(BAR_B_FULL(stage), phase, status, 4);  // both halves of part P0
                        tc_fence_after();
                        const uint32_t has_l = lds_volatile_u32(s_has_l + 4u * stage);
                        const uint64_t b0 = make_desc(smem_u32(sB + stage * SLOT), 128, L::SBO_B);
#pragma unroll
                        for (int q = 0; q < C::NB; q++) {
                            mbar_wait(BAR_T_EMPTY(q), ((t_phase >> q) & 1) ^ 1, status, 5);  // the epilogue warps of both CTAs
                            tc_fence_after();
                            if (elected) {
#pragma unroll
                                for (int s = 0; s < L::KS0; s++) {
                                    const uint64_t ad = a_desc0 + (uint64_t)((q * L::A_BLOCK_BYTES + s * 256) >> 4);
                                    if (F16) tc_mma2_f16(tmem_base + q * kTileN, ad, b0 + (uint64_t)((s * 256) >> 4), kIdescF16Pair, s > 0 ? 1u : 0u);
                                    else tc_mma2_i8(tmem_base + q * kTileN, ad, b0 + (uint64_t)((s * 256) >> 4), kIdescPair, s > 0 ? 1u : 0u);
                                }
                                if (!has_l) tc_commit2(BAR_T_FULL(q), 3u);
                            }
                            __syncwarp();
                            t_phase ^= 1u << q;
                        }
                        if (elected) tc_commit2(BAR_B_EMPTY(stage), 3u);  // both CTAs' slots are free once these MMAs have read them
                        __syncwarp();
                        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                        if (has_l) {
                            mbar_wait(BAR_B_FULL(stage), phase, status, 4);
                            tc_fence_after();
                            const uint64_t b1 = make_desc(smem_u32(sB + stage * SLOT), 128, L::SBO_P1);
#pragma unroll
                            for (int q = 0; q < C::NB; q++) {
                                if (elected) {
#pragma unroll
                                    for (int s = 0; s < C::KS_B - L::KS0; s++) {
                                        const int sa = F16 ? L::KS0 + s : s;  // kind::i8: the low digits meet the r slices again
                                        const uint64_t ad = a_desc0 + (uint64_t)((q * L::A_BLOCK_BYTES + sa * 256) >> 4);
                                        if (F16) tc_mma2_f16(tmem_base + q * kTileN, ad, b1 + (uint64_t)((s * 256) >> 4), kIdescF16Pair, 1u);
                                        else tc_mma2_i8(tmem_base + q * kTileN, ad, b1 + (uint64_t)((s * 256) >> 4), kIdescPair, 1u);
                                    }
                                    tc_commit2(BAR_T_FULL(q), 3u);
                                }
                                __syncwarp();
                            }
                            if (elected) tc_commit2(BAR_B_EMPTY(stage), 3u);
                            __syncwarp();
                            if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                        }
                    }
                    if (elected) tc_commit2(BAR_A_EMPTY, 3u);
                    __syncwarp();
                    a_phase ^= 1;
                }
            } else {
                // ===================== relay (CTA 1 of a K-split pair) =====================
                if (lane == 0) {
                    uint32_t stage = 0, phase = 0, a_phase = 0;
                    const uint32_t ra_full = mapa_u32(BAR_A_FULL, 0);
                    for (int u = u_first; u < n_units; u += u_step) {
                        int ch = u / n_sbu;
                        int t0 = (int)((int64_t)ch * ntiles / n_chunks), t1 = (int)((int64_t)(ch + 1) * ntiles / n_chunks);
                        mbar_wait(BAR_A_FULL, a_phase, status, 3);
                        mbar_arrive_cluster(ra_full);
                        for (int t = t0; t < t1; t++) {
                            mbar_wait(BAR_B_FULL(stage), phase, status, 4);
                            const uint32_t has_l = lds_volatile_u32(s_has_l + 4u * stage);
                            mbar_arrive_cluster(mapa_u32(BAR_B_FULL(stage), 0));
                            if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                            if (has_l) {
                                mbar_wait(BAR_B_FULL(stage), phase, status, 4);
                                mbar_arrive_cluster(mapa_u32(BAR_B_FULL(stage), 0));
                                if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                            }
                        }
                        a_phase ^= 1;
                    }
                }
                __syncwarp();
            }
        } else if constexpr (PAIR) {
            if (rank == 0) {
                const int qi = warp >> 1;  // 0 or 1
                uint32_t stage = 0, phase = 0, a_phase = 0, t_phase = 0;
                const uint32_t elected = elect_one();
                const uint64_t a_desc0 = make_desc(smem_u32(sA), 128, L::SBO_A);
                const uint64_t b_desc0 = make_desc(smem_u32(sB), 128, L::SBO_B);
                for (int u = u_first; u < n_units; u += u_step) {
                    int ch = u / n_sbu;
                    int t0 = (int)((int64_t)ch * ntiles / n_chunks), t1 = (int)((int64_t)(ch + 1) * ntiles / n_chunks);
                    mbar_wait(BAR_A_FULL, a_phase, status, 3);
                    for (int t = t0; t < t1; t++) {
                        mbar_wait(BAR_B_FULL(stage), phase, status, 4);  // both halves: this CTA's copy + the peer's relayed arrival
                        tc_fence_after();
                        const uint64_t b_desc = b_desc0 + (uint64_t)((stage * SLOT) >> 4);
#pragma unroll
                        for (int k = 0; k < 2; k++) {
                            const int q = qi + 2 * k;
                            mbar_wait(BAR_T_EMPTY(q), ((t_phase >> k) & 1) ^ 1, status, 5);  // the epilogue warps of both CTAs
                            tc_fence_after();
                            if (elected) {
#pragma unroll
                                for (int s = 0; s < C::NS; s++) {
                                    const uint64_t ad = a_desc0 + (uint64_t)((q * L::A_BLOCK_BYTES + C::amap(s) * 256) >> 4);
                                    tc_mma2_f16(tmem_base + q * kTileN, ad, b_desc + (uint64_t)((s * 256) >> 4), kIdescF16Pair, s > 0 ? 1u : 0u);
                                }
                                tc_commit2(BAR_T_FULL(q), 3u);
                                if (k == 1) tc_commit2(BAR_B_EMPTY(stage), 3u);  // this issuer's MMAs have read both CTAs' slots
                            }
                            __syncwarp();
                            t_phase ^= 1u << k;
                        }
                        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                    }
                    if (elected) tc_commit2(BAR_A_EMPTY, 3u);  // this issuer's MMAs on the A super-block have completed
                    __syncwarp();
                    a_phase ^= 1;
                }
            } else if (warp == 1) {
                // ===================== relay (CTA 1 of a pair) =====================
                // CTA 0 issues the pair's MMAs and must know that CTA 1's operands have landed: one thread follows this
                // CTA's own full barriers and forwards every completion to the barrier at the same offset in CTA 0.
                if (lane == 0) {
                    uint32_t stage = 0, phase = 0, a_phase = 0;
                    const uint32_t ra_full = mapa_u32(BAR_A_FULL, 0);
                    for (int u = u_first; u < n_units; u += u_step) {
                        int ch = u / n_sbu;
                        int t0 = (int)((int64_t)ch * ntiles / n_chunks), t1 = (int)((int64_t)(ch + 1) * ntiles / n_chunks);
                        mbar_wait(BAR_A_FULL, a_phase, status, 3);
                        mbar_arrive_cluster(ra_full);
                        for (int t = t0; t < t1; t++) {
                            mbar_wait(BAR_B_FULL(stage), phase, status, 4);
                            mbar_arrive_cluster(mapa_u32(BAR_B_FULL(stage), 0));
                            if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                        }
                        a_phase ^= 1;
                    }
                }
                __syncwarp();
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        // The whole warp walks the (warp-uniform) loop so that addresses and descriptors live in
        // uniform registers; one elected lane issues tcgen05.mma / tcgen05.commit.
        uint32_t stage = 0, phase = 0, a_phase = 0, t_phase = 0;  // t_phase: bit q
        const uint32_t elected = elect_one();
        // descriptors differ only in the 14-bit start-address field (16-byte units)
        const uint64_t a_desc0 = make_desc(smem_u32(sA), 128, L::SBO_A);
        const uint64_t b_desc0 = make_desc(smem_u32(sB), 128, L::SBO_B);
        for (int u = u_first; u < n_units; u += u_step) {
            int ch = u / n_sbu;
            int t0 = (int)((int64_t)ch * ntiles / n_chunks), t1 = (int)((int64_t)(ch + 1) * ntiles / n_chunks);
            mbar_wait(BAR_A_FULL, a_phase, status, 3);
            for (int t = t0; t < t1; t++) {
                mbar_wait(BAR_B_FULL(stage), phase, status, 4);
                tc_fence_after();
                // tile flag written by k_umma_pack_domains: 0 -> every low digit of the tile is zero
                const uint32_t has_l = *(volatile const uint32_t *)(sB + stage * L::SLOT_BYTES + L::B_OP_BYTES + kChunksPerTile * 8);
                if (C::KSPLIT) {
                    // part P0: K-slices 0 .. KS0-1 of every accumulator; the slot is released as soon as these MMAs
                    // have read it (commit), so that the next copy overlaps the MMAs on part P1 / the next tile
                    const uint64_t b0 = make_desc(smem_u32(sB + stage * L::SLOT_BYTES), 128, L::SBO_B);
#pragma unroll
                    for (int q = 0; q < C::NB; q++) {
                        mbar_wait(BAR_T_EMPTY(q), ((t_phase >> q) & 1) ^ 1, status, 5);
                        tc_fence_after();
                        if (elected) {
#pragma unroll
                            for (int s = 0; s < L::KS0; s++) {
                                const uint64_t ad = a_desc0 + (uint64_t)((q * L::A_BLOCK_BYTES + s * 256) >> 4);  // A slice s (kind::i8: s = 8 is rmean)
                                if (F16) tc_mma_f16(tmem_base + q * kTileN, ad, b0 + (uint64_t)((s * 256) >> 4), kIdescF16, s > 0 ? 1u : 0u);
                                else tc_mma_i8(tmem_base + q * kTileN, ad, b0 + (uint64_t)((s * 256) >> 4), kIdesc, s > 0 ? 1u : 0u);
                            }
                            if (!has_l) tc_commit(BAR_T_FULL(q));
                        }
                        __syncwarp();
                        t_phase ^= 1u << q;
                    }
                    if (elected) tc_commit(BAR_B_EMPTY(stage));
                    __syncwarp();
                    if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                    if (has_l) {
                        mbar_wait(BAR_B_FULL(stage), phase, status, 4);
                        tc_fence_after();
                        const uint64_t b1 = make_desc(smem_u32(sB + stage * L::SLOT_BYTES), 128, L::SBO_P1);
#pragma unroll
                        for (int q = 0; q < C::NB; q++) {
                            if (elected) {
#pragma unroll
                                for (int s = 0; s < C::KS_B - L::KS0; s++) {
                                    // kind::i8: the low digits meet the r slices again; kind::f16: the second half of K
                                    const int sa = F16 ? L::KS0 + s : s;
                                    const uint64_t ad = a_desc0 + (uint64_t)((q * L::A_BLOCK_BYTES + sa * 256) >> 4);
                                    if (F16) tc_mma_f16(tmem_base + q * kTileN, ad, b1 + (uint64_t)((s * 256) >> 4), kIdescF16, 1u);
                                    else tc_mma_i8(tmem_base + q * kTileN, ad, b1 + (uint64_t)((s * 256) >> 4), kIdesc, 1u);
                                }
                                tc_commit(BAR_T_FULL(q));
                            }
                            __syncwarp();
                        }
                        if (elected) tc_commit(BAR_B_EMPTY(stage));
                        __syncwarp();
                        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
                    }
                    continue;
                }
                const uint64_t b_desc = b_desc0 + (uint64_t)((stage * L::SLOT_BYTES) >> 4);
#pragma unroll
                for (int q = 0; q < C::NB; q++) {
                    mbar_wait(BAR_T_EMPTY(q), ((t_phase >> q) & 1) ^ 1, status, 5);
                    tc_fence_after();
                    if (elected) {
#pragma unroll
                        for (int s = 0; s < C::NS; s++) {
                            if (C::is_l_slice(s) && !has_l) continue;  // sum r*l == 0 for the whole tile
                            const uint64_t ad = a_desc0 + (uint64_t)((q * L::A_BLOCK_BYTES + C::amap(s) * 256) >> 4);
                            const uint64_t bd = b_desc + (uint64_t)((s * 256) >> 4);
                            if (F16) tc_mma_f16(tmem_base + q * kTileN, ad, bd, kIdescF16, s > 0 ? 1u : 0u);
                            else tc_mma_i8(tmem_base + q * kTileN, ad, bd, kIdesc, s > 0 ? 1u : 0u);
                        }
                        tc_commit(BAR_T_FULL(q));
                    }
                    __syncwarp();
                    t_phase ^= 1u << q;
                }
                if (elected) tc_commit(BAR_B_EMPTY(stage));  // the slot is free once these MMAs have read it
                __syncwarp();
                if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
            }
            if (elected) tc_commit(BAR_A_EMPTY);  // every MMA that reads this A super-block has completed
            __syncwarp();
            a_phase ^= 1;
        }
    } else if (warp >= 4) {
        // ===================== epilogue =====================
        // Warp e: TMEM lane quarter lq = e % 4 (== warp % 4, the quarter this warp may access) of accumulator
        // q = e / 4: one thread = one range row, all 128 domains of a tile.  Per tile a warp makes ONE visit (one
        // t_full wait, four 32-column loads, one hand-back); the four warps of an SM sub-partition own the four
        // accumulators, which the issuer completes 1/4 tile apart, so their work is naturally staggered.
        const int e = warp - 4;
        const int lq = e & 3, q = e >> 2;
        const uint32_t ta = tmem_base + ((uint32_t)(lq * 32) << 16) + q * kTileN;
        uint32_t tf_phase = 0;
        // hand-back target: this CTA's t_empty[q]; PAIR: the issuing CTA's (a shared::cluster address)
        const uint32_t bar_hand_back = PAIR ? mapa_u32(BAR_T_EMPTY(q), 0) : BAR_T_EMPTY(q);
        auto hand_back = [&]() {
            if (PAIR) mbar_arrive_cluster(bar_hand_back);
            else mbar_arrive(bar_hand_back);
        };
        // RGB at blockgroesse 16: the float covariances (the reference's sequential sum and the tensor core's) may
        // round once partial sums pass 2^24; see the chunk test below.  Warps of unused accumulators idle.
        constexpr bool SLACK = B == 16 && F16;
        const int n_units_mine = q < C::NB ? n_units : 0;
        for (int u = u_first; u < n_units_mine; u += u_step) {
            // Units are ordered chunk-major (u = ch * n_sb + sb): the units of one super-block run in different
            // waves, so the lower bound a row reached in an earlier unit (row_lb, global memory) can seed the
            // later ones -- any earlier bound is a valid bound, a missed one only costs extra flags.
            int sb = PAIR ? 2 * (u % n_sbu) + (int)rank : u % n_sbu, ch = u / n_sbu;
            int t0 = (int)((int64_t)ch * ntiles / n_chunks), t1 = (int)((int64_t)(ch + 1) * ntiles / n_chunks);
            const uint8_t *const opB_img = GROUP ? opB + (int64_t)(sb / n_sb_img) * opb_stride : opB;
            // Running filter state of this thread's row (see the file header).  vR == 0: every candidate
            // scores error 0 and the first one wins (FC:677-678, FC:627) -> never flag.
            const int64_t row = (int64_t)sb * L::ROWS_SB + q * kBlockM + lq * 32 + lane;
            const int vR = vRarr[row];
            const float nR = SLACK ? nRarr[row] : 0.0f;  // >= ||gR||_2 of this row
            RowFilter st;
            st.thresh = (vR == 0) ? __int_as_float(0x7f800000) : -1.0f;
            st.lbmax = 0.0f;
            st.cnt = 0;
            const float tie_abs = (float)(vR * vR) * 4.76837158203125e-07f;  // vR^2 * 2^-21
            // Isometry extension: the 8 operand rows of a range block (8 adjacent lanes) compete for one winner and
            // have the same vR, so they share one bound through shared memory: a chunk is flagged only if it can
            // beat the best of all 8.
            const uint32_t sh_lb = smem_u32(s_lb + q * kBlockM + (((lq * 32 + lane) >> iso_shift) << iso_shift));
            if (iso_shift) {
                sts_u32(sh_lb, 0u);
                __syncwarp();
            }
            if (ch > 0 && vR != 0) {  // bound reached by the earlier units of this row
                const float seed = __uint_as_float(*(volatile const uint32_t *)(row_lb + ((row >> iso_shift) << iso_shift)));
                if (seed > 0.0f) {
                    st.lbmax = seed;
                    st.thresh = flag_threshold(seed, tie_abs);
                }
            }
            int2 *const list0 = flag_list + (((int64_t)ch * rows_padded + row) * kFlagLists) * kFlagCap;
            int cnt0 = 0, cnt1 = 0;  // entries of the two lists (column halves) of this (row, unit)
            for (int t = t0; t < t1; t++) {
                // (rhi, rlo) of the tile's four chunks, from the tile blob in global memory (the shared-memory ring
                // belongs to the producer and the MMA issuer alone): a broadcast load that every warp of the CTA
                // repeats, so it is an L1 hit for all but the first; its latency hides behind the t_full wait.
                const float4 *gb = (const float4 *)(opB_img + (int64_t)t * L::B_TILE_BYTES + L::B_OP_BYTES);
                const float4 bnd01 = __ldg(gb), bnd23 = __ldg(gb + 1);
                float4 bndn = make_float4(0.0f, 0.0f, 0.0f, 0.0f);  // >= ||gD||_2 of the rows of each chunk
                if (SLACK) bndn = __ldg(gb + 3);
                mbar_wait(BAR_T_FULL(q), tf_phase, status, 7);
                tc_fence_after();
                if (iso_shift) {  // adopt a better bound found by another isometry of the same range block
                    const float other = __uint_as_float(lds_volatile_u32(sh_lb));
                    if (other > st.lbmax) {
                        st.lbmax = other;
                        st.thresh = flag_threshold(other, tie_abs);
                    }
                }
                if constexpr (EPI != 0) {
                    // Software-pipelined visit (kind::f16).  The first level of the |.| max tree reads all 32 registers
                    // of a chunk in 11 instructions; the load of the NEXT chunk is issued behind them (into the same
                    // registers) so that its TMEM latency hides behind the rest of the tree.  EPI == 3 also defers the
                    // four flag tests (multiply, compare, branch) until the accumulator has been handed back: between
                    // two loads only the 16 FMNMX3 remain.  The empty asm statements pin the order where it matters.
                    uint32_t v[32];
                    float Mc[kChunksPerTile];
                    tmem_ld32(ta, v);
                    tmem_ld_wait();
                    pin_order(v);
                    auto test = [&](int c) {
                        const float rhi = c == 0 ? bnd01.x : (c == 1 ? bnd01.z : (c == 2 ? bnd23.x : bnd23.z));
                        const float rlo = c == 0 ? bnd01.y : (c == 1 ? bnd01.w : (c == 2 ? bnd23.y : bnd23.w));
                        const float ub = Mc[c] * rhi;
                        if (ub > st.thresh) {  // may hold the winner or one of its float ties
                            st.cnt = c < 2 ? cnt0 : cnt1;
                            st = flag_chunk(st, Mc[c] * rlo, ub, tie_abs, list0 + (c >> 1) * kFlagCap, t * kChunksPerTile + c, sh_lb, iso_shift ? 1 : 0);
                            if (c < 2) cnt0 = st.cnt;
                            else cnt1 = st.cnt;
                        }
                    };
#pragma unroll
                    for (int c = 0; c < kChunksPerTile; c++) {
                        auto av = [&](int k) { return fabsf(__uint_as_float(v[k])); };
                        float l[11];
#pragma unroll
                        for (int i = 0; i < 10; i++) l[i] = fmaxf(fmaxf(av(3 * i), av(3 * i + 1)), av(3 * i + 2));
                        l[10] = fmaxf(av(30), av(31));
                        if (c + 1 < kChunksPerTile) {
                            uint32_t next = ta + (c + 1) * 32;
                            asm volatile("" : "+r"(next) : "f"(l[0]), "f"(l[1]), "f"(l[2]), "f"(l[3]), "f"(l[4]), "f"(l[5]), "f"(l[6]),
                                         "f"(l[7]), "f"(l[8]), "f"(l[9]), "f"(l[10]));
                            tmem_ld32(next, v);
                        }
                        asm volatile("" : "+f"(l[0]), "+f"(l[1]), "+f"(l[2]), "+f"(l[3]), "+f"(l[4]), "+f"(l[5]), "+f"(l[6]), "+f"(l[7]),
                                     "+f"(l[8]), "+f"(l[9]), "+f"(l[10]));
                        const float m0 = fmaxf(fmaxf(l[0], l[1]), l[2]), m1 = fmaxf(fmaxf(l[3], l[4]), l[5]);
                        const float m2 = fmaxf(fmaxf(l[6], l[7]), l[8]), m3 = fmaxf(fmaxf(l[9], l[10]), m0);
                        Mc[c] = fmaxf(fmaxf(m1, m2), m3);  // max |kov| over the chunk, exact
                        if (EPI == 2) test(c);
                        if (c + 1 < kChunksPerTile) {
                            tmem_ld_wait();
                            pin_order(v);
                            if (c + 1 == kChunksPerTile - 1) {
                                // the accumulator's last chunk is in registers: hand it back
                                tc_fence_before();
                                __syncwarp();
                                if (lane == 0) hand_back();
                                if (EPI == 3) {  // the deferred tests of the first three chunks, in sweep order
                                    asm volatile("" : "+f"(Mc[0]), "+f"(Mc[1]), "+f"(Mc[2]) : : "memory");
                                    test(0);
                                    test(1);
                                    test(2);
                                }
                            }
                        }
                    }
                    if (EPI == 3) test(kChunksPerTile - 1);
                } else {
#pragma unroll
                for (int c = 0; c < kChunksPerTile; c++) {
                    uint32_t v[32];
                    tmem_ld32(ta + c * 32, v);
                    tmem_ld_wait();
                    if (c == kChunksPerTile - 1) {
                        // last read of accumulator q for this tile: hand it back
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) hand_back();
                    }
                    float M;  // max |kov| over the chunk, exact
                    if (F16) {
                        // binary32 accumulators holding exact integers.  FMNMX3 takes |.| on all three
                        // operands: a 3-input tree over 32 values is 16 instructions (four chains of 3, then 4).
                        auto av = [&](int k) { return fabsf(__uint_as_float(v[k])); };
                        float c4[4];
#pragma unroll
                        for (int i = 0; i < 4; i++) {
                            c4[i] = fmaxf(fmaxf(av(8 * i), av(8 * i + 1)), av(8 * i + 2));
                            c4[i] = fmaxf(c4[i], fmaxf(av(8 * i + 3), av(8 * i + 4)));
                            c4[i] = fmaxf(c4[i], fmaxf(av(8 * i + 5), av(8 * i + 6)));
                        }
                        const float m01 = fmaxf(fmaxf(c4[0], c4[1]), av(7));
                        const float m23 = fmaxf(fmaxf(c4[2], c4[3]), av(15));
                        M = fmaxf(fmaxf(fmaxf(m01, m23), av(23)), av(31));
                    } else {
                        int mx0 = 0, mn0 = 0, mx1 = 0, mn1 = 0;  // two independent chains each: ALU latency
#pragma unroll
                        for (int k = 0; k < 32; k += 4) {
                            mx0 = max(mx0, max((int)v[k], (int)v[k + 1]));
                            mn0 = min(mn0, min((int)v[k], (int)v[k + 1]));
                            mx1 = max(mx1, max((int)v[k + 2], (int)v[k + 3]));
                            mn1 = min(mn1, min((int)v[k + 2], (int)v[k + 3]));
                        }
                        M = __int2float_rn(max(max(mx0, mx1), -min(mn0, mn1)));
                    }
                    if (DUMP) {
#pragma unroll
                        for (int k = 0; k < 32; k++) {
                            int iv = (int)v[k];
                            if (F16) {  // a non-integral accumulator must fail the probe's check
                                const float f = __uint_as_float(v[k]);
                                iv = (f == rintf(f) && fabsf(f) < 2.0e9f) ? (int)f : (int)0x80000000;
                            }
                            dump[row * dump_ld + (int64_t)t * kTileN + c * 32 + k] = iv;
                        }
                    }
                    const float rhi = c == 0 ? bnd01.x : (c == 1 ? bnd01.z : (c == 2 ? bnd23.x : bnd23.z));
                    const float rlo = c == 0 ? bnd01.y : (c == 1 ? bnd01.w : (c == 2 ? bnd23.y : bnd23.w));
                    float Mu = M, Ml = M;
                    if (SLACK) {
                        // Every partial sum of sum gR*gD, in any order, is at most ||gR|| ||gD|| (Cauchy-Schwarz).
                        // Below 2^24 all of them are exact integers: the accumulator IS the reference's kov.  Above,
                        // a binary32 sum of 256 exact products is within 255 * 2^-24 * ||gR|| ||gD|| of the true value
                        // when every add rounds to nearest (the reference's sequential sum) and within twice that
                        // if the tensor core truncates: |accumulator - kov_reference| < 4.6e-5 * ||gR|| ||gD||.  The
                        // chunk bounds are widened by that much (6e-5: margin for the norms' own rounding).
                        const float pn = nR * (c == 0 ? bndn.x : (c == 1 ? bndn.y : (c == 2 ? bndn.z : bndn.w)));
                        if (pn >= 16777216.0f) {
                            const float sl = pn * 6.0e-5f;
                            Mu = M + sl;
                            Ml = fmaxf(M - sl, 0.0f);
                        }
                    }
                    const float ub = Mu * rhi;
                    if (ub > st.thresh) {  // may hold the winner or one of its float ties
                        // the refine step reads two lists per (row, unit), one per column half, as the layout of
                        // the earlier two-warps-per-accumulator mapping had it
                        st.cnt = c < 2 ? cnt0 : cnt1;
                        st = flag_chunk(st, Ml * rlo, ub, tie_abs, list0 + (c >> 1) * kFlagCap, t * kChunksPerTile + c, sh_lb, iso_shift ? 1 : 0);
                        if (c < 2) cnt0 = st.cnt;
                        else cnt1 = st.cnt;
                    }
                }
                }
                tf_phase ^= 1;
            }
            flag_cnt[((int64_t)ch * rows_padded + row) * 2] = cnt0;
            flag_cnt[((int64_t)ch * rows_padded + row) * 2 + 1] = cnt1;
            // the row's bound after this unit: seeds its later units and lets the refine step drop stale flags
            if (st.lbmax > 0.0f) atomicMax(row_lb + ((row >> iso_shift) << iso_shift), __float_as_uint(st.lbmax));
        }
    }

    tc_fence_before();
    if (PAIR) cluster_sync_all();  // neither CTA leaves (shared memory, barriers, TMEM) while the other may still touch it
    else __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
        else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ---------------------------------------------------------------- tensor pipe peak -----

// Bare tcgen05.mma loop (M=128, N columns, one 32-byte K-slice per instruction, operands resident
// in shared memory, alternating TMEM accumulators, no epilogue): measures what the tensor pipe of
// this GPU sustains for the instruction shape the search uses -- the denominator of the search
// kernel's roofline (MEASURED_PEAKS.json only carries a cuBLAS bf16 figure).
template <bool F16, int N>
__global__ void __launch_bounds__(128, 1) k_mma_peak(int iters, uint32_t seed)
{
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t *sA = smem;                 // 128 rows x 32 B, core-matrix order (16 groups x 256 B)
    uint8_t *sB = smem + 4096;          // N rows x 32 B
    uint64_t *bar = (uint64_t *)(smem + 4096 + 8192);
    uint32_t *tmem_slot = (uint32_t *)(bar + 1);
    const int warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < (4096 + 8192) / 4; i += blockDim.x) {
        uint32_t x = (uint32_t)i * 2654435761u + seed + blockIdx.x * 40503u;
        x ^= x >> 15; x *= 0x2c1b3c6du; x ^= x >> 12;
        if (F16) x &= 0x3fff3fffu;  // finite binary16 values below 2: no NaN / Inf arithmetic
        ((uint32_t *)smem)[i] = x;
    }
    if (threadIdx.x == 0) {
        mbar_init(smem_u32(bar), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy smem writes -> async proxy (MMA)
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (warp == 1) {
        const uint32_t elected = elect_one();
        const uint64_t ad = make_desc(smem_u32(sA), 128, 256);
        const uint64_t bd = make_desc(smem_u32(sB), 128, 256);
        constexpr uint32_t idesc = (F16 ? ((1u << 4) | (0u << 7) | (0u << 10)) : ((2u << 4) | (0u << 7) | (1u << 10))) |
                                   ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        constexpr int NACC = 512 / N;
        if (elected) {
            for (int i = 0; i < iters; i++) {
                const uint32_t d = tmem_base + (uint32_t)(i & (NACC - 1)) * N;
                if (F16) tc_mma_f16(d, ad, bd, idesc, i >= NACC ? 1u : 0u);
                else tc_mma_i8(d, ad, bd, idesc, i >= NACC ? 1u : 0u);
            }
            tc_commit(smem_u32(bar));
        }
        __syncwarp();
        mbar_wait(smem_u32(bar), 0, nullptr, 9);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// The same loop issued by CTA pairs: tcgen05.mma.cta_group::2, M = 256 (128 rows per CTA), N = 128 (64 operand rows
// per CTA): per MMA an SM reads 4 KB of A and 2 KB of B from its shared memory instead of 4 + 4.  out[blockIdx.x]
// receives the CTA's TMEM base address (both CTAs of a pair must report the same one).
template <bool F16>
__global__ void __launch_bounds__(128, 1) k_mma_peak_pair(int iters, uint32_t seed, uint32_t *out)
{
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t *sA = smem;                 // 128 rows x 32 B, core-matrix order (16 groups x 256 B)
    uint8_t *sB = smem + 4096;          // this CTA's 64 of the 128 B rows x 32 B
    uint64_t *bar = (uint64_t *)(smem + 4096 + 8192);
    uint32_t *tmem_slot = (uint32_t *)(bar + 1);
    const int warp = threadIdx.x >> 5;
    const uint32_t rank = cluster_ctarank();
    for (int i = threadIdx.x; i < (4096 + 8192) / 4; i += blockDim.x) {
        uint32_t x = (uint32_t)i * 2654435761u + seed + blockIdx.x * 40503u;
        x ^= x >> 15; x *= 0x2c1b3c6du; x ^= x >> 12;
        if (F16) x &= 0x3fff3fffu;
        ((uint32_t *)smem)[i] = x;
    }
    if (threadIdx.x == 0) {
        mbar_init(smem_u32(bar), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(256u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (threadIdx.x == 0 && out) out[blockIdx.x] = tmem_base;
    if (warp == 1) {
        if (rank == 0) {
            const uint32_t elected = elect_one();
            const uint64_t ad = make_desc(smem_u32(sA), 128, 256);
            const uint64_t bd = make_desc(smem_u32(sB), 128, 256);
            constexpr uint32_t idesc = (F16 ? ((1u << 4) | (0u << 7) | (0u << 10)) : ((2u << 4) | (0u << 7) | (1u << 10))) |
                                       ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
            if (elected) {
                for (int i = 0; i < iters; i++) {
                    const uint32_t d = tmem_base + (uint32_t)(i & 1) * 128;
                    if (F16) tc_mma2_f16(d, ad, bd, idesc, i >= 2 ? 1u : 0u);
                    else tc_mma2_i8(d, ad, bd, idesc, i >= 2 ? 1u : 0u);
                }
                tc_commit2(smem_u32(bar), 3u);
            }
            __syncwarp();
        }
        mbar_wait(smem_u32(bar), 0, nullptr, 9);  // both CTAs: the pair's MMAs have completed
    }
    tc_fence_before();
    cluster_sync_all();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256u) : "memory");
    }
}

// ---------------------------------------------------------------- refine --------------

// Exact integer covariance of the candidate at sweep position `pos` with one range row, from the raw
// domain pixels (see raw_offset):
//     kov = sum (r - rmean)(d - dmean) = sum r*d - rmean * dsum - dmean * vR      (exact in s32)
// rw[] = the range block as packed u8 words.
template <int B>
__device__ __forceinline__ int refine_kov(const uint32_t *rw, int rmean, int vR, const uint8_t *__restrict__ pos_raw,
                                          int64_t pos, int dsum)
{
    constexpr int n = B * B;
    int kov = 0;
#pragma unroll
    for (int c = 0; c < n / 16; c++) {
        const uint4 d = __ldg((const uint4 *)(pos_raw + raw_offset<n>(pos, c)));
        const uint4 r = *(const uint4 *)(rw + 4 * c);  // registers (B <= 8) or a shared-memory broadcast (B = 16)
        kov = dp4a_uu(r.x, d.x, kov);
        kov = dp4a_uu(r.y, d.y, kov);
        kov = dp4a_uu(r.z, d.z, kov);
        kov = dp4a_uu(r.w, d.w, kov);
    }
    return kov - (rmean * dsum + (dsum / n) * vR);
}

// Calls consider(sweep position) for this lane's candidate of every flagged chunk of operand row i (a warp walks a
// row; lane = candidate within the chunk).  The row's 2 * n_chunks (<= 16) list lengths are read by as many lanes at
// once, a list (<= 32 entries) by one coalesced load: the loop has no dependent global loads besides the candidates
// themselves.  A row whose flag list overflowed is rescanned in full -- slow, exact.
// A chunk whose recorded upper bound does not exceed `th` -- the flag threshold of the row's FINAL lower bound --
// cannot hold a member of T (the search kernel's own criterion, applied with the bound it reached in the end): it
// is skipped without touching its candidates.  Most flags are such early records of a still-low bound.
template <class F>
__device__ __forceinline__ void for_each_flagged(int lane, int64_t i, int64_t rows_padded, int n_chunks, int64_t npos,
                                                 const int2 *__restrict__ flag_list, const int32_t *__restrict__ flag_cnt,
                                                 float th, F &&consider)
{
    const int n_lists = kFlagLists * n_chunks;  // (unit of the row, list of the unit): n_chunks <= 8
    const int my_cnt = lane < n_lists ? flag_cnt[((int64_t)(lane / kFlagLists) * rows_padded + i) * kFlagLists + (lane % kFlagLists)] : 0;
    const bool overflow = __any_sync(0xffffffffu, my_cnt > kFlagCap);
    if (!overflow) {
        for (int lh = 0; lh < n_lists; lh++) {
            const int cnt = __shfl_sync(0xffffffffu, my_cnt, lh);
            if (cnt == 0) continue;
            const int2 *lst = flag_list + (((int64_t)(lh / kFlagLists) * rows_padded + i) * kFlagLists + (lh % kFlagLists)) * kFlagCap;
            const int2 mine = lane < cnt ? lst[lane] : make_int2(0, 0);
            unsigned live = __ballot_sync(0xffffffffu, lane < cnt && __int_as_float(mine.y) > th);
            while (live) {
                const int e = __ffs(live) - 1;
                live &= live - 1;
                consider((int64_t)__shfl_sync(0xffffffffu, mine.x, e) * 32 + lane);
            }
        }
    } else {
        for (int64_t pos = lane; pos < npos; pos += 32) consider(pos);
    }
}

// One warp per range row, lane = candidate within a flagged chunk.  The winner is the
// lexicographic (error, index) minimum over every candidate of every flagged chunk plus domain
// 0 (which wins when the whole row ties, e.g. all scores 0) = the reference's first index with
// the smallest error.  A row whose flag list overflowed is rescanned in full -- slow, exact.
// Each lane runs the search kernel's filter once more on its own candidates (x bounded from the exact
// integer kov and a correctly rounded binary32 1/sqrt(varD)), so the reference's double-precision
// expression (FC:677-683) is only evaluated for candidates that can still win or tie.
// A group of n_img images: warp w refines row w % rows of image w / rows -- operand row image * rp_img + that row of the
// group, that image's planes, range sums, OpBLayout region (opb_stride bytes per image) and rows of `best`.
template <int B>
__global__ void __launch_bounds__(128)
k_umma_refine(const uint8_t *__restrict__ src, const int32_t *__restrict__ rsum, const uint8_t *__restrict__ pos_raw,
              const int4 *__restrict__ pos_info,
              const int2 *__restrict__ flag_list, const int32_t *__restrict__ flag_cnt,
              const uint32_t *__restrict__ row_lb, int n_chunks,
              int64_t rows_padded, int64_t rows, int64_t npos, const int64_t *__restrict__ dom0_pos,
              int32_t *__restrict__ best, Geom g, int64_t j0, int n_img, int64_t rp_img, size_t opb_stride)
{
    constexpr int n = B * B;
    constexpr int NW = n / 4;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t w = (int64_t)blockIdx.x * 4 + warp;
    if (w >= rows * n_img) return;
    const int64_t image = w >= rows ? w / rows : 0, il = w - image * rows;
    const int64_t i = image * rp_img + il;  // operand row == range block (the isometry extension has its own kernel)
    const int64_t j = j0 + il;
    src += image * g.W * g.H;
    rsum += image * g.NR;
    best += image * g.NR;
    pos_raw = image_region(pos_raw, image, opb_stride);
    pos_info = image_region(pos_info, image, opb_stride);
    dom0_pos = image_region(dom0_pos, image, opb_stride);
    int rmean;
    const int vR = centred_sum(rsum[j], n, &rmean);
    if (vR == 0) {  // FC:677-678 + FC:627: all errors are 0, the first candidate wins
        if (lane == 0) best[j] = 0;
        return;
    }
    const int xr = (int)(j % g.rpw), yr = (int)(j / g.rpw);
    // The range block as packed u8 words: registers for B <= 8; for B = 16 (64 words) shared memory, read back as
    // broadcasts -- the registers saved (128 -> see -Xptxas -v) buy the occupancy that hides the raw-pixel reads.
    constexpr bool RW_SMEM = B == 16;
    __shared__ __align__(16) uint32_t s_rw[RW_SMEM ? 4 : 1][RW_SMEM ? NW : 4];
    __align__(16) uint32_t rw_reg[RW_SMEM ? 4 : NW];
    const uint32_t *rw;
    if constexpr (RW_SMEM) {
        for (int w = lane; w < NW; w += 32) {
            const int k = 4 * w;
            s_rw[warp][w] = __ldg((const uint32_t *)(src + (int64_t)(yr * B + k / B) * g.W + xr * B + (k % B)));
        }
        __syncwarp();
        rw = s_rw[warp];
    } else {
#pragma unroll
        for (int w = 0; w < NW; w++) {
            const int k = 4 * w;
            rw_reg[w] = __ldg((const uint32_t *)(src + (int64_t)(yr * B + k / B) * g.W + xr * B + (k % B)));
        }
        rw = rw_reg;
    }
    float be = 10000000.0f;  // FC:615
    int bi = 0x7fffffff;
    const float tie_abs = (float)(vR * vR) * 4.76837158203125e-07f;  // vR^2 * 2^-21
    // lane-local lower bound of the row's max x and the flag threshold from it, seeded with the bound the search
    // kernel reached for this row
    float lb = __uint_as_float(row_lb[i]), th = lb > 0.0f ? flag_threshold(lb, tie_abs) : -1.0f;
    const float th_row = th;
    auto consider = [&](int64_t pos) {
        const int4 pi = __ldg(pos_info + pos);  // {domain index (-1: padding), varD, sum d, -}
        const int idx = pi.x;
        if (idx >= 0) {
            const int varD = pi.y;
            const int kov = refine_kov<B>(rw, rmean, vR, pos_raw, pos, pi.z);
            // x = |kov| / sqrt(varD) within (1 +- 2^-22): |kov| and varD < 2^24 are exact in binary32
            const float ax = varD > 0 ? fabsf((float)kov) * __frsqrt_rn((float)varD) : 0.0f;
            if (ax * (1.0f + 2.384185791015625e-07f) > th) {
                argmin_merge(be, bi, grey_error(kov, vR, __dsqrt_rn((double)varD)), idx);
                const float xlo = ax * (1.0f - 2.384185791015625e-07f);
                if (xlo > lb) { lb = xlo; th = flag_threshold(lb, tie_abs); }
            }
        }
    };
    if (lane == 0) consider(*dom0_pos);
    for_each_flagged(lane, i, rows_padded, n_chunks, npos, flag_list, flag_cnt, th_row, consider);
    warp_argmin(be, bi);
    if (lane == 0) best[j] = bi == 0x7fffffff ? 0 : bi;
}

// Isometry extension: refine of a whole range block by one warp.  The block's 8 operand rows (one per isometry,
// see k_umma_pack_ranges) share the running bound in the search kernel, so most of them carry no flagged chunk at
// all: the warp reads the 16 list lengths of a domain chunk (8 rows x 2 column halves, contiguous) with one load,
// skips the empty rows, and rebuilds the permuted range block (from a shared-memory copy) only for rows that have
// work.  The winner is the lexicographic (error, c, k) minimum = what an ascending (c, k) double loop with strict <
// yields; best[j] = c * 8 + k.
template <int B>
__global__ void __launch_bounds__(128)
k_umma_refine_iso(const uint8_t *__restrict__ src, const int32_t *__restrict__ rsum, const uint8_t *__restrict__ pos_raw,
                  const int4 *__restrict__ pos_info, const int2 *__restrict__ flag_list,
                  const int32_t *__restrict__ flag_cnt, const uint32_t *__restrict__ row_lb, int n_chunks,
                  int64_t rows_padded, int64_t ranges, int64_t npos,
                  const int64_t *__restrict__ dom0_pos, int32_t *__restrict__ best, Geom g, int64_t j0, int n_img, int64_t rp_img,
                  size_t opb_stride)
{
    constexpr int n = B * B;
    constexpr int NW = n / 4;
    __shared__ uint8_t s_blk[4][n];  // the range block of each of the block's 4 warps, raster order
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t w = (int64_t)blockIdx.x * 4 + warp;  // a group of images: see k_umma_refine
    if (w >= ranges * n_img) return;
    const int64_t image = w >= ranges ? w / ranges : 0, r = w - image * ranges;
    const int64_t i0 = image * rp_img + r * 8;  // the block's first operand row in the group
    const int64_t j = j0 + r;
    src += image * g.W * g.H;
    rsum += image * g.NR;
    best += image * g.NR;
    pos_raw = image_region(pos_raw, image, opb_stride);
    pos_info = image_region(pos_info, image, opb_stride);
    dom0_pos = image_region(dom0_pos, image, opb_stride);
    int rmean;
    const int vR = centred_sum(rsum[j], n, &rmean);
    if (vR == 0) {  // FC:677-678 + FC:627: all errors are 0, the first candidate wins
        if (lane == 0) best[j] = 0;
        return;
    }
    const int xr = (int)(j % g.rpw), yr = (int)(j / g.rpw);
    for (int w = lane; w < NW; w += 32) {
        const int k = 4 * w;
        ((uint32_t *)s_blk[warp])[w] = __ldg((const uint32_t *)(src + (int64_t)(yr * B + k / B) * g.W + xr * B + (k % B)));
    }
    __syncwarp();
    // The block permuted for each of the 8 isometries (same layout as the operand rows), built once per range block
    // in shared memory and read back as broadcasts.
    __shared__ __align__(16) uint32_t s_rw[4][8][NW];
    for (int t = lane; t < 8 * NW; t += 32) {
        const int kiso = t / NW, w = t % NW;
        uint32_t word = 0;
#pragma unroll
        for (int e = 0; e < 4; e++) {
            int ry, rx;  // the range pixel that T_kiso sends to domain pixel 4 * w + e
            iso_map(iso_inverse(kiso), B, (4 * w + e) / B, (4 * w + e) % B, &ry, &rx);
            word |= (uint32_t)s_blk[warp][ry * B + rx] << (8 * e);
        }
        s_rw[warp][kiso][w] = word;
    }
    __syncwarp();
    const uint32_t *rw = s_rw[warp][0];
    auto build = [&](int kiso) { rw = s_rw[warp][kiso]; };
    float be = 10000000.0f;  // FC:615
    int bi = 0x7fffffff;     // c * 8 + k
    const float tie_abs = (float)(vR * vR) * 4.76837158203125e-07f;  // vR^2 * 2^-21
    // lane-local bound / threshold, shared by the 8 isometries (they compete for one winner), seeded with the bound
    // the search kernel reached for this range block (its 8 operand rows publish into the first one's slot)
    float lb = __uint_as_float(row_lb[i0]), th = lb > 0.0f ? flag_threshold(lb, tie_abs) : -1.0f;
    const float th_row = th;
    auto consider = [&](int64_t pos, int kiso) {
        const int4 pi = __ldg(pos_info + pos);  // {domain index (-1: padding), varD, sum d, -}
        if (pi.x >= 0) {
            const int kov = refine_kov<B>(rw, rmean, vR, pos_raw, pos, pi.z);
            const float ax = pi.y > 0 ? fabsf((float)kov) * __frsqrt_rn((float)pi.y) : 0.0f;
            if (ax * (1.0f + 2.384185791015625e-07f) > th) {
                argmin_merge(be, bi, grey_error(kov, vR, __dsqrt_rn((double)pi.y)), pi.x * 8 + kiso);
                const float xlo = ax * (1.0f - 2.384185791015625e-07f);
                if (xlo > lb) { lb = xlo; th = flag_threshold(lb, tie_abs); }
            }
        }
    };
    build(0);
    if (lane == 0) consider(*dom0_pos, 0);  // (domain 0, identity) wins when the whole block ties
    int built = 0;
    bool overflow = false;
    for (int ch = 0; ch < n_chunks && !overflow; ch++) {
        // 8 * kFlagLists (<= 32) contiguous list lengths: operand row 8 r + k, list h of the unit at lane kFlagLists * k + h
        const int64_t base = ((int64_t)ch * rows_padded + i0) * kFlagLists;
        const int my_cnt = lane < 8 * kFlagLists ? flag_cnt[base + lane] : 0;
        if (__any_sync(0xffffffffu, my_cnt > kFlagCap)) { overflow = true; break; }
        for (int kiso = 0; kiso < 8; kiso++) {
            int any = 0;
            for (int h = 0; h < kFlagLists; h++) any |= __shfl_sync(0xffffffffu, my_cnt, kFlagLists * kiso + h);
            if (any == 0) continue;
            if (built != kiso) { build(kiso); built = kiso; }
#pragma unroll 1  // one copy of the candidate loop
            for (int h = 0; h < kFlagLists; h++) {
                const int cnt = __shfl_sync(0xffffffffu, my_cnt, kFlagLists * kiso + h);
                if (cnt == 0) continue;
                const int2 *lst = flag_list + (base + kFlagLists * kiso + h) * kFlagCap;
                const int2 mine = lane < cnt ? lst[lane] : make_int2(0, 0);
                unsigned live = __ballot_sync(0xffffffffu, lane < cnt && __int_as_float(mine.y) > th_row);  // see for_each_flagged
                while (live) {
                    const int e = __ffs(live) - 1;
                    live &= live - 1;
                    consider((int64_t)__shfl_sync(0xffffffffu, mine.x, e) * 32 + lane, kiso);
                }
            }
        }
    }
    if (overflow) {  // slow, exact: every candidate under every isometry
        for (int kiso = 0; kiso < 8; kiso++) {
            build(kiso);
            for (int64_t pos = lane; pos < npos; pos += 32) consider(pos, kiso);
        }
    }
    warp_argmin(be, bi);
    if (lane == 0) best[j] = bi == 0x7fffffff ? 0 : bi;
}

// RGB twin of k_umma_refine (see "RGB operands"): kov is rebuilt from the binary16 operand row of the
// candidate with a binary32 FMA chain -- exact, every partial sum being an integer below 2^24 -- and scored with the
// reference's all-float expression (FC:797-803).
template <int B>
__global__ void __launch_bounds__(128)
k_umma_refine_rgb(const uint8_t *__restrict__ src, const int32_t *__restrict__ rsum, const uint8_t *__restrict__ opB,
                  const int4 *__restrict__ pos_info, const int2 *__restrict__ flag_list, const int32_t *__restrict__ flag_cnt,
                  const uint32_t *__restrict__ row_lb, int n_chunks,
                  int64_t rows_padded, int64_t rows, int64_t npos, const int64_t *__restrict__ dom0_pos,
                  int32_t *__restrict__ best, Geom g, int64_t j0, int n_img, int64_t rp_img, size_t opb_stride)
{
    using L = Lay<B, true>;
    constexpr int n = B * B;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t w = (int64_t)blockIdx.x * 4 + warp;  // a group of images: see k_umma_refine
    if (w >= rows * n_img) return;
    const int64_t image = w >= rows ? w / rows : 0, il = w - image * rows;
    const int64_t i = image * rp_img + il;
    const int64_t j = j0 + il;
    src += image * 3 * g.W * g.H;
    rsum += image * 3 * g.NR;
    best += image * g.NR;
    opB = image_region(opB, image, opb_stride);
    pos_info = image_region(pos_info, image, opb_stride);
    dom0_pos = image_region(dom0_pos, image, opb_stride);
    int rm[3];
    const int vRi = centred_sum_rgb(rsum, g.NR, j, n, rm);
    const int rmsum = rm[0] + rm[1] + rm[2];
    if (vRi == 0) {  // FC:797 + FC:710: all errors are 0, the first candidate wins
        if (lane == 0) best[j] = 0;
        return;
    }
    const float vR = (float)vRi;
    const int xr = (int)(j % g.rpw), yr = (int)(j / g.rpw);
    const int64_t plane = (int64_t)g.W * g.H;
    // gR of the warp's range block lives in shared memory (broadcast reads): 64 registers less per thread, and the
    // occupancy they buy hides the latency of the scattered operand-row reads
    __shared__ float s_gR[4][n];
    float *gR = s_gR[warp];
    for (int k = lane; k < n; k += 32) {
        const uint8_t *q = src + (int64_t)(yr * B + k / B) * g.W + xr * B + (k % B);
        gR[k] = (float)((int)__ldg(q) + (int)__ldg(q + plane) + (int)__ldg(q + 2 * plane) - rmsum);
    }
    __syncwarp();
    float be = 10000000.0f;  // FC:698
    int bi = 0x7fffffff;
    const float tie_abs = (float)(vRi * vRi) * 4.76837158203125e-07f;  // vR^2 * 2^-21
    float lb = __uint_as_float(row_lb[i]), th = lb > 0.0f ? flag_threshold(lb, tie_abs) : -1.0f;  // see k_umma_refine
    const float th_row = th;
    auto consider = [&](int64_t pos) {
        const int4 pi = __ldg(pos_info + pos);  // {domain index (-1: padding), vD, -, -}
        const int idx = pi.x;
        if (idx >= 0) {
            const int row = (int)(pos % kTileN);
            uint8_t *const blob = const_cast<uint8_t *>(opB) + (pos / kTileN) * L::B_TILE_BYTES;
            // the reference's kov: sequential binary32 accumulation in pixel order (FC:781-792)
            float kov = 0.0f;
#pragma unroll 8
            for (int c = 0; c < n / 8; c++) {
                const uint4 d = __ldg((const uint4 *)rgb_dom_piece<B>(blob, row, c));
                const uint32_t w[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const float2 f = __half22float2(*(const __half2 *)&w[e]);
                    kov = rgb_kov_step(kov, gR[c * 8 + 2 * e], f.x);
                    kov = rgb_kov_step(kov, gR[c * 8 + 2 * e + 1], f.y);
                }
            }
            const float vD = (float)pi.y;
            const float ax = pi.y > 0 ? __fdiv_rn(fabsf(kov), vD) : 0.0f;  // x within (1 +- 2^-24)
            if (ax * (1.0f + 2.384185791015625e-07f) > th) {
                argmin_merge(be, bi, rgb_error(kov, vR, vD), idx);
                const float xlo = ax * (1.0f - 2.384185791015625e-07f);
                if (xlo > lb) { lb = xlo; th = flag_threshold(lb, tie_abs); }
            }
        }
    };
    if (lane == 0) consider(*dom0_pos);
    for_each_flagged(lane, i, rows_padded, n_chunks, npos, flag_list, flag_cnt, th_row, consider);
    warp_argmin(be, bi);
    if (lane == 0) best[j] = bi == 0x7fffffff ? 0 : bi;
}

// ---------------------------------------------------------------- host side ------------

inline int64_t pad_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }
inline uint64_t gcd_u64(uint64_t a, uint64_t b) { while (b) { uint64_t t = a % b; a = b; b = t; } return a; }

// A group of n_img images: every image's operand rows are padded on their own (rp_img, n_sb_img), the group's rows
// follow each other (rp, n_sb); the domain sweep (ntiles, npos, mult) is per image.
struct Plan {
    int64_t rp;     // rows padded to whole super-blocks (the whole group)
    int64_t rp_img; // ... per image
    int n_img, n_sb, n_sb_img, ntiles, n_chunks;
    uint32_t mult;  // sweep-order multiplier (see sweep_to_sorted)
    int64_t npos;   // ntiles * 128 sweep positions
};

// Split the domain sweep of a super-block into n_chunks units.  More units fill the last wave of num_sms CTAs
// better, but every unit adds flagged chunks for the refine step: the first unit of a row about
// 2 * (ln(chunks per list) + 0.58) (records of a random sequence, two column halves), every later one -- seeded
// with the bound the earlier ones reached -- about 2 * 1.5.  n_chunks minimises a small
// cost model of search + refine time; its constants are B200 measurements (clocks per domain tile of
// k_umma_search, whole-GPU nanoseconds per flagged chunk of k_umma_refine) -- only their ratio matters.
inline int rows_per_sb(const Geom &g) { return (g.C == 3 && g.B == 16 ? 2 : kAccs) * kBlockM; }  // Cfg<...>::NB * 128

inline Plan make_plan(const Geom &g, int64_t rows, int num_sms, int n_img = 1)
{
    Plan p;
    const int rows_sb = rows_per_sb(g);
    // an even number of 512-row super-blocks per image: CTA pairs (k_umma_search<..., PAIR>) take two at a time and
    // never straddle two images; padding rows are zero operands with vR = 0 (never flagged)
    p.n_img = n_img;
    p.rp_img = pad_up(rows, 2 * rows_sb);
    p.rp = p.rp_img * n_img;
    p.n_sb_img = (int)(p.rp_img / rows_sb);
    p.n_sb = p.n_sb_img * n_img;
    p.ntiles = (int)((g.ND + kTileN - 1) / kTileN);
    p.npos = (int64_t)p.ntiles * kTileN;
    p.n_chunks = 1;
    const double tile_s = (g.B == 16 ? (g.C == 3 ? 2300.0 : 4650.0) : (g.B == 8 ? 1550.0 : 1400.0)) / 1.9e9;
    const double flag_s = 0.11e-9 * (g.n / 64.0) * (g.n > 64 ? 0.7 : 1.0);
    double best_cost = 0;
    for (int c = 1; c <= 8 && c <= p.ntiles; c++) {
        const int64_t units = (int64_t)p.n_sb * c;
        const int64_t waves = (units + num_sms - 1) / num_sms;
        const double tiles_per_unit = (double)((p.ntiles + c - 1) / c);
        const double flags_per_row = 2.0 * (log(2.0 * tiles_per_unit) + 0.58) + 2.0 * (c - 1) * 1.5;
        const double cost = (double)waves * tiles_per_unit * tile_s + (double)rows * n_img * flags_per_row * flag_s;
        if (c == 1 || cost < best_cost * 0.98) { best_cost = cost; p.n_chunks = c; }
    }
    const uint64_t nch = (uint64_t)p.ntiles * kChunksPerTile;
    uint64_t m = (uint64_t)((double)nch * 0.6180339887498949) | 1u;  // golden-ratio stride, odd
    while (gcd_u64(m, nch) != 1) m += 2;
    p.mult = nch <= 8 ? 1u : (uint32_t)(m % nch);
    return p;
}

// opB workspace: per image [tile blobs][pos_dom s32][pos_info int4][pos_raw u8 x n][dom0 pos s64], `stride` bytes
// per image (the offsets are image 0's), then [sort of the group's domains: keys x2, vals x2, digit histograms]
template <int B, bool F16>
struct OpBLayout {
    size_t off_posdom, off_posinfo, off_posraw, off_dom0, stride, off_keys0, off_keys1, off_vals0, off_vals1, off_temp,
        temp_bytes, total;
    OpBLayout(const Geom &g, const Plan &p)
    {
        size_t o = (size_t)p.ntiles * Lay<B, F16>::B_TILE_BYTES;
        auto take = [&](size_t bytes) { size_t at = (o + 255) & ~(size_t)255; o = at + bytes; return at; };
        off_posdom = take((size_t)p.npos * 4);
        off_posinfo = take((size_t)p.npos * 16);
        off_posraw = take((size_t)p.npos * (B * B));
        off_dom0 = take(16);  // s64 sweep position of domain 0
        stride = (o + 255) & ~(size_t)255;
        o = stride * p.n_img;
        const int64_t nd = g.ND * p.n_img;
        off_keys0 = take((size_t)nd * 4);
        off_keys1 = take((size_t)nd * 4);
        off_vals0 = take((size_t)nd * 4);
        off_vals1 = take((size_t)nd * 4);
        temp_bytes = sort_hist_bytes(nd);
        off_temp = take(temp_bytes + 256);
        total = o + 256;
    }
};

// opA workspace: [A blobs][vR s32][flag_cnt][flag_list][row_lb u32][row_norm f32], per (unit, operand row) of
// flag_cnt a header of kCntSlots list lengths (s32; the first kFlagLists are used) and of flag_list kFlagLists lists
// of kFlagCap entries (s32 chunk id, f32 bound)
template <int B, bool F16>
struct OpALayout {
    static constexpr int kCntSlots = 4;
    size_t off_vR, off_cnt, off_list, off_lb, off_norm, total;
    explicit OpALayout(const Plan &p)
    {
        off_vR = (size_t)p.n_sb * Lay<B, F16>::A_SB_BYTES;
        off_cnt = off_vR + (size_t)p.rp * 4;
        off_list = off_cnt + (size_t)p.rp * p.n_chunks * kCntSlots * 4;  // 8-byte aligned: the blobs are, and rp is even
        off_lb = off_list + (size_t)p.rp * p.n_chunks * kFlagLists * kFlagCap * sizeof(int2);
        off_norm = off_lb + (size_t)p.rp * 4;
        total = off_norm + (size_t)p.rp * 4 + 1024;
    }
};

template <int B, bool F16>
size_t opA_bytes_t(const Geom &g, int64_t rows, int num_sms, int n_img = 1)
{
    return OpALayout<B, F16>(make_plan(g, rows, num_sms, n_img)).total;
}

using KernelT = void (*)(const uint8_t *, const uint8_t *, const int32_t *, const float *, int2 *, int32_t *, uint32_t *, int, int,
                         int, int, int64_t, int32_t *, int64_t, volatile int *, int, int64_t);

// CTA pairs exist for the kind::f16 kernels (B = 4, 8: grey, RGB and the isometry extension; two issuing warps) and for
// the K-split B = 16 configurations (kind::i8 grey, kind::f16 RGB; one issuing warp, each CTA loads half of either part
// of a tile).  Default where measured faster: B = 8 (17.6 against 20.8 ms at 4096^2) and B = 16 (2.47 against 2.77 ms);
// B = 4 is bound by its epilogue (K = 16 keeps the tensor pipe a quarter busy) and loses 4 % to the pair's extra
// barrier traffic.
template <int B, bool F16>
constexpr bool pair_capable() { return F16 || B == 16; }
template <int B, bool F16>
constexpr bool pair_default() { return pair_capable<B, F16>() && B >= 8; }

// Can a cluster of two CTAs of this kernel be co-scheduled on this device (it cannot under some MIG / MPS partitions)?
inline bool pair_launchable(KernelT kern, int smem_bytes)
{
    // asked once per (kernel, device): the occupancy query is a host-side driver call
    static std::mutex mu;
    static std::vector<std::tuple<KernelT, int, bool>> known;
    int dev = 0;
    cudaGetDevice(&dev);
    {
        std::lock_guard<std::mutex> lock(mu);
        for (const auto &k : known)
            if (std::get<0>(k) == kern && std::get<1>(k) == dev) return std::get<2>(k);
    }
    const bool ok = [&]() {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = (size_t)smem_bytes;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, (const void *)kern, &cfg) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return n >= 1;
    }();
    std::lock_guard<std::mutex> lock(mu);
    known.emplace_back(kern, dev, ok);
    return ok;
}

// n_img > 1: a group of images, every range of each (see launch_search_umma).
template <int B, bool F16>
int launch_t(const Work &w, const Geom &g, int64_t j0, int64_t j1, int num_sms, cudaStream_t s, const char **err,
             cudaEvent_t k0, cudaEvent_t k1, int pair_mode, int *pair_used, int32_t *dump, int64_t dump_ld, int *status_dev,
             int n_img)
{
    using L = Lay<B, F16>;
    if (j1 <= j0) return 0;
    const int64_t rows = (j1 - j0) * g.n_iso;  // operand rows of an image: one per (range, isometry)
    Plan p = make_plan(g, rows, num_sms, n_img);
    const int64_t rp = p.rp;
    uint8_t *opA = w.opA;
    const OpALayout<B, F16> la(p);
    int32_t *vR = (int32_t *)(opA + la.off_vR);
    int32_t *flag_cnt = (int32_t *)(opA + la.off_cnt);
    int2 *flag_list = (int2 *)(opA + la.off_list);
    uint32_t *row_lb = (uint32_t *)(opA + la.off_lb);  // per operand row: best lower bound of max x reached by finished units
    float *row_norm = (float *)(opA + la.off_norm);    // per operand row: >= ||gR||_2 (RGB at blockgroesse 16)
    const bool rgb = g.C == 3;                        // kind::f16 only (see "RGB operands")
    if (rgb && !F16) { *err = "the RGB tensor path is kind::f16 only"; return -1; }
    OpBLayout<B, F16> lay(g, p);
    int32_t *pos_dom = (int32_t *)(w.opB + lay.off_posdom);
    int4 *pos_info = (int4 *)(w.opB + lay.off_posinfo);
    uint8_t *pos_raw = w.opB + lay.off_posraw;
    int64_t *dom0 = (int64_t *)(w.opB + lay.off_dom0);
    int launches = 0;
    cudaError_t ce;
    // 1. domains by increasing varD (a group: by image, then varD -- the image index is a fourth key digit, so a group
    // holds at most 256 images)
    uint32_t *keys0 = (uint32_t *)(w.opB + lay.off_keys0), *keys1 = (uint32_t *)(w.opB + lay.off_keys1);
    int32_t *vals0 = (int32_t *)(w.opB + lay.off_vals0), *vals1 = (int32_t *)(w.opB + lay.off_vals1);
    if (n_img < 1 || n_img > 256) { *err = "a tcgen05 group holds 1 to 256 images"; return -1; }
    const int64_t nd = g.ND * n_img;
    if (rgb) k_umma_sortkeys_rgb<<<(unsigned)((nd + 255) / 256), 256, 0, s>>>(w.dsum, g.n, g.ND, nd, keys0, vals0);
    else k_umma_sortkeys<<<(unsigned)((nd + 255) / 256), 256, 0, s>>>(w.dsum, w.dsq, g.n, g.ND, nd, keys0, vals0);
    const int passes = n_img > 1 ? 4 : 3;
    launches += 1 + launch_sort_pairs(keys0, vals0, keys1, vals1, (uint32_t *)(w.opB + lay.off_temp), nd, passes, s);
    const int32_t *perm = passes & 1 ? vals1 : vals0;  // domains by increasing key
    // 2. operand blobs
    if constexpr (F16) {
        if (rgb) {
            launches += launch_sum_planes(w.dec, w.dec3, g, s, n_img);
            k_umma_pack_domains_rgb<B><<<(unsigned)((p.npos * n_img + 127) / 128), 128, 0, s>>>(
                w.dec3, w.dsum, perm, w.opB, pos_dom, pos_info, dom0, g, p.ntiles, p.mult, p.npos, lay.stride);
            k_umma_pack_ranges_rgb<B><<<(unsigned)((rp + 127) / 128), 128, 0, s>>>(w.src, w.rsum, opA, vR, B == 16 ? row_norm : nullptr, g, j0, j1,
                                                                                p.rp_img, n_img);
        }
    }
    if (!rgb) {
        k_umma_pack_domains<B, F16><<<(unsigned)((p.npos * n_img + 127) / 128), 128, 0, s>>>(
            w.dec, w.dsum, w.dsq, perm, w.opB, pos_dom, pos_info, pos_raw, dom0, g, p.ntiles, p.mult, p.npos, lay.stride);
        k_umma_pack_ranges<B, F16><<<(unsigned)((rp + 127) / 128), 128, 0, s>>>(w.src, w.rsum, opA, vR, g, j0, j1, p.rp_img, n_img);
    }
    launches += 2;
    // 3. the fused search: CTA pairs on request (FIC_UMMA_PAIR_ON / _OFF), else where measured faster (pair_default)
    bool pair = false;
    const bool group = n_img > 1;
    if (dump && group) { *err = "the accumulator dump takes one image"; return -1; }
    KernelT kern = dump ? k_umma_search<B, F16, false, true> : group ? k_umma_search<B, F16, false, false, true> : k_umma_search<B, F16, false, false>;
    if constexpr (pair_capable<B, F16>()) {
        pair = (pair_mode == FIC_UMMA_PAIR_ON || (pair_mode != FIC_UMMA_PAIR_OFF && pair_default<B, F16>())) && num_sms >= 2;
        if (pair) {
            KernelT pk = dump ? k_umma_search<B, F16, true, true> : group ? k_umma_search<B, F16, true, false, true> : k_umma_search<B, F16, true, false>;
            ce = cudaFuncSetAttribute(pk, cudaFuncAttributeMaxDynamicSharedMemorySize, L::SMEM_BYTES);
            if (ce != cudaSuccess) { *err = cudaGetErrorString(ce); return -1; }
            if (pair_launchable(pk, L::SMEM_BYTES)) kern = pk;
            else pair = false;  // no co-scheduled CTA pairs on this device / partition: the single-CTA kernel
        }
    }
    if (pair_used) *pair_used = pair ? 1 : 0;
    ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::SMEM_BYTES);
    if (ce != cudaSuccess) { *err = cudaGetErrorString(ce); return -1; }
    int n_units = pair ? (p.n_sb / 2) * p.n_chunks : p.n_sb * p.n_chunks;
    const int slots = pair ? num_sms / 2 : num_sms;  // CTAs, or CTA pairs (one TPC each)
    int grid = (n_units < slots ? n_units : slots) * (pair ? 2 : 1);
    if (k0) cudaEventRecord(k0, s);
    cudaMemsetAsync(row_lb, 0, (size_t)rp * 4, s);
    {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)grid);
        cfg.blockDim = dim3(kThreads);
        cfg.dynamicSmemBytes = L::SMEM_BYTES;
        cfg.stream = s;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 2;
        at[0].val.clusterDim.y = 1;
        at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = pair ? 1 : 0;
        const uint8_t *opA_c = opA, *opB_c = w.opB;
        const int32_t *vR_c = vR;
        const float *norm_c = row_norm;
        const int iso_shift = g.n_iso > 1 ? 3 : 0;
        volatile int *status_v = status_dev;
        ce = cudaLaunchKernelEx(&cfg, kern, opA_c, opB_c, vR_c, norm_c, flag_list, flag_cnt, row_lb, p.n_sb, p.n_chunks, p.ntiles, iso_shift,
                                rp, dump, dump_ld, status_v, p.n_sb_img, (int64_t)lay.stride);
        if (ce != cudaSuccess) { *err = cudaGetErrorString(ce); return -1; }
    }
    if (k1) cudaEventRecord(k1, s);
    // 4. exact refine of the flagged chunks
    if (rgb) {
        if constexpr (F16)
            k_umma_refine_rgb<B><<<(unsigned)((rows * n_img + 3) / 4), 128, 0, s>>>(
                w.src, w.rsum, w.opB, pos_info, flag_list, flag_cnt, row_lb, p.n_chunks, rp, rows, p.npos, dom0, w.best, g, j0, n_img,
                p.rp_img, lay.stride);
    } else if (g.n_iso > 1)
        k_umma_refine_iso<B><<<(unsigned)(((j1 - j0) * n_img + 3) / 4), 128, 0, s>>>(
            w.src, w.rsum, pos_raw, pos_info, flag_list, flag_cnt, row_lb, p.n_chunks, rp, j1 - j0, p.npos, dom0, w.best, g, j0, n_img,
            p.rp_img, lay.stride);
    else
        k_umma_refine<B><<<(unsigned)((rows * n_img + 3) / 4), 128, 0, s>>>(w.src, w.rsum, pos_raw, pos_info, flag_list, flag_cnt,
                                                                            row_lb, p.n_chunks, rp, rows, p.npos, dom0, w.best, g, j0,
                                                                            n_img, p.rp_img, lay.stride);
    launches += 2;
    ce = cudaGetLastError();
    if (ce != cudaSuccess) { *err = cudaGetErrorString(ce); return -1; }
    return launches;
}

// Dispatch on (block size, MMA kind): grey B = 16 runs kind::i8 only, kind::f16 at B = 16 is the RGB configuration.
#define FIC_UMMA_DISPATCH(B_, F_, EXPR_I8_4, EXPR_I8_8, EXPR_I8_16, EXPR_F16_4, EXPR_F16_8, EXPR_F16_16) \
    ((B_) == 16 ? ((F_) ? (EXPR_F16_16) : (EXPR_I8_16)) : ((F_) ? ((B_) == 8 ? (EXPR_F16_8) : (EXPR_F16_4)) : ((B_) == 8 ? (EXPR_I8_8) : (EXPR_I8_4))))

}  // namespace

// kind::f16 with binary32 accumulation is exact while every partial sum stays below 2^24:
// |kov| <= n * 255^2 = 4.2e6 (B = 8), 2.6e5 (B = 4).  B = 16 (1.66e7, and half the tensor rate of kind::i8
// for a kernel that is tensor-bound there) stays on kind::i8.
int umma_default_kind(const Geom &g) { return g.B == 16 ? FIC_UMMA_KIND_I8 : FIC_UMMA_KIND_F16; }

static bool use_f16(const Geom &g, int kind)
{
    if (g.C == 3) return true;  // the RGB operands need binary16 (see "RGB operands"), at every block size
    if (g.B == 16) return false;
    return (kind == FIC_UMMA_KIND_AUTO ? umma_default_kind(g) : kind) == FIC_UMMA_KIND_F16;
}

void umma_debug_positions(const Work &w, const Geom &g, int64_t rows, int num_sms, int kind, const int32_t **d_pos_dom,
                          int64_t *npos)
{
    Plan p = make_plan(g, rows, num_sms);
    *npos = p.npos;
    const size_t off = FIC_UMMA_DISPATCH(g.B, use_f16(g, kind), (OpBLayout<4, false>(g, p).off_posdom),
                                         (OpBLayout<8, false>(g, p).off_posdom), (OpBLayout<16, false>(g, p).off_posdom),
                                         (OpBLayout<4, true>(g, p).off_posdom), (OpBLayout<8, true>(g, p).off_posdom),
                                         (OpBLayout<16, true>(g, p).off_posdom));
    *d_pos_dom = (const int32_t *)(w.opB + off);
}

// Returns the measured dense rate in TOP/s (2 ops per MAC) of kind::i8 (f16 = 0) or kind::f16 with M = 128 and
// N = n_cols (128 or 256), best of `reps` launches.
double measure_mma_peak(int num_sms, cudaStream_t s, int reps, int f16, int n_cols, const char **err)
{
    const int smem = 200 * 1024;  // far more than needed: guarantees one CTA (one 512-column TMEM allocation) per SM
    void (*kern)(int, uint32_t) = f16 ? (n_cols == 128 ? k_mma_peak<true, 128> : k_mma_peak<true, 256>)
                                      : (n_cols == 128 ? k_mma_peak<false, 128> : k_mma_peak<false, 256>);
    cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (ce != cudaSuccess) { *err = cudaGetErrorString(ce); return -1.0; }
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    const int iters = 200000 * 256 / n_cols;  // ~13 ms at full rate and 1.9 GHz
    const double k_per_mma = f16 ? 16.0 : 32.0;
    double best = 0.0;
    for (int r = 0; r < reps + 1; r++) {
        cudaEventRecord(e0, s);
        kern<<<num_sms, 128, smem, s>>>(iters, 0x9e3779b9u + r);
        cudaEventRecord(e1, s);
        ce = cudaStreamSynchronize(s);
        if (ce != cudaSuccess) { *err = cudaGetErrorString(ce); best = -1.0; break; }
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        double tops = 2.0 * 128.0 * (double)n_cols * k_per_mma * (double)iters * num_sms / (ms * 1e-3) / 1e12;
        if (r > 0 && tops > best) best = tops;  // launch 0 is the warm-up
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return best;
}

// ---------------------------------------------------------------- kind::f16 self-test -

namespace {

// Integer reference of every accumulator the search kernel dumped.  Grey: kov[i][pos] = sum (r - rmean)(d - dmean);
// RGB (g.C == 3): sum gR * gD with the channel-summed centred values, 0 for a domain with vD == 0 (its operand row
// is zeroed, see "RGB operands").
__global__ void k_umma_selftest_check(const uint8_t *__restrict__ src, const uint8_t *__restrict__ dec,
                                      const int32_t *__restrict__ rsum, const int32_t *__restrict__ dsum,
                                      const int32_t *__restrict__ pos_dom, const int32_t *__restrict__ dump, int64_t dump_ld,
                                      int64_t npos, Geom g, unsigned int *__restrict__ bad)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= g.NR * npos) return;
    const int64_t i = t / npos, pos = t % npos;
    const int j = pos_dom[pos];
    if (j < 0) return;
    const int B = g.B, n = g.n;
    int rmean = 0, dmean = 0, vd = 0;
    for (int c = 0; c < g.C; c++) {
        int rm, dm;
        centred_sum(rsum[(int64_t)c * g.NR + i], n, &rm);
        vd += centred_sum(dsum[(int64_t)c * g.ND + j], n, &dm);
        rmean += rm;
        dmean += dm;
    }
    const uint8_t *r = src + (int64_t)((i / g.rpw) * B) * g.W + (i % g.rpw) * B;
    const uint8_t *d = dec + (int64_t)((j / g.dpw) * g.step) * g.sw + (j % g.dpw) * g.step;
    const int64_t rplane = (int64_t)g.W * g.H, dplane = (int64_t)g.sw * g.sh;
    int kov = 0;
    for (int k = 0; k < n; k++) {
        int rv = -rmean, dv = -dmean;
        for (int c = 0; c < g.C; c++) {
            rv += (int)r[c * rplane + (int64_t)(k / B) * g.W + k % B];
            dv += (int)d[c * dplane + (int64_t)(k / B) * g.sw + k % B];
        }
        kov += rv * dv;
    }
    if (g.C == 3 && vd == 0) kov = 0;
    if (dump[i * dump_ld + pos] != kov) atomicAdd(bad, 1u);
}

}  // namespace

// Runs the kind::f16 search on a 128 x 128 test image that mixes the largest covariances the operands can
// produce (0 / 255 cells), noise and smooth content, dumps every accumulator and compares it with integer
// arithmetic.  1: every binary32 accumulator held the exact integer; 0: not (the caller then uses kind::i8);
// < 0: CUDA error.  The encoder's results never depend on this (the refine step recomputes kov in s32), but a
// device whose f16 tensor path rounded would flag the wrong chunks.
int umma_f16_selftest(int num_sms, cudaStream_t s, const char **err)
{
    const int W = 128, B = 8;
    Geom g, g3;  // the grey pass and the RGB pass (three equal channels: 9 x the grey covariances, up to 9.3e6)
    if (make_geom(W, W, B, 2 * (W / B) - 3, FIC_MODE_GREY, &g, err) || make_geom(W, W, B, 2 * (W / B) - 3, FIC_MODE_RGB, &g3, err))
        return -1;
    std::vector<uint8_t> img((size_t)W * W);
    for (int y = 0; y < W; y++)
        for (int x = 0; x < W; x++) {
            uint32_t hpix = (uint32_t)(y * W + x) * 2654435761u;
            hpix ^= hpix >> 15; hpix *= 0x2c1b3c6du; hpix ^= hpix >> 12;
            uint32_t hcell = (uint32_t)((y / 4) * W + x / 4) * 2246822519u;
            hcell ^= hcell >> 13; hcell *= 0x9e3779b1u; hcell ^= hcell >> 16;
            int v;
            if (y < 64 && x < 64) v = (hcell >> 31) ? 255 : 0;          // 0 / 255 in 4x4 cells
            else if (y < 64) v = (int)(hpix >> 24);                      // noise
            else if (x < 64) v = (hpix >> 31) ? 255 : 0;                 // 0 / 255 per pixel
            else v = (3 * x + 2 * y + (int)(hpix >> 29)) & 255;          // ramps
            img[(size_t)y * W + x] = (uint8_t)v;
        }
    Work w;
    Plan p = make_plan(g, g.NR, num_sms);
    const int64_t dump_ld = p.npos;
    int32_t *dump = nullptr;
    unsigned int *bad = nullptr;
    cudaError_t ce = cudaSuccess;
    auto alloc = [&](void **ptr, size_t bytes) { if (ce == cudaSuccess) ce = cudaMalloc(ptr, bytes); };
    alloc((void **)&w.src, 3 * (size_t)W * W);
    alloc((void **)&w.dec, 3 * (size_t)g.sw * g.sh);
    alloc((void **)&w.dec3, 2 * (size_t)g.sw * g.sh);
    alloc((void **)&w.dsum, 3 * 4 * g.ND);
    alloc((void **)&w.dsq, 3 * 4 * g.ND);
    alloc((void **)&w.rsum, 3 * 4 * g.NR);
    alloc((void **)&w.best, 4 * g.NR);
    alloc((void **)&w.opA, opA_bytes_t<8, true>(g, g.NR, num_sms));
    alloc((void **)&w.opB, OpBLayout<8, true>(g, p).total);
    alloc((void **)&dump, (size_t)p.rp * dump_ld * 4);
    alloc((void **)&bad, 4);
    int result = -1;
    if (ce == cudaSuccess) {
        for (int c = 0; c < 3; c++) cudaMemcpyAsync(w.src + (size_t)c * W * W, img.data(), img.size(), cudaMemcpyHostToDevice, s);
        cudaMemsetAsync(bad, 0, 4, s);
        bool launched = true;
        for (const Geom *gp : {(const Geom *)&g, (const Geom *)&g3}) {
            cudaMemsetAsync(dump, 0x7f, (size_t)p.rp * dump_ld * 4, s);
            launch_decimate(w.src, w.dec, *gp, s);
            launch_domain_stats(w.dec, w.dsum, w.dsq, *gp, s);
            launch_range_stats(w.src, w.rsum, *gp, s);
            if (launch_t<8, true>(w, *gp, 0, gp->NR, num_sms, s, err, nullptr, nullptr, FIC_UMMA_PAIR_AUTO, nullptr, dump, dump_ld,
                                  nullptr, 1) < 0) {
                launched = false;
                break;
            }
            const int64_t total = gp->NR * p.npos;
            k_umma_selftest_check<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(
                w.src, w.dec, w.rsum, w.dsum, (const int32_t *)(w.opB + OpBLayout<8, true>(g, p).off_posdom), dump, dump_ld,
                p.npos, *gp, bad);
        }
        if (launched) {
            unsigned int hbad = 1;
            ce = cudaMemcpyAsync(&hbad, bad, 4, cudaMemcpyDeviceToHost, s);
            if (ce == cudaSuccess) ce = cudaStreamSynchronize(s);
            if (ce == cudaSuccess) result = hbad == 0 ? 1 : 0;
        }
    }
    if (ce != cudaSuccess) { *err = cudaGetErrorString(ce); result = -1; }
    for (void *ptr : {(void *)w.src, (void *)w.dec, (void *)w.dec3, (void *)w.dsum, (void *)w.dsq, (void *)w.rsum, (void *)w.best, (void *)w.opA,
                      (void *)w.opB, (void *)dump, (void *)bad})
        if (ptr) cudaFree(ptr);
    return result;
}

// Probe / test entry of the in-tree radix sort: sorts n device pairs by the low 24 key bits (stable); the result is
// written to (d_keys_out, d_vals_out).  Allocates its own histogram scratch.  0 or a CUDA error code.
int umma_debug_sort(uint32_t *d_keys, int32_t *d_vals, uint32_t *d_keys_out, int32_t *d_vals_out, int64_t n, cudaStream_t s)
{
    uint32_t *hist = nullptr;
    cudaError_t ce = cudaMalloc((void **)&hist, sort_hist_bytes(n) + 256);
    if (ce != cudaSuccess) return (int)ce;
    launch_sort_pairs(d_keys, d_vals, d_keys_out, d_vals_out, hist, n, 3, s);
    ce = cudaStreamSynchronize(s);
    cudaFree(hist);
    return (int)ce;
}

// Bare loop of the CTA-pair instruction shape (cta_group::2, M = 256, N = 128): TOP/s, best of `reps`; tmem_bases (if
// not null) receives the TMEM base address each of the first 4 CTAs was given.
double measure_mma_peak_pair(int num_sms, cudaStream_t s, int reps, int f16, uint32_t *tmem_bases, const char **err)
{
    const int smem = 200 * 1024;
    void (*kern)(int, uint32_t, uint32_t *) = f16 ? k_mma_peak_pair<true> : k_mma_peak_pair<false>;
    cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (ce != cudaSuccess) { *err = cudaGetErrorString(ce); return -1.0; }
    uint32_t *d_out = nullptr;
    if (cudaMalloc((void **)&d_out, 4 * (size_t)num_sms) != cudaSuccess) { *err = "cudaMalloc"; return -1.0; }
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    const int iters = 200000 * 2;
    const double k_per_mma = f16 ? 16.0 : 32.0;
    const int grid = num_sms / 2 * 2;
    double best = 0.0;
    for (int r = 0; r < reps + 1; r++) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)grid);
        cfg.blockDim = dim3(128);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = s;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 2;
        at[0].val.clusterDim.y = 1;
        at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        cudaEventRecord(e0, s);
        ce = cudaLaunchKernelEx(&cfg, kern, iters, (uint32_t)(0x9e3779b9u + r), d_out);
        cudaEventRecord(e1, s);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(s);
        if (ce != cudaSuccess) { *err = cudaGetErrorString(ce); best = -1.0; break; }
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        double tops = 2.0 * 256.0 * 128.0 * k_per_mma * (double)iters * (grid / 2) / (ms * 1e-3) / 1e12;
        if (r > 0 && tops > best) best = tops;
    }
    if (tmem_bases && best >= 0.0) cudaMemcpy(tmem_bases, d_out, 16, cudaMemcpyDeviceToHost);
    cudaFree(d_out);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return best;
}

bool umma_applicable(const Geom &g)
{
    if (g.wk != g.dpw || g.wk != g.dph) return false;
    if (g.C == 3) return g.n_iso == 1 && (g.B == 4 || g.B == 8 || g.B == 16);  // kind::f16 only
    return g.B == 4 || g.B == 8 || g.B == 16;
}

size_t umma_opA_bytes(const Geom &g, int64_t j0, int64_t j1, int num_sms, int kind, int n_images)
{
    const int64_t rows = (j1 - j0) * g.n_iso;  // operand rows: one per (range, isometry)
    return FIC_UMMA_DISPATCH(g.B, use_f16(g, kind), (opA_bytes_t<4, false>(g, rows, num_sms, n_images)),
                             (opA_bytes_t<8, false>(g, rows, num_sms, n_images)), (opA_bytes_t<16, false>(g, rows, num_sms, n_images)),
                             (opA_bytes_t<4, true>(g, rows, num_sms, n_images)), (opA_bytes_t<8, true>(g, rows, num_sms, n_images)),
                             (opA_bytes_t<16, true>(g, rows, num_sms, n_images)));
}

size_t umma_opB_bytes(const Geom &g, int kind, int n_images)
{
    Plan p = make_plan(g, rows_per_sb(g), 148, n_images);  // the opB layout depends on the pool and the image count only
    return FIC_UMMA_DISPATCH(g.B, use_f16(g, kind), (OpBLayout<4, false>(g, p).total), (OpBLayout<8, false>(g, p).total),
                             (OpBLayout<16, false>(g, p).total), (OpBLayout<4, true>(g, p).total),
                             (OpBLayout<8, true>(g, p).total), (OpBLayout<16, true>(g, p).total));
}

int launch_search_umma(const Work &w, const Geom &g, int64_t j0, int64_t j1, int num_sms, cudaStream_t s,
                       const char **err, int kind, cudaEvent_t k0, cudaEvent_t k1, int pair, int *pair_used,
                       int32_t *dump, int64_t dump_ld, int *status_dev, int n_images)
{
#define FIC_UMMA_ARGS w, g, j0, j1, num_sms, s, err, k0, k1, pair, pair_used, dump, dump_ld, status_dev, n_images
    return FIC_UMMA_DISPATCH(g.B, use_f16(g, kind), (launch_t<4, false>(FIC_UMMA_ARGS)), (launch_t<8, false>(FIC_UMMA_ARGS)),
                             (launch_t<16, false>(FIC_UMMA_ARGS)), (launch_t<4, true>(FIC_UMMA_ARGS)),
                             (launch_t<8, true>(FIC_UMMA_ARGS)), (launch_t<16, true>(FIC_UMMA_ARGS)));
#undef FIC_UMMA_ARGS
}

}  // namespace fic
