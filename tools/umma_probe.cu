// umma_probe -- development probe for the tcgen05 fused search (not part of the product).
//
//   umma_probe check|time <B> <W> [pattern] [kind] [pair]
//     check : dump every accumulator (kov) and compare with a CPU integer dot
//             product, then compare winners with the direct CUDA-core search
//     time  : no dump; time the fused search (k0 / k1 events around k_umma_search) and the
//             direct search, compare winners
//     B       4 | 8 | 16   W = H, multiple of B
//     pattern 0 = noise, 1 = structured, 2 = flat + sparse dots (tie-heavy), 3 = binary 0/255 noise,
//             4 = binary 0/255 in 4x4 pixel cells (the largest |kov| the operands can produce)
//     kind    0 = auto, 1 = kind::i8, 2 = kind::f16 (B = 16 always runs kind::i8)
//     pair    0 = auto, 1 = off, 2 = on (FIC_UMMA_PAIR_*)
//   umma_probe peak : bare tcgen05.mma loops: tensor-pipe rate by kind and MMA shape
//   umma_probe ldtm | alu | mix | chain | sort : micro-benchmarks and the radix-sort check (below)
//
// Runs each experiment in its own process so that a fault cannot poison the next one;
// every mbarrier wait in the kernel is bounded (trap + status code).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../fractal-image-compression_b200/csrc/fic_device.cuh"

using namespace fic;

#define CK(x)                                                                                  \
    do {                                                                                       \
        cudaError_t e_ = (x);                                                                  \
        if (e_ != cudaSuccess) {                                                               \
            printf("CUDA error %s at %s:%d (%s)\n", cudaGetErrorString(e_), __FILE__, __LINE__, #x); \
            if (g_status) printf("kernel status code: %d\n", *g_status);                      \
            exit(3);                                                                           \
        }                                                                                      \
    } while (0)

static volatile int *g_status = nullptr;

static uint32_t lowbias32(uint32_t x)
{
    x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
    return x;
}

static int tri(int v, int period)
{
    int p = ((v % period) + period) % period;
    int half = period / 2;
    int t = p < half ? p : period - p;
    return t * 255 / half;
}

static void make_image(std::vector<uint8_t> &img, int W, int H, int pattern, uint32_t seed)
{
    img.resize((size_t)W * H);
    for (int y = 0; y < H; y++)
        for (int x = 0; x < W; x++) {
            uint32_t h = lowbias32((uint32_t)(y * W + x) + seed * 0x9E3779B9u);
            int v;
            if (pattern == 0) v = h >> 24;
            else if (pattern == 1) {
                v = (tri(x + (int)seed, 97) + tri(3 * y + x, 211) + tri((x * y) / 64, 151)) / 3 + (int)((h >> 28)) - 8;
                v = v < 0 ? 0 : (v > 255 ? 255 : v);
            } else if (pattern == 2) {
                v = 100 + ((h & 0xff) == 0 ? (int)((h >> 8) & 3) + 1 : 0);
            } else if (pattern == 3) {
                v = (h >> 31) ? 255 : 0;
            } else {
                uint32_t hc = lowbias32((uint32_t)((y / 4) * W + (x / 4)) + seed * 0x9E3779B9u);
                v = (hc >> 31) ? 255 : 0;
            }
            img[(size_t)y * W + x] = (uint8_t)v;
        }
}

// ---- TMEM read-bandwidth microbenchmark ("ldtm" mode) -----------------------------------------
// `nw` warps per SM sub-partition issue `iters` tcgen05.ld.32x32b.x32 (4 KB each) back to back, waiting
// for every `batch`-th load.  Reports clocks per load per sub-partition.
__global__ void __launch_bounds__(512, 1) k_ldtm_bw(int iters, int batch, long long *clk_out)
{
    __shared__ uint32_t slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                         (uint32_t)__cvta_generic_to_shared(&slot)),
                     "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t base = slot + ((uint32_t)((warp & 3) * 32) << 16);
    uint32_t acc = 0;
    __syncthreads();
    long long t0 = clock64();
    for (int i = 0; i < iters; i++) {
        uint32_t v[32];
        const uint32_t a = base + (uint32_t)(((i + (warp >> 2)) & 15) * 32);
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
            : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
              "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
              "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
              "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
            : "r"(a)
            : "memory");
        if ((i % batch) == batch - 1) {
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            acc ^= v[0] ^ v[31];
        }
    }
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    long long t1 = clock64();
    if (lane == 0) clk_out[blockIdx.x * 16 + warp] = (t1 - t0) + (acc == 0x12345u ? 1 : 0);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(slot), "r"(512u) : "memory");
}

// ---- ALU-pipe issue-rate microbenchmark ("alu" mode) -------------------------------------------
// 8 independent chains per thread so that latency never limits; OP selects the instruction.
// One dependent chain per thread: clocks per instruction = the instruction's dependent-issue latency.
template <int OP>
__global__ void __launch_bounds__(32, 1) k_alu_latency(int iters, const float *in, float *out, long long *clk_out)
{
    float f = in[threadIdx.x];
    int v = __float_as_int(f);
    const float x = in[5], y = in[6];
    const int xi = __float_as_int(x), yi = __float_as_int(y);
    long long t0 = clock64();
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int r = 0; r < 64; r++) {
            if (OP == 0) f = fmaxf(f, fmaxf(fabsf(x), fabsf(y)));
            else if (OP == 1) f = fmaxf(f, fabsf(x));
            else if (OP == 2) v = max(v, max(xi, yi));
            else if (OP == 3) f = f + x;
            else v = max(v, xi);
            asm volatile("" : "+f"(f), "+r"(v));
        }
    }
    long long t1 = clock64();
    out[threadIdx.x] = f + (float)v;
    if (threadIdx.x == 0) clk_out[0] = t1 - t0;
}

template <int OP>
__global__ void __launch_bounds__(512, 1) k_alu_rate(int iters, const float *in, float *out, long long *clk_out)
{
    float f[8];
    int v[8];
#pragma unroll
    for (int i = 0; i < 8; i++) { f[i] = in[threadIdx.x + 32 * i]; v[i] = __float_as_int(f[i]); }
    const float x = in[5], y = in[6];
    const int xi = __float_as_int(x), yi = __float_as_int(y);
    __syncthreads();
    long long t0 = clock64();
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int r = 0; r < 8; r++) {
#pragma unroll
            for (int i = 0; i < 8; i++) {
                if (OP == 0) f[i] = fmaxf(f[i], fmaxf(fabsf(x), fabsf(y)));        // FMNMX3 |a|,|b|,c
                else if (OP == 1) f[i] = fmaxf(f[i], fabsf(x));                        // FMNMX
                else if (OP == 2) v[i] = max(v[i], max(xi, yi));                       // VIMNMX3
                else if (OP == 3) f[i] = f[i] + x;                                     // FADD (FMA pipe)
                else v[i] = max(v[i], xi);                                             // VIMNMX (2-input)
            }
            // keep the compiler from collapsing the chains
            asm volatile("" : "+f"(f[0]), "+f"(f[1]), "+f"(f[2]), "+f"(f[3]), "+f"(f[4]), "+f"(f[5]), "+f"(f[6]), "+f"(f[7]));
            asm volatile("" : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]));
        }
    }
    long long t1 = clock64();
    float acc = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) acc += f[i] + (float)v[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = acc;
    if ((threadIdx.x & 31) == 0) clk_out[blockIdx.x * 16 + (threadIdx.x >> 5)] = t1 - t0;
}

static int run_alu()
{
    float *in, *out;
    long long *d;
    cudaMalloc(&in, 4096 * 4);
    cudaMalloc(&out, 148 * 512 * 4);
    cudaMalloc(&d, 148 * 16 * 8);
    std::vector<float> h(4096);
    for (int i = 0; i < 4096; i++) h[i] = (float)(i % 97) - 40.0f;
    cudaMemcpy(in, h.data(), 4096 * 4, cudaMemcpyHostToDevice);
    const int iters = 2000;
    const char *names[5] = {"FMNMX3 |a|,|b|,c", "FMNMX |a|,b", "VIMNMX3", "FADD", "VIMNMX"};
    for (int op = 0; op < 5; op++) {
        if (op == 0) k_alu_latency<0><<<1, 32>>>(iters, in, out, d);
        else if (op == 1) k_alu_latency<1><<<1, 32>>>(iters, in, out, d);
        else if (op == 2) k_alu_latency<2><<<1, 32>>>(iters, in, out, d);
        else if (op == 3) k_alu_latency<3><<<1, 32>>>(iters, in, out, d);
        else k_alu_latency<4><<<1, 32>>>(iters, in, out, d);
        if (cudaDeviceSynchronize() != cudaSuccess) { printf("alu latency kernel failed\n"); return 3; }
        long long lc = 0;
        cudaMemcpy(&lc, d, 8, cudaMemcpyDeviceToHost);
        printf("alu: %-18s dependent chain: %.2f clk per instruction\n", names[op], (double)lc / ((double)iters * 64.0));
        for (int nw = 1; nw <= 4; nw *= 2) {
            if (op == 0) k_alu_rate<0><<<8, nw * 128>>>(iters, in, out, d);
            else if (op == 1) k_alu_rate<1><<<8, nw * 128>>>(iters, in, out, d);
            else if (op == 2) k_alu_rate<2><<<8, nw * 128>>>(iters, in, out, d);
            else if (op == 3) k_alu_rate<3><<<8, nw * 128>>>(iters, in, out, d);
            else k_alu_rate<4><<<8, nw * 128>>>(iters, in, out, d);
            if (cudaDeviceSynchronize() != cudaSuccess) { printf("alu kernel failed\n"); return 3; }
            long long hc[16];
            cudaMemcpy(hc, d, sizeof hc, cudaMemcpyDeviceToHost);
            long long mx = 0;
            for (int w = 0; w < nw * 4; w++) mx = hc[w] > mx ? hc[w] : mx;
            printf("alu: %-18s %d warp(s)/sub-partition: %.2f clk per warp-instruction per sub-partition\n", names[op], nw,
                   (double)mx / ((double)iters * 64.0 * nw));
        }
    }
    return 0;
}

// ---- does a tcgen05.ld in flight block the sub-partition's issue port? ("mix" mode) --------------
// Per sub-partition: `nl` warps loop over tcgen05.ld.x32 (+ wait), `na` warps loop over independent FMNMX3.
__global__ void __launch_bounds__(1024, 1) k_mix(int iters, int nl, int na, const float *in, float *out, long long *clk_out)
{
    __shared__ uint32_t slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                         (uint32_t)__cvta_generic_to_shared(&slot)),
                     "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int idx = warp >> 2;  // index of the warp within its sub-partition
    const uint32_t base = slot + ((uint32_t)((warp & 3) * 32) << 16);
    float f[8];
#pragma unroll
    for (int i = 0; i < 8; i++) f[i] = in[threadIdx.x % 64 + 32 * i];
    const float x = in[5], y = in[6];
    uint32_t acc = 0;
    __syncthreads();
    long long t0 = clock64();
    if (idx < nl) {
        for (int i = 0; i < iters; i++) {
            uint32_t v[32];
            const uint32_t a = base + (uint32_t)(((i + idx) & 15) * 32);
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                  "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                  "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                  "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                : "r"(a)
                : "memory");
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            acc ^= v[0] ^ v[31];
        }
    } else if (idx < nl + na) {
        for (int it = 0; it < iters; it++) {
#pragma unroll
            for (int r = 0; r < 4; r++) {
#pragma unroll
                for (int i = 0; i < 8; i++) f[i] = fmaxf(f[i], fmaxf(fabsf(x), fabsf(y)));
                asm volatile("" : "+f"(f[0]), "+f"(f[1]), "+f"(f[2]), "+f"(f[3]), "+f"(f[4]), "+f"(f[5]), "+f"(f[6]), "+f"(f[7]));
            }
        }
    }
    long long t1 = clock64();
    float s = (float)acc;
#pragma unroll
    for (int i = 0; i < 8; i++) s += f[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
    if (lane == 0) clk_out[blockIdx.x * 32 + warp] = t1 - t0;
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(slot), "r"(512u) : "memory");
}

static int run_mix()
{
    float *in, *out;
    long long *d;
    cudaMalloc(&in, 4096 * 4);
    cudaMalloc(&out, 8 * 1024 * 4);
    cudaMalloc(&d, 8 * 32 * 8);
    std::vector<float> h(4096);
    for (int i = 0; i < 4096; i++) h[i] = (float)(i % 97) - 40.0f;
    cudaMemcpy(in, h.data(), 4096 * 4, cudaMemcpyHostToDevice);
    const int iters = 20000;
    const int cfg[6][2] = {{2, 0}, {0, 2}, {2, 2}, {4, 0}, {0, 4}, {4, 4}};
    for (int c = 0; c < 6; c++) {
        const int nl = cfg[c][0], na = cfg[c][1];
        k_mix<<<8, (nl + na) * 128>>>(iters, nl, na, in, out, d);
        if (cudaDeviceSynchronize() != cudaSuccess) { printf("mix kernel failed\n"); return 3; }
        long long hc[32];
        cudaMemcpy(hc, d, sizeof hc, cudaMemcpyDeviceToHost);
        long long ml = 0, ma = 0;
        for (int w = 0; w < (nl + na) * 4; w++) {
            if ((w >> 2) < nl) ml = hc[w] > ml ? hc[w] : ml;
            else ma = hc[w] > ma ? hc[w] : ma;
        }
        printf("mix: %d load warp(s) + %d FMNMX3 warp(s) per sub-partition:", nl, na);
        if (nl) printf("  %.1f clk per 4 KB tcgen05.ld per sub-partition", (double)ml / iters / nl);
        if (na) printf("  %.2f clk per FMNMX3 per sub-partition", (double)ma / ((double)iters * 32.0 * na));
        printf("\n");
    }
    return 0;
}


// ---- accumulator hand-over round trip ("chain" mode) ----------------------------------------------
// One MMA-issuer warp and four "epilogue" warps (one per TMEM lane quarter) play the search kernel's accumulator
// protocol with nothing else in the way: issuer waits empty[q], issues ks tcgen05.mma (M = N = 128, K = 16,
// kind::f16), commits -> full[q]; each epilogue warp waits full[q], does nload tcgen05.ld.x32 (+ wait), arrives on
// empty[q].  nacc accumulators are used round-robin.  Reports clocks per round: with nacc = 1 that is
// ks * 64 (the MMAs) + the synchronisation latency of the whole hand-over.
namespace chain {
__device__ __forceinline__ uint32_t s32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mb_init(uint32_t b, uint32_t c) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(b), "r"(c)); }
__device__ __forceinline__ void mb_arrive(uint32_t b) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(b) : "memory"); }
__device__ __forceinline__ uint32_t mb_try(uint32_t b, uint32_t par)
{
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(b), "r"(par) : "memory");
    return ok;
}
__device__ __forceinline__ uint32_t mb_test(uint32_t b, uint32_t par)
{
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(b), "r"(par) : "memory");
    return ok;
}
__device__ __forceinline__ void mb_wait(uint32_t b, uint32_t par, int spin)
{
    if (spin) { while (!mb_test(b, par)) {} }
    else { while (!mb_try(b, par)) {} }
}
__device__ __forceinline__ uint64_t desc(uint32_t saddr, uint32_t lbo, uint32_t sbo)
{
    return (uint64_t)((saddr >> 4) & 0x3fff) | ((uint64_t)((lbo >> 4) & 0x3fff) << 16) | ((uint64_t)((sbo >> 4) & 0x3fff) << 32) | ((uint64_t)1 << 46);
}
}  // namespace chain

__global__ void __launch_bounds__(192, 1) k_chain(int iters, int ks, int nload, int nacc, int flags, long long *clk_out)
{
    using namespace chain;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t *sA = smem, *sB = smem + 16384;              // 4 K-slices each: 128 rows x 64 binary16
    uint64_t *bars = (uint64_t *)(smem + 32768);
    uint32_t *slot = (uint32_t *)(bars + 16);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < 32768 / 4; i += blockDim.x) {
        uint32_t x = (uint32_t)i * 2654435761u + 12345u;
        x ^= x >> 15; x *= 0x2c1b3c6du; x ^= x >> 12;
        ((uint32_t *)smem)[i] = x & 0x3fff3fffu;
    }
    const uint32_t bar0 = s32(bars);
    if (threadIdx.x == 0) {
        for (int q = 0; q < 4; q++) { mb_init(bar0 + 8 * q, 1); mb_init(bar0 + 32 + 8 * q, 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *slot;
    const int spin_epi = flags & 1, spin_iss = flags & 2;
    const int freerun = flags & 4;   // issuer never waits for the hand-back: pure MMA + commit throughput
    const int selfwait = flags & 8;  // issuer waits for its own commit (full[q]) each round: commit -> visible latency
    if (warp == 1) {
        const uint64_t ad = desc(s32(sA), 128, 1024), bd = desc(s32(sB), 128, 1024);
        constexpr uint32_t idesc = (1u << 4) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
        long long t0 = clock64();
        for (int i = 0; i < iters; i++) {
            const int q = i % nacc;
            if (!freerun && !selfwait) mb_wait(bar0 + 32 + 8 * q, ((i / nacc) & 1) ^ 1, spin_iss);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (lane == 0) {
                for (int s = 0; s < ks; s++) {
                    const uint32_t acc = s > 0;
                    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem + q * 128),
                                 "l"(ad + (uint64_t)((s & 3) * 16)), "l"(bd + (uint64_t)((s & 3) * 16)), "r"(idesc), "r"(acc)
                                 : "memory");
                }
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar0 + 8 * q) : "memory");
            }
            __syncwarp();
            if (selfwait) mb_wait(bar0 + 8 * q, (i / nacc) & 1, spin_iss);
        }
        // drain: wait until the last round of every accumulator came back (free-running: until the last commit fired)
        if (freerun || selfwait) {
            const int q = (iters - 1) % nacc;
            mb_wait(bar0 + 8 * q, ((iters - 1) / nacc) & 1, 0);
        } else {
            for (int q = 0; q < nacc; q++) {
                const int rounds = (iters - q + nacc - 1) / nacc;  // rounds accumulator q went through
                mb_wait(bar0 + 32 + 8 * q, (rounds & 1) ^ 1, 0);
            }
        }
        long long t1 = clock64();
        if (lane == 0) clk_out[blockIdx.x] = t1 - t0;
    } else if (warp >= 2 && !freerun && !selfwait) {
        const uint32_t ta = tmem + ((uint32_t)((warp & 3) * 32) << 16);
        uint32_t sink = 0;
        for (int i = 0; i < iters; i++) {
            const int q = i % nacc;
            mb_wait(bar0 + 8 * q, (i / nacc) & 1, spin_epi);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            for (int c = 0; c < nload; c++) {
                uint32_t v[32];
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                    "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                    "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                    : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                      "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                      "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                      "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                    : "r"(ta + q * 128 + c * 32)
                    : "memory");
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                sink ^= v[0] ^ v[31];
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mb_arrive(bar0 + 32 + 8 * q);
        }
        if (sink == 0x12345u) clk_out[1000] = 1;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
}

static int run_chain()
{
    long long *d;
    if (cudaMalloc(&d, 2048 * 8) != cudaSuccess) return 3;
    const int smem = 40 * 1024;
    cudaFuncSetAttribute(k_chain, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    const int iters = 20000;
    struct Cfg { int ks, nload, nacc, flags; };
    const Cfg cfgs[] = {{1, 0, 1, 0}, {4, 0, 1, 0}, {1, 0, 1, 1}, {1, 0, 1, 2}, {1, 0, 1, 3}, {1, 1, 1, 0}, {1, 4, 1, 0}, {4, 4, 1, 0},
                        {4, 0, 4, 0}, {4, 1, 4, 0}, {4, 2, 4, 0}, {4, 3, 4, 0}, {4, 4, 4, 0}, {4, 4, 4, 1}, {4, 4, 4, 3}, {4, 0, 2, 0}, {4, 2, 2, 0},
                        {2, 0, 4, 0}, {2, 2, 4, 0}, {2, 4, 4, 0}, {1, 0, 4, 0}, {1, 4, 4, 0},
                        {1, 0, 4, 4}, {4, 0, 4, 4}, {1, 0, 1, 8}, {4, 0, 1, 8}, {1, 0, 1, 10}, {4, 0, 4, 8}};
    for (const Cfg &c : cfgs) {
        for (int grid : {1, 148}) {
            cudaMemset(d, 0, 2048 * 8);
            k_chain<<<grid, 192, smem>>>(iters, c.ks, c.nload, c.nacc, c.flags, d);
            if (cudaDeviceSynchronize() != cudaSuccess) { printf("chain kernel failed: %s\n", cudaGetErrorString(cudaGetLastError())); return 3; }
            long long h[148];
            cudaMemcpy(h, d, sizeof h, cudaMemcpyDeviceToHost);
            long long mx = 0;
            for (int b = 0; b < grid; b++) mx = h[b] > mx ? h[b] : mx;
            printf("chain: ks=%d nload=%d nacc=%d spin(epi=%d,iss=%d)%s%s grid=%3d: %.1f clk per round (MMA alone %d)\n", c.ks, c.nload, c.nacc,
                   c.flags & 1, (c.flags >> 1) & 1, (c.flags & 4) ? " free-running" : "", (c.flags & 8) ? " issuer waits its own commit" : "",
                   grid, (double)mx / iters, c.ks * 64);
        }
    }
    return 0;
}

// ---- in-tree radix sort against std::stable_sort ("sort" mode) ----------------------------------
#include <algorithm>
static int run_sort()
{
    cudaStream_t s;
    cudaStreamCreate(&s);
    int rc = 0;
    const long long sizes[] = {1, 31, 2048, 2049, 100000, 1042441, 4182025, 16752649};
    for (long long n : sizes)
        for (int mode = 0; mode < 3; mode++) {
            std::vector<uint32_t> k(n);
            std::vector<int32_t> v(n);
            uint32_t x = 12345u + (uint32_t)n + mode;
            for (long long i = 0; i < n; i++) {
                x = lowbias32(x + (uint32_t)i);
                k[i] = mode == 0 ? (x & 0xffffffu) : (mode == 1 ? (x & 0xffu) * 65793u % 16777216u : (uint32_t)(i % 7 == 0 ? 0 : 5));  // wide / few values / ties
                v[i] = (int32_t)i;
            }
            uint32_t *dk, *dko;
            int32_t *dv, *dvo;
            cudaMalloc(&dk, n * 4 + 16); cudaMalloc(&dko, n * 4 + 16); cudaMalloc(&dv, n * 4 + 16); cudaMalloc(&dvo, n * 4 + 16);
            cudaMemcpy(dk, k.data(), n * 4, cudaMemcpyHostToDevice);
            cudaMemcpy(dv, v.data(), n * 4, cudaMemcpyHostToDevice);
            cudaEvent_t e0, e1;
            cudaEventCreate(&e0); cudaEventCreate(&e1);
            cudaEventRecord(e0, s);
            int e = umma_debug_sort(dk, dv, dko, dvo, n, s);
            cudaEventRecord(e1, s);
            cudaEventSynchronize(e1);
            float ms = 0;
            cudaEventElapsedTime(&ms, e0, e1);
            std::vector<uint32_t> ko(n);
            std::vector<int32_t> vo(n);
            cudaMemcpy(ko.data(), dko, n * 4, cudaMemcpyDeviceToHost);
            cudaMemcpy(vo.data(), dvo, n * 4, cudaMemcpyDeviceToHost);
            std::vector<int32_t> ref(n);
            for (long long i = 0; i < n; i++) ref[i] = (int32_t)i;
            std::stable_sort(ref.begin(), ref.end(), [&](int32_t a, int32_t b) { return k[a] < k[b]; });
            long long bad = 0;
            for (long long i = 0; i < n; i++) bad += (vo[i] != ref[i]) || (ko[i] != k[ref[i]]);
            printf("sort: n=%lld mode=%d rc=%d %.3f ms (incl. scratch allocation): %lld mismatches vs std::stable_sort\n", n, mode, e, ms, bad);
            if (bad || e) rc = 1;
            cudaFree(dk); cudaFree(dko); cudaFree(dv); cudaFree(dvo);
        }
    printf(rc ? "SORT FAIL\n" : "SORT PASS\n");
    return rc;
}

static int run_ldtm()
{
    long long *d;
    if (cudaMalloc(&d, 148 * 16 * 8) != cudaSuccess) return 3;
    const int iters = 20000;
    for (int nw = 1; nw <= 4; nw *= 2)
        for (int batch = 1; batch <= 2; batch++) {
            cudaMemset(d, 0, 148 * 16 * 8);
            k_ldtm_bw<<<8, nw * 128>>>(iters, batch, d);
            if (cudaDeviceSynchronize() != cudaSuccess) { printf("ldtm kernel failed\n"); return 3; }
            long long h[16];
            cudaMemcpy(h, d, sizeof h, cudaMemcpyDeviceToHost);
            long long mx = 0;
            for (int w = 0; w < nw * 4; w++) mx = h[w] > mx ? h[w] : mx;
            const double clk_per_ld = (double)mx / iters / nw;  // per sub-partition: nw warps share it
            printf("ldtm: %d warp(s)/sub-partition, wait every %d load(s): %.1f clk per 4 KB load per sub-partition -> %.1f B/clk/SMSP\n",
                   nw, batch, clk_per_ld, 4096.0 / clk_per_ld);
        }
    return 0;
}

int main(int argc, char **argv)
{
    if (argc > 1 && !strcmp(argv[1], "ldtm")) return run_ldtm();
    if (argc > 1 && !strcmp(argv[1], "alu")) return run_alu();
    if (argc > 1 && !strcmp(argv[1], "mix")) return run_mix();
    if (argc > 1 && !strcmp(argv[1], "chain")) return run_chain();
    if (argc > 1 && !strcmp(argv[1], "sort")) return run_sort();
    if (argc > 1 && !strcmp(argv[1], "peak")) {  // bare MMA loops: rate by kind and shape
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, 0));
        cudaStream_t s;
        CK(cudaStreamCreate(&s));
        for (int f16 = 0; f16 < 2; f16++)
            for (int n = 128; n <= 256; n += 128) {
                const char *err = "";
                double t = measure_mma_peak(prop.multiProcessorCount, s, 3, f16, n, &err);
                printf("peak kind::%s M=128 N=%d: %.1f TOP/s %s\n", f16 ? "f16" : "i8", n, t, t < 0 ? err : "");
            }
        for (int f16 = 0; f16 < 2; f16++) {  // CTA pairs: cta_group::2, M = 256, N = 128
            const char *err = "";
            uint32_t bases[4] = {0xdeadu, 0xdeadu, 0xdeadu, 0xdeadu};
            double t = measure_mma_peak_pair(prop.multiProcessorCount, s, 3, f16, bases, &err);
            printf("peak kind::%s cta_group::2 M=256 N=128: %.1f TOP/s %s  (TMEM bases of CTAs 0-3: %x %x %x %x)\n", f16 ? "f16" : "i8", t,
                   t < 0 ? err : "", bases[0], bases[1], bases[2], bases[3]);
        }
        return 0;
    }
    if (argc < 4 || (strcmp(argv[1], "check") && strcmp(argv[1], "time"))) {
        printf("usage: umma_probe check|time B W [pattern] [kind] [pair]   or   umma_probe peak|ldtm|alu|mix|chain|sort\n");
        return 2;
    }
    bool check = !strcmp(argv[1], "check");
    int B = atoi(argv[2]), W = atoi(argv[3]);
    int pattern = argc > 4 ? atoi(argv[4]) : 0;
    int kind = argc > 5 ? atoi(argv[5]) : 0;
    int pair = argc > 6 ? atoi(argv[6]) : FIC_UMMA_PAIR_AUTO;
    int H = W;
    Geom g;
    const char *why = "";
    int wk = 2 * (W / B) - 3;
    if (make_geom(W, H, B, wk, 0, &g, &why)) { printf("bad geometry: %s\n", why); return 2; }
    if (!umma_applicable(g)) { printf("umma not applicable\n"); return 2; }
    printf("probe mode=%s B=%d W=%d pattern=%d kind=%d pair=%d NR=%lld ND=%lld\n", argv[1], B, W, pattern, kind, pair,
           (long long)g.NR, (long long)g.ND);

    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    printf("device: %s sm_%d%d, %d SMs\n", prop.name, prop.major, prop.minor, prop.multiProcessorCount);
    int *status_h = nullptr, *status_d = nullptr;
    CK(cudaHostAlloc((void **)&status_h, 64, cudaHostAllocMapped));
    *status_h = 0;
    CK(cudaHostGetDevicePointer((void **)&status_d, status_h, 0));
    g_status = status_h;

    std::vector<uint8_t> img;
    make_image(img, W, H, pattern, 1);
    Work w;
    CK(cudaMalloc(&w.src, (size_t)W * H));
    CK(cudaMalloc(&w.dec, (size_t)g.sw * g.sh));
    CK(cudaMalloc(&w.dsum, 4 * g.ND));
    CK(cudaMalloc(&w.dsq, 4 * g.ND));
    CK(cudaMalloc(&w.rsum, 4 * g.NR));
    CK(cudaMalloc(&w.best, 4 * g.NR));
    CK(cudaMalloc(&w.opA, umma_opA_bytes(g, 0, g.NR, prop.multiProcessorCount, kind)));
    CK(cudaMalloc(&w.opB, umma_opB_bytes(g, kind)));
    CK(cudaMemcpy(w.src, img.data(), (size_t)W * H, cudaMemcpyHostToDevice));
    cudaStream_t s;
    CK(cudaStreamCreate(&s));
    launch_decimate(w.src, w.dec, g, s);
    launch_domain_stats(w.dec, w.dsum, w.dsq, g, s);
    launch_range_stats(w.src, w.rsum, g, s);
    CK(cudaStreamSynchronize(s));

    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    float ms_direct = 0, ms_umma = 0;

    // reference winners: direct CUDA-core search
    std::vector<int32_t> best_direct(g.NR), best_umma(g.NR);
    CK(cudaEventRecord(e0, s));
    launch_search_direct(w, g, 0, g.NR, s);
    CK(cudaEventRecord(e1, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaEventElapsedTime(&ms_direct, e0, e1));
    CK(cudaMemcpy(best_direct.data(), w.best, 4 * g.NR, cudaMemcpyDeviceToHost));
    CK(cudaMemset(w.best, 0xff, 4 * g.NR));

    int ntiles = (int)((g.ND + 127) / 128);
    int64_t dump_ld = (int64_t)ntiles * 128;
    int64_t rp = (g.NR + 1023) / 1024 * 1024;  // make_plan pads the rows to an even number of super-blocks
    int32_t *dump = nullptr;
    if (check) {
        CK(cudaMalloc(&dump, (size_t)rp * dump_ld * 4));
        CK(cudaMemset(dump, 0x7f, (size_t)rp * dump_ld * 4));
    }
    const char *err = "";
    int reps = check ? 1 : 3;
    for (int r = 0; r < reps; r++) {
        CK(cudaEventRecord(e0, s));
        cudaEvent_t k0, k1;
        CK(cudaEventCreate(&k0));
        CK(cudaEventCreate(&k1));
        int pair_used = 0;
        int n = launch_search_umma(w, g, 0, g.NR, prop.multiProcessorCount, s, &err, kind, k0, k1, pair, &pair_used, dump, dump_ld,
                                   status_d);
        if (n < 0) { printf("launch failed: %s\n", err); return 3; }
        CK(cudaEventRecord(e1, s));
        CK(cudaStreamSynchronize(s));
        CK(cudaEventElapsedTime(&ms_umma, e0, e1));
        float ms_k = 0;
        CK(cudaEventElapsedTime(&ms_k, k0, k1));
        printf("umma search run %d: pack+search+merge %.3f ms, k_umma_search alone %.3f ms   pairs=%d status=%d\n", r, ms_umma, ms_k,
               pair_used, *status_h);
    }
    CK(cudaMemcpy(best_umma.data(), w.best, 4 * g.NR, cudaMemcpyDeviceToHost));
    double evals = (double)g.NR * (double)g.ND;
    printf("direct search: %.3f ms (%.3e evals/s)   umma: %.3f ms (%.3e evals/s, %.1f%% of 4.5 POPS int8 / %.1f%% of 2.25 PFLOPS f16 at 2*B*B ops/eval)\n",
           ms_direct, evals / (ms_direct * 1e-3), ms_umma, evals / (ms_umma * 1e-3),
           100.0 * evals * 2 * g.n / (ms_umma * 1e-3) / 4.5e15, 100.0 * evals * 2 * g.n / (ms_umma * 1e-3) / 2.25e15);

    int rc = 0;
    if (check) {
        std::vector<int32_t> hd((size_t)rp * dump_ld);
        CK(cudaMemcpy(hd.data(), dump, hd.size() * 4, cudaMemcpyDeviceToHost));
        std::vector<uint8_t> dec((size_t)g.sw * g.sh);
        CK(cudaMemcpy(dec.data(), w.dec, dec.size(), cudaMemcpyDeviceToHost));
        long long bad = 0, shown = 0;
        const int32_t *d_pos_dom;
        int64_t npos;
        umma_debug_positions(w, g, g.NR, prop.multiProcessorCount, kind, &d_pos_dom, &npos);
        std::vector<int32_t> pos_dom(npos);
        CK(cudaMemcpy(pos_dom.data(), d_pos_dom, npos * 4, cudaMemcpyDeviceToHost));
        std::vector<int64_t> pos_of(g.ND, -1);
        for (int64_t p = 0; p < npos; p++)
            if (pos_dom[p] >= 0) pos_of[pos_dom[p]] = p;
        for (int64_t j = 0; j < g.ND; j++)
            if (pos_of[j] < 0) { printf("sweep order is not a permutation (domain %lld missing)\n", (long long)j); return 1; }
        for (int64_t i = 0; i < g.NR; i++) {
            int xr = (int)(i % g.rpw), yr = (int)(i / g.rpw);
            int rs = 0;
            int r[256];
            for (int k = 0; k < g.n; k++) {
                r[k] = img[(size_t)(yr * B + k / B) * W + xr * B + k % B];
                rs += r[k];
            }
            int rmean = rs / g.n;
            for (int64_t j = 0; j < g.ND; j++) {
                int gx = (int)(j % g.dpw), gy = (int)(j / g.dpw);
                int ds = 0, d[256];
                for (int k = 0; k < g.n; k++) {
                    d[k] = dec[(size_t)(gy * g.step + k / B) * g.sw + gx * g.step + k % B];
                    ds += d[k];
                }
                int dmean = ds / g.n;
                int kov = 0;
                for (int k = 0; k < g.n; k++) kov += (r[k] - rmean) * (d[k] - dmean);
                if ((B == 16 || kind == 1) && dmean == 0) kov = -kov;  // kind::i8 stores the rows of mean-0 blocks negated (only |kov| is used)
                int got = hd[(size_t)i * dump_ld + pos_of[j]];
                if (got != kov) {
                    bad++;
                    if (shown < 12) {
                        printf("  kov mismatch row %lld dom %lld: got %d want %d\n", (long long)i, (long long)j, got, kov);
                        shown++;
                    }
                }
            }
        }
        printf("accumulator check: %lld mismatches of %lld\n", bad, (long long)(g.NR * g.ND));
        if (bad) rc = 1;
    }
    long long diff = 0, shown = 0;
    for (int64_t i = 0; i < g.NR; i++)
        if (best_direct[i] != best_umma[i]) {
            diff++;
            if (shown++ < 12) printf("  winner mismatch row %lld: direct %d umma %d\n", (long long)i, best_direct[i], best_umma[i]);
        }
    printf("winner check: %lld of %lld rows differ\n", diff, (long long)g.NR);
    if (diff) rc = 1;
    printf(rc ? "PROBE FAIL\n" : "PROBE PASS\n");
    return rc;
}
