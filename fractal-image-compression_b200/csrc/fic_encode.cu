// fic_encode.cu -- the encoder's host side: which engine and tcgen05 instruction kind a call runs (and how many images a
// batch group holds), one run of that plan on device-resident pixels, and the stage times of the last run.  The kernels
// live in fic_kernels.cu and fic_search_umma.cu; the entries, the handle and the copies in fic_api.cu.
#include "fic_internal.h"

namespace fic {

// The stage events of a run, each recorded where its stage starts (kDone: after the solve).  The fused engine records
// kPool and kDone only; the tcgen05 launcher records kKernel0 / kKernel1 around its search kernel.
enum { kPool, kSearch, kSolve, kDone, kKernel0, kKernel1 };

#define ECU(call) \
    do { const cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(FIC_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)

#define ENSURE(ptr, slot, bytes) \
    do { const Status st_ = ensure(w, ptr, slot, (size_t)(bytes)); if (st_.rc) return st_; } while (0)

// Input pixels one group of a batch uploads at most: the grow-only workspace does not grow with the batch.
constexpr size_t kBatchGroupBytes = (size_t)64 << 20;
// A group on the tcgen05 engine also holds at most 256 images (the image index is the top digit of the pool sort's
// keys) and at most this much operand workspace (opA + opB: packed operands, flag lists, position tables and sort
// scratch, about 2-6 MB per image of 256^2 - 512^2 at blockgroesse 8) -- or one image, however large.
constexpr int kBatchUmmaImages = 256;
constexpr size_t kBatchUmmaBytes = (size_t)1 << 30;
// AUTO on a batch of full-pool images that a single call would give to the CUDA-core search picks the tcgen05 group
// search for groups of at least this many images.  Measured on a B200 (tools/batch_bench.py,
// profiles/r4_batch_fullpool.json): the tensor chain costs 160-190 us per call at 128^2-256^2 plus 5-10 us per image,
// the direct search 70-130 us per image, so the group pays from about three images on (n = 8: 2.5-4x faster per image).
// Where the single call runs the fused one-launch kernel (full pools of at most 16 x 16 domains, e.g. 64^2 at B = 8)
// that kernel stays faster at every batch size (0.6 against 1.0 us per image at n = 256), so AUTO keeps it.
constexpr int kBatchUmmaMinImages = 4;

Status f16_selftest(Encoder &e, cudaStream_t s)
{
    if (e.f16_state == 0) {
        const char *why = nullptr;
        const int ok = umma_f16_selftest(e.num_sms, s, &why);
        if (ok < 0) return fail(FIC_E_CUDA, "kind::f16 self-test failed to run: %s", why ? why : "?");
        e.f16_state = ok ? 1 : -1;
    }
    return Status();
}

Status plan_encode(Encoder &e, const Geom &g, int64_t j0, int64_t j1, int n_images, bool argb, cudaStream_t s,
                   EncodePlan *plan)
{
    // The engine of one image (FIC_OPT_ENGINE): the tcgen05 search for whole-pool windows with enough work to fill the
    // GPU, else the fused one-launch encode for the reference's GUI windows (widthKernel <= 16), else the multi-kernel
    // direct path.
    int engine = FIC_ENGINE_DIRECT;
    if (e.engine_opt == FIC_ENGINE_UMMA) {
        if (!umma_applicable(g))
            return fail(FIC_E_ARG, "tcgen05 search needs widthKernel == domain blocks per width == per height (and no isometries for RGB)");
        engine = FIC_ENGINE_UMMA;
    } else if (e.engine_opt == FIC_ENGINE_FUSED) {
        if (!fused_encode_applicable(g)) return fail(FIC_E_ARG, "the fused encode needs widthKernel <= 16 and no isometries");
        engine = FIC_ENGINE_FUSED;
    } else if (e.engine_opt == FIC_ENGINE_AUTO) {
        // the fused kernel spends one CTA per range block and wins where launches dominate (<= 16 K range blocks,
        // 1.8 ms against 0.45 ms for the multi-kernel path at 4096^2, widthKernel 2: measured, profiles/README.md)
        if (umma_applicable(g) && (j1 - j0) * g.ND >= (int64_t)1 << 22) engine = FIC_ENGINE_UMMA;
        else if (fused_encode_applicable(g) && g.NR <= 16384) engine = FIC_ENGINE_FUSED;
    }
    const size_t image_bytes = (argb ? sizeof(int32_t) : (size_t)g.C) * g.W * g.H;
    const size_t fit = kBatchGroupBytes / image_bytes;
    int group = fit < (size_t)n_images ? (fit > 0 ? (int)fit : 1) : n_images;
    // AUTO on a batch: the tcgen05 group search instead of the CUDA-core search for groups of enough images
    int want = n_images > 1 && e.engine_opt == FIC_ENGINE_AUTO && engine == FIC_ENGINE_DIRECT && umma_applicable(g) ? FIC_ENGINE_UMMA : engine;
    // The first kind::f16 search of a handle verifies, once, that this device's f16 tensor path accumulates the integer
    // covariances exactly; a device that does not runs kind::i8 instead.  RGB has a kind::f16 tensor path only; without
    // an exact f16 path it stays on the CUDA-core kernel.  (The self-test allocates and synchronises on this stream:
    // one-time cost of the first such call; fic_get_option(FIC_OPT_F16_EXACT) runs it ahead of time.)
    int kind = e.umma_kind;
    const bool rgb = g.C == 3;
    if (want == FIC_ENGINE_UMMA && (rgb || (g.B != 16 && (kind == FIC_UMMA_KIND_F16 || (kind == FIC_UMMA_KIND_AUTO && umma_default_kind(g) == FIC_UMMA_KIND_F16))))) {
        const Status st = f16_selftest(e, s);
        if (st.rc) return st;
        if (e.f16_state < 0) {
            if (rgb) want = FIC_ENGINE_DIRECT;
            else kind = FIC_UMMA_KIND_I8;
        }
    }
    if (want == FIC_ENGINE_UMMA) {
        // images per tcgen05 group (kBatchUmmaImages, kBatchUmmaBytes)
        int n = group < kBatchUmmaImages ? group : kBatchUmmaImages;
        auto bytes = [&](int k) { return umma_opA_bytes(g, 0, g.NR, e.num_sms, kind, k) + umma_opB_bytes(g, kind, k); };
        for (size_t b; n > 1 && (b = bytes(n)) > kBatchUmmaBytes;) n = (int)((double)n * kBatchUmmaBytes / b);
        if (n < 1) n = 1;
        if (engine == FIC_ENGINE_UMMA || n >= kBatchUmmaMinImages) {
            engine = FIC_ENGINE_UMMA;
            group = n;
        }
    } else if (engine == FIC_ENGINE_UMMA) {
        engine = want;  // RGB on a device without an exact kind::f16 path: the CUDA-core search, image by image
    }
    *plan = EncodePlan{engine, kind, group};
    return Status();
}

Status run_encode(Encoder &e, Work &w, const Geom &g, const EncodePlan &p, const void *d_pixels, bool argb, int64_t j0,
                  int64_t j1, int n_images, float *d_info, int32_t *d_q, fic_timings *tm, cudaStream_t s)
{
    int launches = 0;
    if (p.engine == FIC_ENGINE_FUSED) {  // one kernel straight from the pixels, between kPool and kDone
        ECU(cudaEventRecord(e.ev[kPool], s));
        launches += launch_encode_fused(d_pixels, argb, g, j0, j1, d_info, d_q, s, n_images);
        ECU(cudaEventRecord(e.ev[kDone], s));
    } else {
        const size_t n = (size_t)n_images;
        const uint8_t *d_src = (const uint8_t *)d_pixels;
        if (argb) {  // planes for the pool builders; the unpack runs before kPool, so it counts as upload
            ENSURE(w.src, S_SRC, (size_t)g.C * g.W * g.H * n);
            launches += launch_unpack((const int32_t *)d_pixels, w.src, g.W, g.H, g.C, s, n_images);
            d_src = w.src;
        }
        ENSURE(w.dec, S_DEC, (size_t)g.C * g.sw * g.sh * n);
        ENSURE(w.dsum, S_DSUM, sizeof(int32_t) * g.C * g.ND * n);
        ENSURE(w.dsq, S_DSQ, sizeof(int32_t) * g.C * g.ND * n);
        ENSURE(w.rsum, S_RSUM, sizeof(int32_t) * g.C * g.NR * n);
        ENSURE(w.best, S_BEST, sizeof(int32_t) * g.NR * n);
        if (g.C == 3) ENSURE(w.dec3, S_DEC3, sizeof(uint16_t) * (size_t)g.sw * g.sh * n);  // R + G + B of the decimated planes
        e.pair_used = 0;
        if (p.engine == FIC_ENGINE_UMMA) {
            ENSURE(w.opA, S_OPA, umma_opA_bytes(g, j0, j1, e.num_sms, p.kind, n_images));
            ENSURE(w.opB, S_OPB, umma_opB_bytes(g, p.kind, n_images));
        }
        Work call = w;  // per-call view: the source planes may belong to the caller
        call.src = const_cast<uint8_t *>(d_src);
        ECU(cudaEventRecord(e.ev[kPool], s));
        launches += launch_decimate(d_src, w.dec, g, s, n_images);
        launches += launch_domain_stats(w.dec, w.dsum, w.dsq, g, s, n_images);
        launches += launch_range_stats(d_src, w.rsum, g, s, n_images);
        ECU(cudaEventRecord(e.ev[kSearch], s));
        ECU(cudaEventRecord(e.ev[kKernel0], s));  // (the tcgen05 launcher re-records both around its search kernel)
        ECU(cudaEventRecord(e.ev[kKernel1], s));
        if (p.engine == FIC_ENGINE_UMMA) {
            const char *why = nullptr;
            const int nl = launch_search_umma(call, g, j0, j1, e.num_sms, s, &why, p.kind, e.ev[kKernel0], e.ev[kKernel1],
                                              e.umma_pair, &e.pair_used, nullptr, 0, nullptr, n_images);
            if (nl < 0) return fail(FIC_E_CUDA, "tcgen05 search launch failed: %s", why ? why : "?");
            launches += nl;
        } else {
            if (g.C == 3) launches += launch_sum_planes(w.dec, w.dec3, g, s);
            ECU(cudaEventRecord(e.ev[kKernel0], s));
            launches += launch_search_direct(call, g, j0, j1, s);
            ECU(cudaEventRecord(e.ev[kKernel1], s));
        }
        ECU(cudaEventRecord(e.ev[kSolve], s));
        launches += launch_solve(call, g, j0, j0 + (j1 - j0) * n_images, d_info, d_q, s);  // a group: the flat range [0, n * NR)
        ECU(cudaEventRecord(e.ev[kDone], s));
    }
    ECU(cudaGetLastError());
    e.run_engine = p.engine;
    tm->engine = p.engine;
    tm->launches += launches;
    tm->search_evals += (double)(j1 - j0) * (double)g.wk * (double)g.wk * (double)g.n_iso * (double)n_images;
    return Status();
}

bool run_done(const Encoder &e) { return cudaEventQuery(e.ev[kDone]) == cudaSuccess; }

void read_stages(const Encoder &e, fic_timings *acc, cudaEvent_t begin, cudaEvent_t end)
{
    float ms = 0;
    auto span = [&](cudaEvent_t a, cudaEvent_t b) { return cudaEventElapsedTime(&ms, a, b) == cudaSuccess; };
    if (e.run_engine == FIC_ENGINE_FUSED) {  // a single kernel between kPool and kDone
        if (span(e.ev[kPool], e.ev[kDone])) {
            acc->search_ms += ms;
            acc->kernel_ms += ms;
        }
    } else {
        if (span(e.ev[kPool], e.ev[kSearch])) acc->pool_ms += ms;
        if (span(e.ev[kSearch], e.ev[kSolve])) acc->search_ms += ms;
        if (span(e.ev[kKernel0], e.ev[kKernel1])) acc->kernel_ms += ms;
        if (span(e.ev[kSolve], e.ev[kDone])) acc->solve_ms += ms;
    }
    if (begin && span(begin, e.ev[kPool])) acc->h2d_ms = ms;
    if (end && span(e.ev[kDone], end)) acc->d2h_ms = ms;
    if (span(begin ? begin : e.ev[kPool], end ? end : e.ev[kDone])) acc->total_ms = ms;
}

}  // namespace fic
