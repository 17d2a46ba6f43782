// fic_api.cu -- the C ABI of libfic_b200.so (see include/fic_b200.h): handle, workspace,
// call sequencing on one CUDA stream, timings, and the .run stream helpers.
#include <math.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>

#include "fic_device.cuh"

using namespace fic;

// ------------------------------------------------------------------------------------
// geometry / argument checking
// ------------------------------------------------------------------------------------
int fic::make_geom(int W, int H, int B, int wk, int mode, Geom *g, const char **why)
{
    const char *dummy;
    if (!why) why = &dummy;
    if (mode < FIC_MODE_GREY || mode > FIC_MODE_GREY_ISO) { *why = "mode must be FIC_MODE_GREY, FIC_MODE_RGB or FIC_MODE_GREY_ISO"; return FIC_E_ARG; }
    // FC:1019 `abstand = blockgroesse / 4` is 0 for B < 4 (ArithmeticException); the
    // reference GUI offers 4, 8, 16 (RLEAppView.fxml:55).  Larger blocks leave the range
    // in which the reference's float covariance is an exact integer, so they are refused.
    if (!(B == 4 || B == 8 || B == 16)) { *why = "blockgroesse must be 4, 8 or 16"; return FIC_E_ARG; }
    if (W <= 0 || H <= 0 || W % B || H % B) { *why = "width and height must be positive multiples of blockgroesse"; return FIC_E_ARG; }
    if (W > 32768 || H > 32768) { *why = "image larger than 32768 pixels on a side"; return FIC_E_ARG; }
    int rpw = W / B, rph = H / B;
    if (rpw < 2 || rph < 2) { *why = "need at least 2x2 range blocks"; return FIC_E_ARG; }
    int dpw = 2 * rpw - 3, dph = 2 * rph - 3;
    if (wk < 1 || wk > dpw || wk > dph) { *why = "widthKernel must be in [1, min(domain blocks per width, per height)]"; return FIC_E_ARG; }
    int64_t ND = (int64_t)dpw * dph;
    // The reference keeps indices in float (FC:124, FC:629): exact only below 2^24.
    if (ND >= (1 << 24) || (int64_t)wk * wk >= (1 << 24)) { *why = "domain pool too large for the reference's float index (>= 2^24)"; return FIC_E_ARG; }
    g->W = W; g->H = H; g->B = B; g->n = B * B; g->wk = wk;
    g->rpw = rpw; g->rph = rph; g->dpw = dpw; g->dph = dph;
    g->sw = W / 2; g->sh = H / 2; g->step = B / 4; g->C = mode == FIC_MODE_RGB ? 3 : 1;
    g->n_iso = mode == FIC_MODE_GREY_ISO ? 8 : 1;
    g->NR = (int64_t)rpw * rph; g->ND = ND;
    return FIC_OK;
}

// ------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------
struct fic_handle {
    int device = 0;
    int num_sms = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[8] = {nullptr};
    Work w;
    int engine_opt = FIC_ENGINE_AUTO;
    int umma_kind = FIC_UMMA_KIND_AUTO;
    int umma_pair = FIC_UMMA_PAIR_AUTO;  // FIC_OPT_UMMA_PAIR
    int pair_used = 0;                   // did the last tcgen05 search run the CTA-pair kernel
    int f16_state = 0;  // kind::f16 self-test: 0 not run yet, 1 exact, -1 not exact on this device (use kind::i8)
    fic_timings tm;
    char err[512];
    bool tm_pending_dev = false;
    // pinned scratch for small device->host reads
    unsigned long long *h_acc = nullptr;
    // pinned staging for small code tables: one device->host copy instead of two (info and qcodes are adjacent on the
    // device), then a host memcpy into the caller's arrays -- the reference's default image (1024 ranges) is all latency
    uint8_t *h_stage = nullptr;
};

static char g_create_err[512] = "";
constexpr size_t kStageBytes = 128 << 10;

static int set_err(fic_handle *h, int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(h ? h->err : g_create_err, 512, fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return set_err(h, FIC_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// Host entries copy from / to caller-owned buffers asynchronously and synchronise before they return.  This guard
// makes that hold on EVERY return path: an early `return rc` after the first enqueue would otherwise leave a copy in
// flight on a buffer the caller is free to reuse (pinned buffers are read by the copy engine directly).
struct DrainOnExit {
    cudaStream_t s;
    explicit DrainOnExit(cudaStream_t st) : s(st) {}
    ~DrainOnExit() { cudaStreamSynchronize(s); }
};

enum Slot { S_ARGB, S_SRC, S_DEC, S_DSUM, S_DSQ, S_RSUM, S_BEST, S_INFO, S_Q, S_OPA, S_OPB, S_IMG, S_DEC2, S_DCODE, S_PERR, S_STATE, S_DEC3, S_REPLAY };

template <typename T>
static int ensure(fic_handle *h, T *&p, int slot, size_t bytes)
{
    if (bytes == 0) bytes = 16;
    if (h->w.cap[slot] >= bytes && p) return FIC_OK;
    if (p) cudaFree(p);
    p = nullptr;
    h->w.cap[slot] = 0;
    size_t want = (bytes + 255) & ~(size_t)255;
    cudaError_t e = cudaMalloc((void **)&p, want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(h, FIC_E_NOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
    }
    h->w.cap[slot] = want;
    return FIC_OK;
}

#define ENSURE(ptr, slot, bytes)                       \
    do {                                               \
        int rc_ = ensure(h, ptr, slot, (size_t)(bytes)); \
        if (rc_) return rc_;                           \
    } while (0)

// The error of a decoder entry (fic_decode.cu); out_of_pool: the message for a code outside the domain pool.
static int decode_err(fic_handle *h, const DecodeStatus &st, const char *out_of_pool)
{
    if (st.rc == FIC_E_CUDA) return set_err(h, FIC_E_CUDA, "%s failed: %s (%s:%d)", st.call, cudaGetErrorString(st.cuda), st.file, st.line);
    return st.rc ? set_err(h, st.rc, "%s", out_of_pool) : FIC_OK;
}

extern "C" {

const char *fic_version(void) { return "fic_b200 0.2 (sm_100a)"; }

int fic_create(int device, fic_handle **out)
{
    fic_handle *h = nullptr;
    if (!out) return set_err(nullptr, FIC_E_ARG, "fic_create: out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return set_err(nullptr, FIC_E_CUDA, "no CUDA device available (%s); libfic_b200 has no CPU fallback",
                       e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    }
    if (device < 0 || device >= count) return set_err(nullptr, FIC_E_ARG, "device %d out of range [0,%d)", device, count);
    h = new (std::nothrow) fic_handle();
    if (!h) return set_err(nullptr, FIC_E_NOMEM, "out of host memory");
    h->err[0] = 0;
    memset(&h->tm, 0, sizeof h->tm);
    h->device = device;
    cudaDeviceProp prop;
    if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
        set_err(nullptr, FIC_E_CUDA, "cudaSetDevice(%d): %s", device, cudaGetErrorString(e));
        delete h;
        return FIC_E_CUDA;
    }
    if (prop.major != 10) {
        set_err(nullptr, FIC_E_CUDA, "device %d is sm_%d%d; libfic_b200 is built for sm_100a (B200) only", device,
                prop.major, prop.minor);
        delete h;
        return FIC_E_CUDA;
    }
    h->num_sms = prop.multiProcessorCount;
    if ((e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking)) != cudaSuccess) {
        set_err(nullptr, FIC_E_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
        delete h;
        return FIC_E_CUDA;
    }
    h->stream = h->own_stream;
    for (int i = 0; i < 8 && e == cudaSuccess; i++) e = cudaEventCreate(&h->ev[i]);
    if (e == cudaSuccess) e = cudaHostAlloc((void **)&h->h_acc, 64 * sizeof(unsigned long long), cudaHostAllocDefault);
    if (e == cudaSuccess) e = cudaHostAlloc((void **)&h->h_stage, kStageBytes, cudaHostAllocDefault);
    if (e != cudaSuccess) {
        set_err(nullptr, FIC_E_CUDA, "creating events / pinned scratch: %s", cudaGetErrorString(e));
        fic_destroy(h);
        return FIC_E_CUDA;
    }
    *out = h;
    return FIC_OK;
}

void fic_destroy(fic_handle *h)
{
    if (!h) return;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    Work &w = h->w;
    void *ptrs[] = {w.argb, w.src, w.dec, w.dsum, w.dsq, w.rsum, w.best, w.info, w.q, w.opA, w.opB,
                    w.img, w.dec2, w.dcode, w.perr, w.state, w.dec3, w.replay};
    for (void *p : ptrs)
        if (p) cudaFree(p);
    for (int i = 0; i < 8; i++)
        if (h->ev[i]) cudaEventDestroy(h->ev[i]);
    if (h->h_acc) cudaFreeHost(h->h_acc);
    if (h->h_stage) cudaFreeHost(h->h_stage);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
}

const char *fic_last_error(const fic_handle *h) { return h ? h->err : g_create_err; }

int fic_set_option(fic_handle *h, int option, int value)
{
    if (!h) return FIC_E_ARG;
    if (option == FIC_OPT_ENGINE && value >= FIC_ENGINE_AUTO && value <= FIC_ENGINE_FUSED) {
        h->engine_opt = value;
        return FIC_OK;
    }
    if (option == FIC_OPT_UMMA_KIND && value >= FIC_UMMA_KIND_AUTO && value <= FIC_UMMA_KIND_F16) {
        h->umma_kind = value;
        return FIC_OK;
    }
    if (option == FIC_OPT_UMMA_PAIR && value >= FIC_UMMA_PAIR_AUTO && value <= FIC_UMMA_PAIR_ON) {
        h->umma_pair = value;
        return FIC_OK;
    }
    return set_err(h, FIC_E_ARG, "unknown option %d / value %d", option, value);
}

int fic_get_option(fic_handle *h, int option, int *value)
{
    if (!h || !value) return FIC_E_ARG;
    if (option == FIC_OPT_ENGINE) { *value = h->engine_opt; return FIC_OK; }
    if (option == FIC_OPT_UMMA_KIND) { *value = h->umma_kind; return FIC_OK; }
    if (option == FIC_OPT_UMMA_PAIR) { *value = h->umma_pair; return FIC_OK; }
    if (option == FIC_OPT_UMMA_PAIR_USED) { *value = h->pair_used; return FIC_OK; }
    if (option == FIC_OPT_F16_EXACT) {
        if (h->f16_state == 0) {
            CU(cudaSetDevice(h->device));
            const char *why = nullptr;
            int ok = umma_f16_selftest(h->num_sms, h->stream, &why);
            if (ok < 0) return set_err(h, FIC_E_CUDA, "kind::f16 self-test failed to run: %s", why ? why : "?");
            h->f16_state = ok ? 1 : -1;
        }
        *value = h->f16_state > 0;
        return FIC_OK;
    }
    return set_err(h, FIC_E_ARG, "unknown option %d", option);
}

int fic_set_stream(fic_handle *h, void *cuda_stream)
{
    if (!h) return FIC_E_ARG;
    h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
    return FIC_OK;
}

static void collect_timings(fic_handle *h, bool with_copies);

int fic_get_timings(const fic_handle *h, fic_timings *out)
{
    if (!h || !out) return FIC_E_ARG;
    fic_handle *hm = const_cast<fic_handle *>(h);
    if (hm->tm_pending_dev) {  // asynchronous device entry: events are final once the stream has drained
        if (cudaEventQuery(hm->ev[4]) == cudaSuccess) {
            collect_timings(hm, false);
            hm->tm_pending_dev = false;
        }
    }
    *out = h->tm;
    return FIC_OK;
}

int fic_geometry(int W, int H, int B, int wk, int64_t *n_ranges, int64_t *n_domains)
{
    Geom g;
    int rc = make_geom(W, H, B, wk, 0, &g, nullptr);
    if (rc) return rc;
    if (n_ranges) *n_ranges = g.NR;
    if (n_domains) *n_domains = g.ND;
    return FIC_OK;
}

int fic_sync(fic_handle *h)
{
    if (!h) return FIC_E_ARG;
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    return FIC_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------
// encode
// ------------------------------------------------------------------------------------

// Which search engine a call runs (FIC_OPT_ENGINE): the tcgen05 search for whole-pool windows with enough work to
// fill the GPU, else the fused one-launch encode for the reference's GUI windows (widthKernel <= 16), else the
// multi-kernel direct path.
static int pick_engine(fic_handle *h, const Geom &g, int64_t j0, int64_t j1, int *engine)
{
    *engine = FIC_ENGINE_DIRECT;
    if (h->engine_opt == FIC_ENGINE_UMMA) {
        if (!umma_applicable(g))
            return set_err(h, FIC_E_ARG, "tcgen05 search needs widthKernel == domain blocks per width == per height (and no isometries for RGB)");
        *engine = FIC_ENGINE_UMMA;
    } else if (h->engine_opt == FIC_ENGINE_FUSED) {
        if (!fused_encode_applicable(g)) return set_err(h, FIC_E_ARG, "the fused encode needs widthKernel <= 16 and no isometries");
        *engine = FIC_ENGINE_FUSED;
    } else if (h->engine_opt == FIC_ENGINE_AUTO) {
        // the fused kernel spends one CTA per range block and wins where launches dominate (<= 16 K range blocks,
        // 1.8 ms against 0.45 ms for the multi-kernel path at 4096^2, widthKernel 2: measured, profiles/README.md)
        if (umma_applicable(g) && (j1 - j0) * g.ND >= (int64_t)1 << 22) *engine = FIC_ENGINE_UMMA;
        else if (fused_encode_applicable(g) && g.NR <= 16384) *engine = FIC_ENGINE_FUSED;
    }
    return FIC_OK;
}

// Fused windowed encode straight from the caller's pixels (ARGB ints or planes).  Records events 1..4.  n_images > 1: a
// batch, every range of that many images back to back (launch_encode_fused).
static int encode_fused_on_device(fic_handle *h, const Geom &g, const void *d_pixels, int is_argb, int64_t j0, int64_t j1,
                                  float *d_info, int32_t *d_q, int n_images = 1)
{
    cudaStream_t s = h->stream;
    // one kernel: events 1 and 4 bracket it (collect_timings reads the stages of this engine from those two alone)
    CU(cudaEventRecord(h->ev[1], s));
    const int launches = launch_encode_fused(d_pixels, is_argb, g, j0, j1, d_info, d_q, s, n_images);
    CU(cudaEventRecord(h->ev[4], s));
    CU(cudaGetLastError());
    h->tm.engine = FIC_ENGINE_FUSED;
    h->tm.launches += launches;
    h->tm.search_evals = (double)(j1 - j0) * (double)g.wk * (double)g.wk;
    return FIC_OK;
}

// The MMA kind a tcgen05 search runs with, and whether it runs at all: the first kind::f16 search of a handle verifies,
// once, that this device's f16 tensor path accumulates the integer covariances exactly; a device that does not runs
// kind::i8 instead.  RGB has a kind::f16 tensor path only; without an exact f16 path it stays on the CUDA-core kernel
// (*engine becomes FIC_ENGINE_DIRECT).  (The self-test allocates and synchronises on this stream: one-time cost of the
// first such call; fic_get_option(FIC_OPT_F16_EXACT) runs it ahead of time.)
static int umma_kind_of(fic_handle *h, const Geom &g, int *engine, int *kind)
{
    *kind = h->umma_kind;
    if (*engine != FIC_ENGINE_UMMA) return FIC_OK;
    const bool rgb = g.C == 3;
    const bool wants_f16 = rgb || (g.B != 16 && (*kind == FIC_UMMA_KIND_F16 || (*kind == FIC_UMMA_KIND_AUTO && umma_default_kind(g) == FIC_UMMA_KIND_F16)));
    if (wants_f16 && h->f16_state == 0) {
        const char *why = nullptr;
        int ok = umma_f16_selftest(h->num_sms, h->stream, &why);
        if (ok < 0) return set_err(h, FIC_E_CUDA, "kind::f16 self-test failed to run: %s", why ? why : "?");
        h->f16_state = ok ? 1 : -1;
    }
    if (wants_f16 && h->f16_state < 0) {
        if (rgb) *engine = FIC_ENGINE_DIRECT;
        else *kind = FIC_UMMA_KIND_I8;
    }
    return FIC_OK;
}

// Pool build + search + solve on device-resident planes.  Records events 1..4.  n_images > 1 (tcgen05 engine only):
// a group of images, planes back to back at d_src, ranges [0, NR) of each, codes in [n][NR] tables -- one launch of
// every kernel for the whole group (launch_search_umma).
static int encode_on_device(fic_handle *h, const Geom &g, const uint8_t *d_src, int64_t j0, int64_t j1,
                            float *d_info, int32_t *d_q, int engine, int n_images = 1)
{
    Work &w = h->w;
    cudaStream_t s = h->stream;
    if (engine == FIC_ENGINE_FUSED) return encode_fused_on_device(h, g, d_src, 0, j0, j1, d_info, d_q);
    const size_t n = (size_t)n_images;
    ENSURE(w.dec, S_DEC, (size_t)g.C * g.sw * g.sh * n);
    ENSURE(w.dsum, S_DSUM, sizeof(int32_t) * g.C * g.ND * n);
    ENSURE(w.dsq, S_DSQ, sizeof(int32_t) * g.C * g.ND * n);
    ENSURE(w.rsum, S_RSUM, sizeof(int32_t) * g.C * g.NR * n);
    ENSURE(w.best, S_BEST, sizeof(int32_t) * g.NR * n);
    if (g.C == 3) ENSURE(w.dec3, S_DEC3, sizeof(uint16_t) * (size_t)g.sw * g.sh * n);  // R + G + B of the decimated planes
    int kind, rc;
    h->pair_used = 0;
    if ((rc = umma_kind_of(h, g, &engine, &kind))) return rc;
    if (n_images > 1 && engine != FIC_ENGINE_UMMA) return set_err(h, FIC_E_ARG, "a group of images runs the tcgen05 search only");
    if (engine == FIC_ENGINE_UMMA) {
        ENSURE(w.opA, S_OPA, umma_opA_bytes(g, j0, j1, h->num_sms, kind, n_images));
        ENSURE(w.opB, S_OPB, umma_opB_bytes(g, kind, n_images));
    }
    Work call = w;  // per-call view: the source planes may belong to the caller
    call.src = const_cast<uint8_t *>(d_src);
    int launches = 0;
    CU(cudaEventRecord(h->ev[1], s));
    launches += launch_decimate(d_src, w.dec, g, s, n_images);
    launches += launch_domain_stats(w.dec, w.dsum, w.dsq, g, s, n_images);
    launches += launch_range_stats(d_src, w.rsum, g, s, n_images);
    CU(cudaEventRecord(h->ev[2], s));
    CU(cudaEventRecord(h->ev[6], s));  // (the tcgen05 launcher re-records 6 / 7 around its search kernel)
    CU(cudaEventRecord(h->ev[7], s));
    if (engine == FIC_ENGINE_UMMA) {
        const char *why = nullptr;
        int nl = launch_search_umma(call, g, j0, j1, h->num_sms, s, &why, kind, h->ev[6], h->ev[7], h->umma_pair, &h->pair_used,
                                    nullptr, 0, nullptr, n_images);
        if (nl < 0) return set_err(h, FIC_E_CUDA, "tcgen05 search launch failed: %s", why ? why : "?");
        launches += nl;
    } else {
        if (g.C == 3) launches += launch_sum_planes(w.dec, w.dec3, g, s);
        CU(cudaEventRecord(h->ev[6], s));
        launches += launch_search_direct(call, g, j0, j1, s);
        CU(cudaEventRecord(h->ev[7], s));
    }
    CU(cudaEventRecord(h->ev[3], s));
    if (n_images > 1) launches += launch_solve(call, g, 0, g.NR * n_images, d_info, d_q, s);  // the flat range of the group
    else launches += launch_solve(call, g, j0, j1, d_info, d_q, s);
    CU(cudaEventRecord(h->ev[4], s));
    CU(cudaGetLastError());
    h->tm.engine = engine;
    h->tm.launches += launches;
    h->tm.search_evals = (double)(j1 - j0) * (double)g.wk * (double)g.wk * (double)g.n_iso * (double)n_images;
    return FIC_OK;
}

static void collect_timings(fic_handle *h, bool with_copies)
{
    float ms = 0;
    if (h->tm.engine == FIC_ENGINE_FUSED) {  // a single kernel between events 1 and 4
        if (with_copies && cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]) == cudaSuccess) h->tm.h2d_ms = ms;
        if (cudaEventElapsedTime(&ms, h->ev[1], h->ev[4]) == cudaSuccess) h->tm.search_ms = h->tm.kernel_ms = ms;
        if (with_copies && cudaEventElapsedTime(&ms, h->ev[4], h->ev[5]) == cudaSuccess) h->tm.d2h_ms = ms;
        if (cudaEventElapsedTime(&ms, h->ev[with_copies ? 0 : 1], h->ev[with_copies ? 5 : 4]) == cudaSuccess) h->tm.total_ms = ms;
        return;
    }
    if (with_copies && cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]) == cudaSuccess) h->tm.h2d_ms = ms;
    if (cudaEventElapsedTime(&ms, h->ev[1], h->ev[2]) == cudaSuccess) h->tm.pool_ms = ms;
    if (cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]) == cudaSuccess) h->tm.search_ms = ms;
    if (cudaEventElapsedTime(&ms, h->ev[6], h->ev[7]) == cudaSuccess) h->tm.kernel_ms = ms;
    if (cudaEventElapsedTime(&ms, h->ev[3], h->ev[4]) == cudaSuccess) h->tm.solve_ms = ms;
    if (with_copies && cudaEventElapsedTime(&ms, h->ev[4], h->ev[5]) == cudaSuccess) h->tm.d2h_ms = ms;
    if (cudaEventElapsedTime(&ms, h->ev[with_copies ? 0 : 1], h->ev[with_copies ? 5 : 4]) == cudaSuccess)
        h->tm.total_ms = ms;
}

// `pixels` is the reference's int32 ARGB array (src_u8 == 0: FC:109 / FC:171 hand over RasterImage.argb) or 8-bit
// planes (src_u8 == 1: grey W*H bytes = the red channel, RGB 3*W*H bytes R, G, B) -- a quarter of the upload.
static int encode_host(fic_handle *h, int is_rgb, const void *pixels, int src_u8, int W, int H, int B, int wk, int64_t j0,
                       int64_t j1, float *info, int32_t *qcodes)
{
    if (!h) return FIC_E_ARG;
    if (!pixels || (!info && !qcodes)) return set_err(h, FIC_E_ARG, "the image and at least one of info/qcodes must be non-NULL");
    Geom g;
    const char *why = "";
    int rc = make_geom(W, H, B, wk, is_rgb, &g, &why);
    if (rc) return set_err(h, rc, "%s", why);
    if (j0 < 0 || j1 > g.NR || j0 > j1) return set_err(h, FIC_E_ARG, "range interval [%lld,%lld) outside [0,%lld]", (long long)j0, (long long)j1, (long long)g.NR);
    CU(cudaSetDevice(h->device));
    memset(&h->tm, 0, sizeof h->tm);
    Work &w = h->w;
    cudaStream_t s = h->stream;
    int S = code_stride(g);
    int engine;
    if ((rc = pick_engine(h, g, j0, j1, &engine))) return rc;
    const bool fused_argb = engine == FIC_ENGINE_FUSED && !src_u8;  // the fused kernel reads the ARGB ints itself
    if (!src_u8) ENSURE(w.argb, S_ARGB, sizeof(int32_t) * (size_t)W * H);
    if (!fused_argb) ENSURE(w.src, S_SRC, (size_t)g.C * W * H);
    const size_t table = sizeof(float) * (size_t)g.NR * S;  // bytes of one code table (float and int32 entries alike)
    const bool staged = info && qcodes && 2 * table <= kStageBytes;  // small tables: one copy through pinned staging
    if (staged) {
        ENSURE(w.info, S_INFO, 2 * table);  // [imageInfo floats][writeData ints], adjacent
    } else {
        ENSURE(w.info, S_INFO, table);
        ENSURE(w.q, S_Q, table);
    }
    float *const d_info = w.info;
    int32_t *const d_q = staged ? (int32_t *)((uint8_t *)w.info + table) : w.q;
    DrainOnExit drain(s);
    CU(cudaEventRecord(h->ev[0], s));
    if (src_u8) {
        CU(cudaMemcpyAsync(w.src, pixels, (size_t)g.C * W * H, cudaMemcpyHostToDevice, s));
    } else {
        CU(cudaMemcpyAsync(w.argb, pixels, sizeof(int32_t) * (size_t)W * H, cudaMemcpyHostToDevice, s));
        if (!fused_argb) h->tm.launches += launch_unpack(w.argb, w.src, W, H, g.C, s);
    }
    rc = fused_argb ? encode_fused_on_device(h, g, w.argb, 1, j0, j1, d_info, d_q)
                    : encode_on_device(h, g, w.src, j0, j1, d_info, d_q, engine);
    if (rc) return rc;
    if (j1 > j0) {
        if (staged) {
            CU(cudaMemcpyAsync(h->h_stage, d_info, 2 * table, cudaMemcpyDeviceToHost, s));
        } else {
            if (info) CU(cudaMemcpyAsync(info + j0 * S, d_info + j0 * S, sizeof(float) * (j1 - j0) * S, cudaMemcpyDeviceToHost, s));
            if (qcodes) CU(cudaMemcpyAsync(qcodes + j0 * S, d_q + j0 * S, sizeof(int32_t) * (j1 - j0) * S, cudaMemcpyDeviceToHost, s));
        }
    }
    CU(cudaEventRecord(h->ev[5], s));
    CU(cudaStreamSynchronize(s));
    if (staged && j1 > j0) {
        memcpy(info + j0 * S, h->h_stage + sizeof(float) * j0 * S, sizeof(float) * (j1 - j0) * S);
        memcpy(qcodes + j0 * S, h->h_stage + table + sizeof(int32_t) * j0 * S, sizeof(int32_t) * (j1 - j0) * S);
    }
    collect_timings(h, true);
    return FIC_OK;
}

// ---- batches of same-size images ----------------------------------------------------------------------------------

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
static_assert(kDecodeBatchMax * sizeof(DecodeState) <= kStageBytes, "a decode group's state blocks come back through h_stage");

// The checks every batch entry adds to make_geom's: n_images >= 1 and byte counts of the whole batch that fit.
static int batch_geom(fic_handle *h, int mode, int n_images, int W, int H, int B, int wk, Geom *g)
{
    if (n_images < 1) return set_err(h, FIC_E_ARG, "n_images must be >= 1");
    const char *why = "";
    const int rc = make_geom(W, H, B, wk, mode, g, &why);
    if (rc) return set_err(h, rc, "%s", why);
    int64_t bytes;
    if (__builtin_mul_overflow((int64_t)n_images, (int64_t)W * H * 4, &bytes) ||
        __builtin_mul_overflow((int64_t)n_images, g->NR * code_stride(*g) * 4, &bytes))
        return set_err(h, FIC_E_ARG, "n_images = %d images of %d x %d overflow a byte count", n_images, W, H);
    return FIC_OK;
}

// Images per tcgen05 group of a batch (see kBatchUmmaImages / kBatchUmmaBytes), at most `limit`.
static int umma_group_size(fic_handle *h, const Geom &g, int kind, int limit)
{
    int n = limit < kBatchUmmaImages ? limit : kBatchUmmaImages;
    auto bytes = [&](int k) { return umma_opA_bytes(g, 0, g.NR, h->num_sms, kind, k) + umma_opB_bytes(g, kind, k); };
    for (size_t b; n > 1 && (b = bytes(n)) > kBatchUmmaBytes;) n = (int)((double)n * kBatchUmmaBytes / b);
    return n > 1 ? n : 1;
}

// Per-stage times of the last encode_on_device (events 1..4, 6, 7) added to the call's.
static void add_stage_times(fic_handle *h, fic_timings *acc)
{
    float ms = 0;
    if (cudaEventElapsedTime(&ms, h->ev[1], h->ev[2]) == cudaSuccess) acc->pool_ms += ms;
    if (cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]) == cudaSuccess) acc->search_ms += ms;
    if (cudaEventElapsedTime(&ms, h->ev[6], h->ev[7]) == cudaSuccess) acc->kernel_ms += ms;
    if (cudaEventElapsedTime(&ms, h->ev[3], h->ev[4]) == cudaSuccess) acc->solve_ms += ms;
}

// A batch encode: the codes of n_images images back to back, [n][NR][S], each equal to a single encode of that image.
// Where pick_engine chooses the fused encode, one launch per group covers every range of every image; on the tcgen05
// engine (full-pool windows: forced, AUTO where the single call runs it, or AUTO instead of the CUDA-core search for
// groups of kBatchUmmaMinImages and more) every group is one
// block-diagonal search -- one launch of each pool, sort, pack, search, refine and solve kernel; otherwise each image
// runs encode_on_device.  Groups of images go up in one copy and their codes come down in one.
static int encode_batch_host(fic_handle *h, int mode, const void *pixels, int src_u8, int n_images, int W, int H, int B, int wk,
                             float *info, int32_t *qcodes)
{
    if (!h) return FIC_E_ARG;
    if (!pixels || (!info && !qcodes)) return set_err(h, FIC_E_ARG, "the images and at least one of info/qcodes must be non-NULL");
    Geom g;
    int rc = batch_geom(h, mode, n_images, W, H, B, wk, &g);
    if (rc) return rc;
    CU(cudaSetDevice(h->device));
    memset(&h->tm, 0, sizeof h->tm);
    Work &w = h->w;
    cudaStream_t s = h->stream;
    int engine;
    if ((rc = pick_engine(h, g, 0, g.NR, &engine))) return rc;
    const int S = code_stride(g);
    const size_t plane = (size_t)W * H, image_bytes = src_u8 ? g.C * plane : sizeof(int32_t) * plane;
    const size_t codes = (size_t)g.NR * S, table = sizeof(float) * codes;  // one image's code table (float and int32 alike)
    int group = (int)(kBatchGroupBytes / image_bytes < (size_t)n_images ? (kBatchGroupBytes / image_bytes > 0 ? kBatchGroupBytes / image_bytes : 1) : n_images);
    // AUTO: the tcgen05 group search instead of the CUDA-core search for groups of enough images, else the single
    // call's engine
    int want = h->engine_opt == FIC_ENGINE_AUTO && engine == FIC_ENGINE_DIRECT && umma_applicable(g) ? FIC_ENGINE_UMMA : engine, kind = 0;
    if ((rc = umma_kind_of(h, g, &want, &kind))) return rc;
    if (want == FIC_ENGINE_UMMA) {
        const int ug = umma_group_size(h, g, kind, group);
        if (engine == FIC_ENGINE_UMMA || ug >= kBatchUmmaMinImages) {
            engine = FIC_ENGINE_UMMA;
            group = ug;
        }
    } else if (engine == FIC_ENGINE_UMMA) {
        engine = want;  // RGB on a device without an exact kind::f16 path: the CUDA-core search, image by image
    }
    const bool fused = engine == FIC_ENGINE_FUSED, grouped = engine == FIC_ENGINE_UMMA;
    if (src_u8) {
        ENSURE(w.src, S_SRC, image_bytes * group);
    } else {
        ENSURE(w.argb, S_ARGB, image_bytes * group);
        if (!fused) ENSURE(w.src, S_SRC, g.C * plane * (grouped ? group : 1));  // planes unpacked before the encode
    }
    ENSURE(w.info, S_INFO, table * group);
    ENSURE(w.q, S_Q, table * group);
    DrainOnExit drain(s);
    fic_timings stages;  // the tcgen05 engine: per-stage times summed over the groups
    memset(&stages, 0, sizeof stages);
    CU(cudaEventRecord(h->ev[0], s));
    for (int i0 = 0; i0 < n_images; i0 += group) {
        const int gn = n_images - i0 < group ? n_images - i0 : group;
        void *d_pixels = src_u8 ? (void *)w.src : (void *)w.argb;
        if (grouped && i0 > 0) {  // the previous group's stage events, before this group records them again
            CU(cudaStreamSynchronize(s));
            add_stage_times(h, &stages);
        }
        CU(cudaMemcpyAsync(d_pixels, (const uint8_t *)pixels + i0 * image_bytes, image_bytes * gn, cudaMemcpyHostToDevice, s));
        if (fused) {
            if ((rc = encode_fused_on_device(h, g, d_pixels, !src_u8, 0, g.NR, w.info, w.q, gn))) return rc;
        } else if (grouped) {
            if (!src_u8) h->tm.launches += launch_unpack(w.argb, w.src, W, H, g.C, s, gn);
            if ((rc = encode_on_device(h, g, w.src, 0, g.NR, w.info, w.q, engine, gn))) return rc;
        } else {
            for (int i = 0; i < gn; i++) {
                const uint8_t *d_src = w.src + i * g.C * plane;
                if (!src_u8) {
                    h->tm.launches += launch_unpack(w.argb + i * plane, w.src, W, H, g.C, s);
                    d_src = w.src;
                }
                if ((rc = encode_on_device(h, g, d_src, 0, g.NR, w.info + i * codes, w.q + i * codes, engine))) return rc;
            }
        }
        if (info) CU(cudaMemcpyAsync(info + i0 * codes, w.info, table * gn, cudaMemcpyDeviceToHost, s));
        if (qcodes) CU(cudaMemcpyAsync(qcodes + i0 * codes, w.q, table * gn, cudaMemcpyDeviceToHost, s));
    }
    CU(cudaEventRecord(h->ev[5], s));
    CU(cudaStreamSynchronize(s));
    CU(cudaGetLastError());
    if (grouped) add_stage_times(h, &stages);
    const int launches = h->tm.launches, used = h->tm.engine;
    memset(&h->tm, 0, sizeof h->tm);  // the per-stage events saw the last image or group only: report the whole call
    if (grouped) {
        h->tm.pool_ms = stages.pool_ms;
        h->tm.search_ms = stages.search_ms;
        h->tm.kernel_ms = stages.kernel_ms;
        h->tm.solve_ms = stages.solve_ms;
    }
    float ms = 0;
    if (cudaEventElapsedTime(&ms, h->ev[0], h->ev[5]) == cudaSuccess) h->tm.total_ms = ms;
    h->tm.engine = used;
    h->tm.launches = launches;
    h->tm.search_evals = (double)n_images * (double)g.NR * (double)g.wk * (double)g.wk * (double)g.n_iso;
    return FIC_OK;
}

// A batch decode (decode_batch_run): every image as a single decode with its own carry-in would give it.
static int decode_batch_host(fic_handle *h, int mode, int n_images, int W, int H, int B, int wk, const int32_t *qcodes,
                             int max_iters, int32_t *argb_out, uint8_t *planes_out, float *avg_error, int *iterations)
{
    if (!h) return FIC_E_ARG;
    if (!qcodes || (!argb_out && !planes_out)) return set_err(h, FIC_E_ARG, "codes and the output images must be non-NULL");
    if (max_iters < 1) return set_err(h, FIC_E_ARG, "max_iters must be >= 1");
    Geom g;
    int rc = batch_geom(h, mode, n_images, W, H, B, wk, &g);
    if (rc) return rc;
    CU(cudaSetDevice(h->device));
    memset(&h->tm, 0, sizeof h->tm);
    Work &w = h->w;
    cudaStream_t s = h->stream;
    const int S = code_stride(g);
    const size_t plane = (size_t)W * H;
    const int batch = decode_batch_group(g), group = batch < n_images ? batch : n_images;
    const size_t k = group > 0 ? group : 1;  // images the one-launch workspace holds (decode_run needs one)
    ENSURE(w.q, S_Q, sizeof(int32_t) * g.NR * S * k);
    ENSURE(w.dcode, S_DCODE, sizeof(float) * g.NR * (S + 1) * k);
    ENSURE(w.img, S_IMG, g.C * plane * k);
    ENSURE(w.dec, S_DEC, (size_t)g.C * g.sw * g.sh * k);
    ENSURE(w.dec2, S_DEC2, (size_t)g.C * g.sw * g.sh * k);
    ENSURE(w.state, S_STATE, (sizeof(DecodeState) + sizeof(float)) * k);  // state blocks, then the carries
    if (argb_out) ENSURE(w.argb, S_ARGB, sizeof(int32_t) * plane * k);
    ENSURE(w.perr, S_PERR, sizeof(int32_t) * plane);
    const size_t replay_bytes = decode_replay_bytes((int64_t)plane);
    if (replay_bytes) ENSURE(w.replay, S_REPLAY, replay_bytes);
    DrainOnExit drain(s);
    CU(cudaEventRecord(h->ev[0], s));
    int bad = -1;
    const DecodeStatus st = decode_batch_run(w, g, n_images, group, qcodes, argb_out, planes_out, max_iters, avg_error, iterations,
                                             h->h_stage, h->h_acc, h->ev[0], h->ev[5], &h->tm, &bad, s);
    if (st.rc == FIC_E_STREAM)
        return set_err(h, FIC_E_STREAM, "image %d: a code indexes outside the domain pool (the reference would throw ArrayIndexOutOfBounds)", bad);
    return decode_err(h, st, "");
}

extern "C" {

int fic_encode_batch(fic_handle *h, int mode, const int32_t *argb, int n_images, int W, int H, int B, int wk, float *info,
                     int32_t *qcodes)
{
    return encode_batch_host(h, mode, argb, 0, n_images, W, H, B, wk, info, qcodes);
}

int fic_encode_batch_u8(fic_handle *h, int mode, const uint8_t *planes, int n_images, int W, int H, int B, int wk, float *info,
                        int32_t *qcodes)
{
    return encode_batch_host(h, mode, planes, 1, n_images, W, H, B, wk, info, qcodes);
}

int fic_decode_batch(fic_handle *h, int mode, int n_images, int W, int H, int B, int wk, const int32_t *qcodes, int max_iters,
                     int32_t *argb_out, float *avg_error, int *iterations)
{
    return decode_batch_host(h, mode, n_images, W, H, B, wk, qcodes, max_iters, argb_out, nullptr, avg_error, iterations);
}

int fic_decode_batch_u8(fic_handle *h, int mode, int n_images, int W, int H, int B, int wk, const int32_t *qcodes, int max_iters,
                        uint8_t *planes_out, float *avg_error, int *iterations)
{
    return decode_batch_host(h, mode, n_images, W, H, B, wk, qcodes, max_iters, nullptr, planes_out, avg_error, iterations);
}

int fic_encode_grey(fic_handle *h, const int32_t *argb, int W, int H, int B, int wk, int64_t range_begin,
                    int64_t range_end, float *info, int32_t *qcodes)
{
    return encode_host(h, 0, argb, 0, W, H, B, wk, range_begin, range_end, info, qcodes);
}

int fic_encode_grey_u8(fic_handle *h, const uint8_t *plane, int W, int H, int B, int wk, int64_t range_begin,
                       int64_t range_end, float *info, int32_t *qcodes)
{
    return encode_host(h, FIC_MODE_GREY, plane, 1, W, H, B, wk, range_begin, range_end, info, qcodes);
}

int fic_encode_rgb_planes(fic_handle *h, const uint8_t *planes, int W, int H, int B, int wk, int64_t range_begin,
                          int64_t range_end, float *info, int32_t *qcodes)
{
    return encode_host(h, FIC_MODE_RGB, planes, 1, W, H, B, wk, range_begin, range_end, info, qcodes);
}

int fic_encode_rgb(fic_handle *h, const int32_t *argb, int W, int H, int B, int wk, int64_t range_begin,
                   int64_t range_end, float *info, int32_t *qcodes)
{
    return encode_host(h, 1, argb, 0, W, H, B, wk, range_begin, range_end, info, qcodes);
}

int fic_encode_grey_iso(fic_handle *h, const int32_t *argb, int W, int H, int B, int wk, int64_t range_begin,
                        int64_t range_end, float *info, int32_t *qcodes)
{
    return encode_host(h, FIC_MODE_GREY_ISO, argb, 0, W, H, B, wk, range_begin, range_end, info, qcodes);
}

int fic_encode_planes_dev(fic_handle *h, const uint8_t *d_planes, int is_rgb, int W, int H, int B, int wk,
                          int64_t range_begin, int64_t range_end, float *d_info, int32_t *d_qcodes)
{
    if (!h) return FIC_E_ARG;
    if (!d_planes || (!d_info && !d_qcodes)) return set_err(h, FIC_E_ARG, "d_planes and at least one output must be non-NULL");
    if ((uintptr_t)d_planes & 15) return set_err(h, FIC_E_ARG, "d_planes must be 16-byte aligned (the kernels read it with vector loads)");
    Geom g;
    const char *why = "";
    int rc = make_geom(W, H, B, wk, is_rgb, &g, &why);
    if (rc) return set_err(h, rc, "%s", why);
    if (range_begin < 0 || range_end > g.NR || range_begin > range_end) return set_err(h, FIC_E_ARG, "range interval outside [0,NR]");
    CU(cudaSetDevice(h->device));
    // Timings of the previous asynchronous call are final once its events completed.
    memset(&h->tm, 0, sizeof h->tm);
    int engine;
    if ((rc = pick_engine(h, g, range_begin, range_end, &engine))) return rc;
    rc = encode_on_device(h, g, d_planes, range_begin, range_end, d_info, d_qcodes, engine);
    h->tm_pending_dev = rc == FIC_OK;
    return rc;
}

int fic_pin_host_buffer(fic_handle *h, void *ptr, size_t bytes)
{
    if (!h) return FIC_E_ARG;
    if (!ptr || bytes == 0) return set_err(h, FIC_E_ARG, "fic_pin_host_buffer: empty buffer");
    CU(cudaSetDevice(h->device));
    cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(h, e == cudaErrorMemoryAllocation ? FIC_E_NOMEM : FIC_E_CUDA, "cudaHostRegister(%zu bytes): %s", bytes,
                       cudaGetErrorString(e));
    }
    return FIC_OK;
}

int fic_unpin_host_buffer(fic_handle *h, void *ptr)
{
    if (!h) return FIC_E_ARG;
    if (!ptr) return set_err(h, FIC_E_ARG, "fic_unpin_host_buffer: NULL");
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));  // no copy of this handle may still be reading the buffer
    cudaError_t e = cudaHostUnregister(ptr);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(h, FIC_E_ARG, "cudaHostUnregister: %s", cudaGetErrorString(e));
    }
    return FIC_OK;
}

int fic_measure_mma_peak(fic_handle *h, int kind, int n_cols, double *tops)
{
    if (!h || !tops || (kind != FIC_UMMA_KIND_I8 && kind != FIC_UMMA_KIND_F16) || (n_cols != 128 && n_cols != 256))
        return FIC_E_ARG;
    CU(cudaSetDevice(h->device));
    const char *why = nullptr;
    double v = measure_mma_peak(h->num_sms, h->stream, 3, kind == FIC_UMMA_KIND_F16, n_cols, &why);
    if (v < 0) return set_err(h, FIC_E_CUDA, "tensor peak measurement failed: %s", why ? why : "?");
    *tops = v;
    return FIC_OK;
}

int fic_measure_int8_peak(fic_handle *h, double *tops) { return fic_measure_mma_peak(h, FIC_UMMA_KIND_I8, 256, tops); }

int fic_measure_mma_peak_pair(fic_handle *h, int kind, double *tops)
{
    if (!h || !tops || (kind != FIC_UMMA_KIND_I8 && kind != FIC_UMMA_KIND_F16)) return FIC_E_ARG;
    CU(cudaSetDevice(h->device));
    const char *why = nullptr;
    double v = measure_mma_peak_pair(h->num_sms, h->stream, 3, kind == FIC_UMMA_KIND_F16, nullptr, &why);
    if (v < 0) return set_err(h, FIC_E_CUDA, "tensor peak measurement (CTA pairs) failed: %s", why ? why : "?");
    *tops = v;
    return FIC_OK;
}

int fic_debug_float_sum(fic_handle *h, const int32_t *terms, int64_t count, float carry, float *sum)
{
    if (!h || !terms || !sum || count < 1) return FIC_E_ARG;
    CU(cudaSetDevice(h->device));
    Work &w = h->w;
    cudaStream_t s = h->stream;
    ENSURE(w.perr, S_PERR, sizeof(int32_t) * (size_t)count);
    ENSURE(w.state, S_STATE, sizeof(DecodeState));
    const size_t replay_bytes = decode_replay_bytes(count);
    if (replay_bytes) ENSURE(w.replay, S_REPLAY, replay_bytes);
    for (int64_t i = 0; i < count; i++)
        if (terms[i] < 0 || terms[i] > 3 * 255 * 255) return set_err(h, FIC_E_ARG, "terms must lie in [0, 3 * 255^2]");
    DrainOnExit drain(s);
    return decode_err(h, decode_float_sum(w, terms, count, carry, h->h_acc, sum, s), "");
}

int fic_build_pool(fic_handle *h, const int32_t *argb, int is_rgb, int W, int H, int B, uint8_t *decimated,
                   int32_t *dom_sum, int32_t *dom_sumsq)
{
    if (!h || !argb) return FIC_E_ARG;
    Geom g;
    const char *why = "";
    int rc = make_geom(W, H, B, 1, is_rgb, &g, &why);
    if (rc) return set_err(h, rc, "%s", why);
    CU(cudaSetDevice(h->device));
    Work &w = h->w;
    cudaStream_t s = h->stream;
    ENSURE(w.argb, S_ARGB, sizeof(int32_t) * (size_t)W * H);
    ENSURE(w.src, S_SRC, (size_t)g.C * W * H);
    ENSURE(w.dec, S_DEC, (size_t)g.C * g.sw * g.sh);
    ENSURE(w.dsum, S_DSUM, sizeof(int32_t) * g.C * g.ND);
    ENSURE(w.dsq, S_DSQ, sizeof(int32_t) * g.C * g.ND);
    DrainOnExit drain(s);
    CU(cudaMemcpyAsync(w.argb, argb, sizeof(int32_t) * (size_t)W * H, cudaMemcpyHostToDevice, s));
    launch_unpack(w.argb, w.src, W, H, g.C, s);
    launch_decimate(w.src, w.dec, g, s);
    launch_domain_stats(w.dec, w.dsum, w.dsq, g, s);
    CU(cudaGetLastError());
    if (decimated) CU(cudaMemcpyAsync(decimated, w.dec, (size_t)g.C * g.sw * g.sh, cudaMemcpyDeviceToHost, s));
    if (dom_sum) CU(cudaMemcpyAsync(dom_sum, w.dsum, sizeof(int32_t) * g.C * g.ND, cudaMemcpyDeviceToHost, s));
    if (dom_sumsq) CU(cudaMemcpyAsync(dom_sumsq, w.dsq, sizeof(int32_t) * g.C * g.ND, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    return FIC_OK;
}

// ------------------------------------------------------------------------------------
// decode / collage
// ------------------------------------------------------------------------------------

// Decoder entries.  Codes come from the host (`qcodes`) or from device memory (`d_qcodes`); the image goes to host ARGB
// ints (the reference's RasterImage.argb), host 8-bit planes or device 8-bit planes -- exactly one of the three.
static int decode_core(fic_handle *h, int is_rgb, int W, int H, int B, int wk, const int32_t *qcodes, const int32_t *d_qcodes,
                       int max_iters, int32_t *argb_out, uint8_t *planes_out, uint8_t *d_planes_out, float *avg_error,
                       int *iterations)
{
    if (!h) return FIC_E_ARG;
    if ((!qcodes && !d_qcodes) || (!argb_out && !planes_out && !d_planes_out)) return set_err(h, FIC_E_ARG, "codes and an output image must be non-NULL");
    if (max_iters < 1) return set_err(h, FIC_E_ARG, "max_iters must be >= 1");
    Geom g;
    const char *why = "";
    int rc = make_geom(W, H, B, wk, is_rgb, &g, &why);
    if (rc) return set_err(h, rc, "%s", why);
    CU(cudaSetDevice(h->device));
    memset(&h->tm, 0, sizeof h->tm);
    Work &w = h->w;
    cudaStream_t s = h->stream;
    int S = code_stride(g);
    size_t plane = (size_t)W * H;
    if (!d_qcodes) ENSURE(w.q, S_Q, sizeof(int32_t) * g.NR * S);
    ENSURE(w.dcode, S_DCODE, sizeof(float) * g.NR * (S + 1));
    if (!d_planes_out) ENSURE(w.img, S_IMG, g.C * plane);
    ENSURE(w.dec, S_DEC, (size_t)g.C * g.sw * g.sh);
    ENSURE(w.dec2, S_DEC2, (size_t)g.C * g.sw * g.sh);
    ENSURE(w.state, S_STATE, sizeof(DecodeState));
    if (argb_out) ENSURE(w.argb, S_ARGB, sizeof(int32_t) * plane);
    ENSURE(w.perr, S_PERR, sizeof(int32_t) * plane);  // per-pixel squared changes of the sweeps that may need a replay
    const size_t replay_bytes = decode_replay_bytes((int64_t)plane);
    if (replay_bytes) ENSURE(w.replay, S_REPLAY, replay_bytes);
    DrainOnExit drain(s);
    CU(cudaEventRecord(h->ev[0], s));
    if (!d_qcodes) CU(cudaMemcpyAsync(w.q, qcodes, sizeof(int32_t) * g.NR * S, cudaMemcpyHostToDevice, s));
    const DecodeStatus st = decode_run(w, g, d_qcodes ? d_qcodes : w.q, d_planes_out ? d_planes_out : w.img, argb_out, planes_out,
                                       max_iters, avg_error, iterations, h->h_acc, h->ev[0], h->ev[5], &h->tm, s);
    return decode_err(h, st, "a code indexes outside the domain pool (the reference would throw ArrayIndexOutOfBounds)");
}

int fic_decode(fic_handle *h, int is_rgb, int W, int H, int B, int wk, const int32_t *qcodes, int max_iters,
               int32_t *argb_out, float *avg_error, int *iterations)
{
    return decode_core(h, is_rgb, W, H, B, wk, qcodes, nullptr, max_iters, argb_out, nullptr, nullptr, avg_error, iterations);
}

int fic_decode_u8(fic_handle *h, int is_rgb, int W, int H, int B, int wk, const int32_t *qcodes, int max_iters,
                  uint8_t *planes_out, float *avg_error, int *iterations)
{
    return decode_core(h, is_rgb, W, H, B, wk, qcodes, nullptr, max_iters, nullptr, planes_out, nullptr, avg_error, iterations);
}

int fic_decode_planes_dev(fic_handle *h, int is_rgb, int W, int H, int B, int wk, const int32_t *d_qcodes, int max_iters,
                          uint8_t *d_planes_out, float *avg_error, int *iterations)
{
    if (h && ((uintptr_t)d_planes_out & 15)) return set_err(h, FIC_E_ARG, "d_planes_out must be 16-byte aligned");
    return decode_core(h, is_rgb, W, H, B, wk, nullptr, d_qcodes, max_iters, nullptr, nullptr, d_planes_out, avg_error, iterations);
}

int fic_collage(fic_handle *h, int is_rgb, const int32_t *argb, int W, int H, int B, int wk, float *info,
                int32_t *argb_out)
{
    if (!h) return FIC_E_ARG;
    if (!argb || !info || !argb_out) return set_err(h, FIC_E_ARG, "argb, info and argb_out must be non-NULL");
    Geom g;
    const char *why = "";
    int rc = make_geom(W, H, B, wk, is_rgb, &g, &why);
    if (rc) return set_err(h, rc, "%s", why);
    CU(cudaSetDevice(h->device));
    Work &w = h->w;
    cudaStream_t s = h->stream;
    int S = code_stride(g);
    size_t plane = (size_t)W * H;
    ENSURE(w.argb, S_ARGB, sizeof(int32_t) * plane);
    ENSURE(w.src, S_SRC, g.C * plane);
    ENSURE(w.dec, S_DEC, (size_t)g.C * g.sw * g.sh);
    ENSURE(w.info, S_INFO, sizeof(float) * g.NR * S);
    ENSURE(w.dcode, S_DCODE, sizeof(float) * g.NR * (S + 1));
    ENSURE(w.img, S_IMG, g.C * plane);
    ENSURE(w.state, S_STATE, sizeof(DecodeState));
    DrainOnExit drain(s);
    CU(cudaMemcpyAsync(w.argb, argb, sizeof(int32_t) * plane, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(w.info, info, sizeof(float) * g.NR * S, cudaMemcpyHostToDevice, s));
    launch_unpack(w.argb, w.src, W, H, g.C, s);
    launch_decimate(w.src, w.dec, g, s);  // FC:275 codebook of the source
    return decode_err(h, collage_run(w, g, argb_out, info, h->h_acc, s), "a code indexes outside the domain pool");
}

}  // extern "C"

// ------------------------------------------------------------------------------------
// multi-GPU handle (SURVEY 8b/8e): one process, n devices, one NCCL communicator
// ------------------------------------------------------------------------------------
//
// Range blocks are independent (FC:125-159 carries no state but the output index): device r encodes a contiguous
// slice of range rows.  Every device needs the whole image -- the domain pool spans it -- so the 8-bit plane(s) are
// uploaded ONCE (to the first device) and broadcast over NVLink with ncclBroadcast; each device then builds the full
// pool and searches its rows, and copies its code rows straight into the caller's arrays.  No other exchange exists
// on this path (there is no compute step followed by a collective to fuse).
//
// NCCL is bound at run time (dlopen of libnccl.so.2) so that the single-GPU library has no NCCL dependency; a multi
// handle over more than one device fails with FIC_E_CUDA when it cannot be loaded.
#include <dlfcn.h>

namespace {

typedef struct ncclComm *nccl_comm_t;
struct NcclApi {
    void *so = nullptr;
    int (*CommInitAll)(nccl_comm_t *, int, const int *) = nullptr;
    int (*CommDestroy)(nccl_comm_t) = nullptr;
    int (*Broadcast)(const void *, void *, size_t, int /*ncclDataType_t*/, int, nccl_comm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool load(char *err, size_t errlen)
    {
        if (so) return true;
        const char *names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char *n : names)
            if ((so = dlopen(n, RTLD_NOW | RTLD_GLOBAL))) break;
        if (!so) {
            snprintf(err, errlen, "cannot load NCCL (libnccl.so.2): %s", dlerror());
            return false;
        }
        CommInitAll = (decltype(CommInitAll))dlsym(so, "ncclCommInitAll");
        CommDestroy = (decltype(CommDestroy))dlsym(so, "ncclCommDestroy");
        Broadcast = (decltype(Broadcast))dlsym(so, "ncclBroadcast");
        GroupStart = (decltype(GroupStart))dlsym(so, "ncclGroupStart");
        GroupEnd = (decltype(GroupEnd))dlsym(so, "ncclGroupEnd");
        GetErrorString = (decltype(GetErrorString))dlsym(so, "ncclGetErrorString");
        if (!CommInitAll || !CommDestroy || !Broadcast || !GroupStart || !GroupEnd || !GetErrorString) {
            snprintf(err, errlen, "libnccl.so.2 lacks an expected symbol");
            dlclose(so);
            so = nullptr;
            return false;
        }
        return true;
    }
};
NcclApi g_nccl;
constexpr int kNcclUint8 = 1;  // ncclUint8 (nccl.h ncclDataType_t)
constexpr int kMaxDevices = 64;

}  // namespace

struct fic_multi {
    int n = 0;
    int devices[kMaxDevices];
    fic_handle *h[kMaxDevices] = {nullptr};
    nccl_comm_t comm[kMaxDevices] = {nullptr};
    bool has_comm = false;
    int64_t j0[kMaxDevices], j1[kMaxDevices];  // row slices of the last encode
    fic_timings tm;
    char err[512];
};

static char g_multi_err[512] = "";

static int merr(fic_multi *m, int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(m ? m->err : g_multi_err, 512, fmt, ap);
    va_end(ap);
    return code;
}

// Contiguous split of the rph range rows over n devices, in range-block units (the first rph % n devices get one
// row more) -- the same split as dist.py's partition_range_rows.
static void split_rows(int rph, int rpw, int n, int64_t *j0, int64_t *j1)
{
    const int base = rph / n, extra = rph % n;
    int row = 0;
    for (int r = 0; r < n; r++) {
        const int rows = base + (r < extra ? 1 : 0);
        j0[r] = (int64_t)row * rpw;
        j1[r] = (int64_t)(row + rows) * rpw;
        row += rows;
    }
}

// `pixels`: the reference's ARGB ints (src_u8 == 0) or 8-bit planes (src_u8 == 1), host memory.
static int multi_encode(fic_multi *m, int mode, const void *pixels, int src_u8, int W, int H, int B, int wk, float *info,
                        int32_t *qcodes)
{
    if (!m) return FIC_E_ARG;
    if (!pixels || (!info && !qcodes)) return merr(m, FIC_E_ARG, "the image and at least one of info/qcodes must be non-NULL");
    Geom g;
    const char *why = "";
    int rc = make_geom(W, H, B, wk, mode, &g, &why);
    if (rc) return merr(m, rc, "%s", why);
    const int S = code_stride(g);
    const size_t plane_bytes = (size_t)g.C * W * H;
    split_rows(g.rph, g.rpw, m->n, m->j0, m->j1);
    cudaError_t ce;
#define MCU(call)                                                                                     \
    do {                                                                                              \
        if ((ce = (call)) != cudaSuccess) {                                                           \
            for (int r_ = 0; r_ < m->n; r_++) { cudaSetDevice(m->devices[r_]); cudaStreamSynchronize(m->h[r_]->stream); } \
            return merr(m, FIC_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(ce), __FILE__, __LINE__); \
        }                                                                                             \
    } while (0)
    // workspaces
    for (int r = 0; r < m->n; r++) {
        fic_handle *h = m->h[r];
        MCU(cudaSetDevice(m->devices[r]));
        memset(&h->tm, 0, sizeof h->tm);
        if (r == 0 && !src_u8 && (rc = ensure(h, h->w.argb, S_ARGB, sizeof(int32_t) * (size_t)W * H))) return merr(m, rc, "%s", h->err);
        if ((rc = ensure(h, h->w.src, S_SRC, plane_bytes)) || (rc = ensure(h, h->w.info, S_INFO, sizeof(float) * g.NR * S)) ||
            (rc = ensure(h, h->w.q, S_Q, sizeof(int32_t) * g.NR * S)))
            return merr(m, rc, "%s", h->err);
    }
    // one upload, to the first device
    fic_handle *h0 = m->h[0];
    MCU(cudaSetDevice(m->devices[0]));
    MCU(cudaEventRecord(h0->ev[0], h0->stream));
    if (src_u8) {
        MCU(cudaMemcpyAsync(h0->w.src, pixels, plane_bytes, cudaMemcpyHostToDevice, h0->stream));
    } else {
        MCU(cudaMemcpyAsync(h0->w.argb, pixels, sizeof(int32_t) * (size_t)W * H, cudaMemcpyHostToDevice, h0->stream));
        h0->tm.launches += launch_unpack(h0->w.argb, h0->w.src, W, H, g.C, h0->stream);
    }
    // one broadcast of the planes over NVLink (every device's stream orders its own part)
    if (m->n > 1) {
        int nrc = g_nccl.GroupStart();
        for (int r = 0; r < m->n && nrc == 0; r++) {
            MCU(cudaSetDevice(m->devices[r]));
            nrc = g_nccl.Broadcast(h0->w.src, m->h[r]->w.src, plane_bytes, kNcclUint8, 0, m->comm[r], m->h[r]->stream);
        }
        const int nrc2 = g_nccl.GroupEnd();
        if (nrc == 0) nrc = nrc2;
        if (nrc) {
            for (int r = 0; r < m->n; r++) { cudaSetDevice(m->devices[r]); cudaStreamSynchronize(m->h[r]->stream); }
            return merr(m, FIC_E_CUDA, "ncclBroadcast failed: %s", g_nccl.GetErrorString(nrc));
        }
    }
    // every device: full pool, its own range rows, codes straight into the caller's arrays
    for (int r = 0; r < m->n; r++) {
        fic_handle *h = m->h[r];
        MCU(cudaSetDevice(m->devices[r]));
        int engine;
        rc = pick_engine(h, g, m->j0[r], m->j1[r], &engine);
        if (!rc) rc = encode_on_device(h, g, h->w.src, m->j0[r], m->j1[r], h->w.info, h->w.q, engine);
        if (rc) {
            for (int q = 0; q < m->n; q++) { cudaSetDevice(m->devices[q]); cudaStreamSynchronize(m->h[q]->stream); }
            return merr(m, rc, "device %d: %s", m->devices[r], h->err);
        }
        const int64_t a = m->j0[r], b = m->j1[r];
        if (b > a) {
            if (info) MCU(cudaMemcpyAsync(info + a * S, h->w.info + a * S, sizeof(float) * (b - a) * S, cudaMemcpyDeviceToHost, h->stream));
            if (qcodes) MCU(cudaMemcpyAsync(qcodes + a * S, h->w.q + a * S, sizeof(int32_t) * (b - a) * S, cudaMemcpyDeviceToHost, h->stream));
        }
        MCU(cudaEventRecord(h->ev[5], h->stream));
    }
    memset(&m->tm, 0, sizeof m->tm);
    for (int r = 0; r < m->n; r++) {
        fic_handle *h = m->h[r];
        MCU(cudaSetDevice(m->devices[r]));
        MCU(cudaStreamSynchronize(h->stream));
        collect_timings(h, r == 0);
        if (r != 0) {  // ev[0] is recorded on the first device only: this device's time runs from its pool build
            float ms = 0;
            if (cudaEventElapsedTime(&ms, h->ev[1], h->ev[5]) == cudaSuccess) h->tm.total_ms = ms;
            if (cudaEventElapsedTime(&ms, h->ev[4], h->ev[5]) == cudaSuccess) h->tm.d2h_ms = ms;
        }
        // the handle's view of the call: the slowest device per stage
        const fic_timings &t = h->tm;
        m->tm.h2d_ms = fmaxf(m->tm.h2d_ms, t.h2d_ms);
        m->tm.pool_ms = fmaxf(m->tm.pool_ms, t.pool_ms);
        m->tm.search_ms = fmaxf(m->tm.search_ms, t.search_ms);
        m->tm.kernel_ms = fmaxf(m->tm.kernel_ms, t.kernel_ms);
        m->tm.solve_ms = fmaxf(m->tm.solve_ms, t.solve_ms);
        m->tm.d2h_ms = fmaxf(m->tm.d2h_ms, t.d2h_ms);
        m->tm.total_ms = fmaxf(m->tm.total_ms, t.total_ms);
        m->tm.engine = t.engine;
        m->tm.launches += t.launches;
        m->tm.search_evals += t.search_evals;
    }
#undef MCU
    return FIC_OK;
}

extern "C" {

int fic_create_multi(const int *devices, int n_devices, fic_multi **out)
{
    if (!out) return merr(nullptr, FIC_E_ARG, "fic_create_multi: out is NULL");
    *out = nullptr;
    if (!devices || n_devices < 1 || n_devices > kMaxDevices) return merr(nullptr, FIC_E_ARG, "fic_create_multi: need 1..%d devices", kMaxDevices);
    for (int a = 0; a < n_devices; a++)
        for (int b = a + 1; b < n_devices; b++)
            if (devices[a] == devices[b]) return merr(nullptr, FIC_E_ARG, "fic_create_multi: device %d listed twice", devices[a]);
    fic_multi *m = new (std::nothrow) fic_multi();
    if (!m) return merr(nullptr, FIC_E_NOMEM, "out of host memory");
    m->err[0] = 0;
    memset(&m->tm, 0, sizeof m->tm);
    m->n = n_devices;
    for (int r = 0; r < n_devices; r++) {
        m->devices[r] = devices[r];
        int rc = fic_create(devices[r], &m->h[r]);
        if (rc) {
            merr(nullptr, rc, "device %d: %s", devices[r], fic_last_error(nullptr));
            fic_destroy_multi(m);
            return rc;
        }
    }
    if (n_devices > 1) {
        if (!g_nccl.load(g_multi_err, sizeof g_multi_err)) {
            fic_destroy_multi(m);
            return FIC_E_CUDA;
        }
        int nrc = g_nccl.CommInitAll(m->comm, n_devices, m->devices);
        if (nrc) {
            merr(nullptr, FIC_E_CUDA, "ncclCommInitAll over %d devices failed: %s", n_devices, g_nccl.GetErrorString(nrc));
            fic_destroy_multi(m);
            return FIC_E_CUDA;
        }
        m->has_comm = true;
    }
    *out = m;
    return FIC_OK;
}

void fic_destroy_multi(fic_multi *m)
{
    if (!m) return;
    for (int r = 0; r < m->n; r++) {
        if (m->h[r]) {
            cudaSetDevice(m->devices[r]);
            cudaStreamSynchronize(m->h[r]->stream);
        }
    }
    if (m->has_comm)
        for (int r = 0; r < m->n; r++)
            if (m->comm[r]) g_nccl.CommDestroy(m->comm[r]);
    for (int r = 0; r < m->n; r++) fic_destroy(m->h[r]);
    delete m;
}

const char *fic_multi_last_error(const fic_multi *m) { return m ? m->err : g_multi_err; }
int fic_multi_device_count(const fic_multi *m) { return m ? m->n : 0; }
fic_handle *fic_multi_handle(fic_multi *m, int rank) { return (m && rank >= 0 && rank < m->n) ? m->h[rank] : nullptr; }

int fic_multi_set_option(fic_multi *m, int option, int value)
{
    if (!m) return FIC_E_ARG;
    for (int r = 0; r < m->n; r++) {
        int rc = fic_set_option(m->h[r], option, value);
        if (rc) return merr(m, rc, "%s", m->h[r]->err);
    }
    return FIC_OK;
}

int fic_multi_get_timings(const fic_multi *m, int rank, fic_timings *out)
{
    if (!m || !out || rank >= m->n) return FIC_E_ARG;
    *out = rank < 0 ? m->tm : m->h[rank]->tm;
    return FIC_OK;
}

int fic_multi_range_slice(const fic_multi *m, int rank, int64_t *range_begin, int64_t *range_end)
{
    if (!m || rank < 0 || rank >= m->n) return FIC_E_ARG;
    if (range_begin) *range_begin = m->j0[rank];
    if (range_end) *range_end = m->j1[rank];
    return FIC_OK;
}

int fic_multi_encode_grey(fic_multi *m, const int32_t *argb, int W, int H, int B, int wk, float *info, int32_t *qcodes)
{
    return multi_encode(m, FIC_MODE_GREY, argb, 0, W, H, B, wk, info, qcodes);
}
int fic_multi_encode_rgb(fic_multi *m, const int32_t *argb, int W, int H, int B, int wk, float *info, int32_t *qcodes)
{
    return multi_encode(m, FIC_MODE_RGB, argb, 0, W, H, B, wk, info, qcodes);
}
int fic_multi_encode_grey_iso(fic_multi *m, const int32_t *argb, int W, int H, int B, int wk, float *info, int32_t *qcodes)
{
    return multi_encode(m, FIC_MODE_GREY_ISO, argb, 0, W, H, B, wk, info, qcodes);
}
int fic_multi_encode_grey_u8(fic_multi *m, const uint8_t *plane, int W, int H, int B, int wk, float *info, int32_t *qcodes)
{
    return multi_encode(m, FIC_MODE_GREY, plane, 1, W, H, B, wk, info, qcodes);
}
int fic_multi_encode_rgb_planes(fic_multi *m, const uint8_t *planes, int W, int H, int B, int wk, float *info, int32_t *qcodes)
{
    return multi_encode(m, FIC_MODE_RGB, planes, 1, W, H, B, wk, info, qcodes);
}

}  // extern "C"

extern "C" {

// ------------------------------------------------------------------------------------
// .run stream helpers (host only; DataOutputStream.writeInt is big endian)
// ------------------------------------------------------------------------------------
static void put_be32(uint8_t *p, int32_t v)
{
    uint32_t u = (uint32_t)v;
    p[0] = (uint8_t)(u >> 24); p[1] = (uint8_t)(u >> 16); p[2] = (uint8_t)(u >> 8); p[3] = (uint8_t)u;
}
static int32_t get_be32(const uint8_t *p)
{
    return (int32_t)(((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3]);
}

size_t fic_stream_size(int is_rgb, int W, int H, int B)
{
    if (B <= 0 || W <= 0 || H <= 0) return 0;
    const size_t per_range = is_rgb == FIC_MODE_GREY_ISO ? 16 : (is_rgb ? 20 : 12);
    return 20 + per_range * (size_t)(W / B) * (size_t)(H / B);
}

int fic_stream_write(int is_rgb, int W, int H, int B, int wk, const int32_t *qcodes, uint8_t *out, size_t out_bytes)
{
    size_t need = fic_stream_size(is_rgb, W, H, B);
    if (!qcodes || !out || need == 0 || out_bytes < need) return FIC_E_ARG;
    put_be32(out, is_rgb == FIC_MODE_GREY_ISO ? 2 : (is_rgb ? 1 : 0));  // FC:234-238; 2 = isometry extension
    put_be32(out + 4, W);
    put_be32(out + 8, H);
    put_be32(out + 12, B);
    put_be32(out + 16, wk);
    size_t n = (need - 20) / 4;
    for (size_t i = 0; i < n; i++) put_be32(out + 20 + 4 * i, qcodes[i]);
    return FIC_OK;
}

int fic_stream_read_header(const uint8_t *stream, size_t nbytes, int *is_rgb, int *W, int *H, int *B, int *wk,
                           size_t *qcodes_off)
{
    if (!stream || nbytes < 20) return FIC_E_STREAM;
    // FC:548-552: 0 -> grey, anything else -> RGB; this library's isometry extension writes 2
    int rgb = get_be32(stream) == 2 ? FIC_MODE_GREY_ISO : (get_be32(stream) != 0);
    int w = get_be32(stream + 4), hh = get_be32(stream + 8), b = get_be32(stream + 12), k = get_be32(stream + 16);
    Geom g;
    if (make_geom(w, hh, b, k, rgb, &g, nullptr)) return FIC_E_STREAM;
    if (nbytes < fic_stream_size(rgb, w, hh, b)) return FIC_E_STREAM;
    if (is_rgb) *is_rgb = rgb;
    if (W) *W = w;
    if (H) *H = hh;
    if (B) *B = b;
    if (wk) *wk = k;
    if (qcodes_off) *qcodes_off = 20;
    return FIC_OK;
}

int fic_stream_read_codes(const uint8_t *stream, size_t nbytes, int32_t *qcodes)
{
    int rgb, W, H, B, wk;
    size_t off;
    int rc = fic_stream_read_header(stream, nbytes, &rgb, &W, &H, &B, &wk, &off);
    if (rc) return rc;
    if (!qcodes) return FIC_E_ARG;
    size_t n = (fic_stream_size(rgb, W, H, B) - 20) / 4;
    for (size_t i = 0; i < n; i++) qcodes[i] = get_be32(stream + off + 4 * i);
    return FIC_OK;
}

}  // extern "C"
