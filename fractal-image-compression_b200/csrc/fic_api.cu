// fic_api.cu -- the C ABI of libfic_b200.so (see include/fic_b200.h): handle, workspace,
// call sequencing on one CUDA stream, timings, and the .run stream helpers.
#include <math.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

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
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t call_begin = nullptr, call_end = nullptr;  // bracket a whole call (total_ms of encodes and decodes)
    Work w;
    Encoder enc;
    fic_timings tm;
    char err[512];
    bool tm_pending_dev = false;  // fic_encode_planes_dev: tm's stage times are read once its run has completed
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

Status fic::fail(int rc, const char *fmt, ...)
{
    Status st(rc);
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(st.msg, sizeof st.msg, fmt, ap);
    va_end(ap);
    return st;
}

// The handle's error for the Status of an encoder or decoder entry; out_of_pool: the message of a decoder's FIC_E_STREAM
// (a code outside the domain pool), which the decoder leaves to its caller.
static int status_err(fic_handle *h, const Status &st, const char *out_of_pool = "")
{
    return st.rc ? set_err(h, st.rc, "%s", st.msg[0] ? st.msg : out_of_pool) : FIC_OK;
}

#define ENSURE(ptr, slot, bytes)                                             \
    do {                                                                     \
        int rc_ = status_err(h, ensure(h->w, ptr, slot, (size_t)(bytes))); \
        if (rc_) return rc_;                                                 \
    } while (0)

// Every timed entry starts from zeroed timings; a pending read of fic_encode_planes_dev's stage times is dropped.
static void reset_timings(fic_handle *h)
{
    memset(&h->tm, 0, sizeof h->tm);
    h->tm_pending_dev = false;
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
    h->enc.num_sms = prop.multiProcessorCount;
    if ((e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking)) != cudaSuccess) {
        set_err(nullptr, FIC_E_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
        delete h;
        return FIC_E_CUDA;
    }
    h->stream = h->own_stream;
    e = cudaEventCreate(&h->call_begin);
    if (e == cudaSuccess) e = cudaEventCreate(&h->call_end);
    for (cudaEvent_t &ev : h->enc.ev)
        if (e == cudaSuccess) e = cudaEventCreate(&ev);
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
                    w.img, w.dec2, w.dcode, w.perr, w.state, w.dec3, w.replay, w.qt_stream, w.qt_codes, w.qt_err,
                    w.qt_leaf, w.qt_map, w.qt_keys};
    for (void *p : ptrs)
        if (p) cudaFree(p);
    for (cudaEvent_t ev : {h->call_begin, h->call_end})
        if (ev) cudaEventDestroy(ev);
    for (cudaEvent_t ev : h->enc.ev)
        if (ev) cudaEventDestroy(ev);
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
        h->enc.engine_opt = value;
        return FIC_OK;
    }
    if (option == FIC_OPT_UMMA_KIND && value >= FIC_UMMA_KIND_AUTO && value <= FIC_UMMA_KIND_F16) {
        h->enc.umma_kind = value;
        return FIC_OK;
    }
    if (option == FIC_OPT_UMMA_PAIR && value >= FIC_UMMA_PAIR_AUTO && value <= FIC_UMMA_PAIR_ON) {
        h->enc.umma_pair = value;
        return FIC_OK;
    }
    return set_err(h, FIC_E_ARG, "unknown option %d / value %d", option, value);
}

int fic_get_option(fic_handle *h, int option, int *value)
{
    if (!h || !value) return FIC_E_ARG;
    if (option == FIC_OPT_ENGINE) { *value = h->enc.engine_opt; return FIC_OK; }
    if (option == FIC_OPT_UMMA_KIND) { *value = h->enc.umma_kind; return FIC_OK; }
    if (option == FIC_OPT_UMMA_PAIR) { *value = h->enc.umma_pair; return FIC_OK; }
    if (option == FIC_OPT_UMMA_PAIR_USED) { *value = h->enc.pair_used; return FIC_OK; }
    if (option == FIC_OPT_F16_EXACT) {
        if (h->enc.f16_state == 0) {
            CU(cudaSetDevice(h->device));
            if (int rc = status_err(h, f16_selftest(h->enc, h->stream))) return rc;
        }
        *value = h->enc.f16_state > 0;
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

int fic_get_timings(const fic_handle *h, fic_timings *out)
{
    if (!h || !out) return FIC_E_ARG;
    fic_handle *hm = const_cast<fic_handle *>(h);
    if (hm->tm_pending_dev && run_done(hm->enc)) {  // asynchronous device entry: events are final once the run has completed
        read_stages(hm->enc, &hm->tm, nullptr, nullptr);
        hm->tm_pending_dev = false;
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
    reset_timings(h);
    Work &w = h->w;
    cudaStream_t s = h->stream;
    int S = code_stride(g);
    EncodePlan plan;
    if ((rc = status_err(h, plan_encode(h->enc, g, j0, j1, 1, !src_u8, s, &plan)))) return rc;
    if (src_u8) ENSURE(w.src, S_SRC, (size_t)g.C * W * H);
    else ENSURE(w.argb, S_ARGB, sizeof(int32_t) * (size_t)W * H);
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
    CU(cudaEventRecord(h->call_begin, s));
    if (src_u8) CU(cudaMemcpyAsync(w.src, pixels, (size_t)g.C * W * H, cudaMemcpyHostToDevice, s));
    else CU(cudaMemcpyAsync(w.argb, pixels, sizeof(int32_t) * (size_t)W * H, cudaMemcpyHostToDevice, s));
    const void *d_pixels = src_u8 ? (const void *)w.src : (const void *)w.argb;
    if ((rc = status_err(h, run_encode(h->enc, w, g, plan, d_pixels, !src_u8, j0, j1, 1, d_info, d_q, &h->tm, s)))) return rc;
    if (j1 > j0) {
        if (staged) {
            CU(cudaMemcpyAsync(h->h_stage, d_info, 2 * table, cudaMemcpyDeviceToHost, s));
        } else {
            if (info) CU(cudaMemcpyAsync(info + j0 * S, d_info + j0 * S, sizeof(float) * (j1 - j0) * S, cudaMemcpyDeviceToHost, s));
            if (qcodes) CU(cudaMemcpyAsync(qcodes + j0 * S, d_q + j0 * S, sizeof(int32_t) * (j1 - j0) * S, cudaMemcpyDeviceToHost, s));
        }
    }
    CU(cudaEventRecord(h->call_end, s));
    CU(cudaStreamSynchronize(s));
    if (staged && j1 > j0) {
        memcpy(info + j0 * S, h->h_stage + sizeof(float) * j0 * S, sizeof(float) * (j1 - j0) * S);
        memcpy(qcodes + j0 * S, h->h_stage + table + sizeof(int32_t) * j0 * S, sizeof(int32_t) * (j1 - j0) * S);
    }
    read_stages(h->enc, &h->tm, h->call_begin, h->call_end);
    return FIC_OK;
}

// ---- batches of same-size images ----------------------------------------------------------------------------------

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

// A batch encode: the codes of n_images images back to back, [n][NR][S], each equal to a single encode of that image.
// The plan (plan_encode) splits the batch into groups of images that go up in one copy and whose codes come down in one.
// The fused engine covers every range of a group's images in one launch; the tcgen05 engine searches a group as one
// block-diagonal problem -- one launch of each pool, sort, pack, search, refine and solve kernel; the direct engine runs
// the group image by image.
static int encode_batch_host(fic_handle *h, int mode, const void *pixels, int src_u8, int n_images, int W, int H, int B, int wk,
                             float *info, int32_t *qcodes)
{
    if (!h) return FIC_E_ARG;
    if (!pixels || (!info && !qcodes)) return set_err(h, FIC_E_ARG, "the images and at least one of info/qcodes must be non-NULL");
    Geom g;
    int rc = batch_geom(h, mode, n_images, W, H, B, wk, &g);
    if (rc) return rc;
    CU(cudaSetDevice(h->device));
    reset_timings(h);
    Work &w = h->w;
    cudaStream_t s = h->stream;
    EncodePlan plan;
    if ((rc = status_err(h, plan_encode(h->enc, g, 0, g.NR, n_images, !src_u8, s, &plan)))) return rc;
    const int S = code_stride(g), group = plan.group;
    const size_t plane = (size_t)W * H, image_bytes = src_u8 ? g.C * plane : sizeof(int32_t) * plane;
    const size_t codes = (size_t)g.NR * S, table = sizeof(float) * codes;  // one image's code table (float and int32 alike)
    if (src_u8) ENSURE(w.src, S_SRC, image_bytes * group);
    else ENSURE(w.argb, S_ARGB, image_bytes * group);
    ENSURE(w.info, S_INFO, table * group);
    ENSURE(w.q, S_Q, table * group);
    const uint8_t *d_pixels = src_u8 ? w.src : (const uint8_t *)w.argb;
    const bool grouped = plan.engine == FIC_ENGINE_UMMA;
    DrainOnExit drain(s);
    CU(cudaEventRecord(h->call_begin, s));
    for (int i0 = 0; i0 < n_images; i0 += group) {
        const int gn = n_images - i0 < group ? n_images - i0 : group;
        if (grouped && i0 > 0) {  // the previous group's stage events, before this group records them again
            CU(cudaStreamSynchronize(s));
            read_stages(h->enc, &h->tm, nullptr, nullptr);
        }
        CU(cudaMemcpyAsync((void *)d_pixels, (const uint8_t *)pixels + i0 * image_bytes, image_bytes * gn, cudaMemcpyHostToDevice, s));
        const int per_run = plan.engine == FIC_ENGINE_DIRECT ? 1 : gn;
        for (int i = 0; i < gn; i += per_run) {
            rc = status_err(h, run_encode(h->enc, w, g, plan, d_pixels + i * image_bytes, !src_u8, 0, g.NR, per_run,
                                          w.info + i * codes, w.q + i * codes, &h->tm, s));
            if (rc) return rc;
        }
        if (info) CU(cudaMemcpyAsync(info + i0 * codes, w.info, table * gn, cudaMemcpyDeviceToHost, s));
        if (qcodes) CU(cudaMemcpyAsync(qcodes + i0 * codes, w.q, table * gn, cudaMemcpyDeviceToHost, s));
    }
    CU(cudaEventRecord(h->call_end, s));
    CU(cudaStreamSynchronize(s));
    CU(cudaGetLastError());
    if (grouped) read_stages(h->enc, &h->tm, nullptr, nullptr);
    // the per-stage times are the tcgen05 groups' sums (0 on the other engines); total_ms is the whole call
    float ms = 0;
    h->tm.total_ms = cudaEventElapsedTime(&ms, h->call_begin, h->call_end) == cudaSuccess ? ms : 0.0f;
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
    reset_timings(h);
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
    CU(cudaEventRecord(h->call_begin, s));
    int bad = -1;
    const Status st = decode_batch_run(w, g, n_images, group, qcodes, argb_out, planes_out, max_iters, avg_error, iterations,
                                             h->h_stage, h->h_acc, h->call_begin, h->call_end, &h->tm, &bad, s);
    if (st.rc == FIC_E_STREAM)
        return set_err(h, FIC_E_STREAM, "image %d: a code indexes outside the domain pool (the reference would throw ArrayIndexOutOfBounds)", bad);
    return status_err(h, st);
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
    reset_timings(h);
    EncodePlan plan;
    if ((rc = status_err(h, plan_encode(h->enc, g, range_begin, range_end, 1, false, h->stream, &plan)))) return rc;
    rc = status_err(h, run_encode(h->enc, h->w, g, plan, d_planes, false, range_begin, range_end, 1, d_info, d_qcodes, &h->tm, h->stream));
    h->tm_pending_dev = rc == FIC_OK;  // fic_get_timings reads the stage times once the run has completed
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
    double v = measure_mma_peak(h->enc.num_sms, h->stream, 3, kind == FIC_UMMA_KIND_F16, n_cols, &why);
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
    double v = measure_mma_peak_pair(h->enc.num_sms, h->stream, 3, kind == FIC_UMMA_KIND_F16, nullptr, &why);
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
    return status_err(h, decode_float_sum(w, terms, count, carry, h->h_acc, sum, s));
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
    reset_timings(h);
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
    CU(cudaEventRecord(h->call_begin, s));
    if (!d_qcodes) CU(cudaMemcpyAsync(w.q, qcodes, sizeof(int32_t) * g.NR * S, cudaMemcpyHostToDevice, s));
    const Status st = decode_run(w, g, d_qcodes ? d_qcodes : w.q, d_planes_out ? d_planes_out : w.img, argb_out, planes_out,
                                       max_iters, avg_error, iterations, h->h_acc, h->call_begin, h->call_end, &h->tm, s);
    return status_err(h, st, "a code indexes outside the domain pool (the reference would throw ArrayIndexOutOfBounds)");
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
    return status_err(h, collage_run(w, g, argb_out, info, h->h_acc, s), "a code indexes outside the domain pool");
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
        reset_timings(h);
        if (r == 0 && !src_u8 && (rc = status_err(h, ensure(h->w, h->w.argb, S_ARGB, sizeof(int32_t) * (size_t)W * H))))
            return merr(m, rc, "%s", h->err);
        if ((rc = status_err(h, ensure(h->w, h->w.src, S_SRC, plane_bytes))) ||
            (rc = status_err(h, ensure(h->w, h->w.info, S_INFO, sizeof(float) * g.NR * S))) ||
            (rc = status_err(h, ensure(h->w, h->w.q, S_Q, sizeof(int32_t) * g.NR * S))))
            return merr(m, rc, "%s", h->err);
    }
    // one upload, to the first device
    fic_handle *h0 = m->h[0];
    MCU(cudaSetDevice(m->devices[0]));
    MCU(cudaEventRecord(h0->call_begin, h0->stream));
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
        EncodePlan plan;
        rc = status_err(h, plan_encode(h->enc, g, m->j0[r], m->j1[r], 1, false, h->stream, &plan));
        if (!rc)
            rc = status_err(h, run_encode(h->enc, h->w, g, plan, h->w.src, false, m->j0[r], m->j1[r], 1, h->w.info, h->w.q,
                                          &h->tm, h->stream));
        if (rc) {
            for (int q = 0; q < m->n; q++) { cudaSetDevice(m->devices[q]); cudaStreamSynchronize(m->h[q]->stream); }
            return merr(m, rc, "device %d: %s", m->devices[r], h->err);
        }
        const int64_t a = m->j0[r], b = m->j1[r];
        if (b > a) {
            if (info) MCU(cudaMemcpyAsync(info + a * S, h->w.info + a * S, sizeof(float) * (b - a) * S, cudaMemcpyDeviceToHost, h->stream));
            if (qcodes) MCU(cudaMemcpyAsync(qcodes + a * S, h->w.q + a * S, sizeof(int32_t) * (b - a) * S, cudaMemcpyDeviceToHost, h->stream));
        }
        MCU(cudaEventRecord(h->call_end, h->stream));
    }
    memset(&m->tm, 0, sizeof m->tm);
    for (int r = 0; r < m->n; r++) {
        fic_handle *h = m->h[r];
        MCU(cudaSetDevice(m->devices[r]));
        MCU(cudaStreamSynchronize(h->stream));
        // the call's start event is recorded on the first device only: the other devices' times run from their pool build
        read_stages(h->enc, &h->tm, r == 0 ? h->call_begin : nullptr, h->call_end);
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

// ---- quadtree extension (FIC_MODE_GREY_QT, FIC_MODE_RGB_QT) ---------------------------------------------------------
// One body per entry for both modes: the mode decides the channel count (the level encodes, the planes in and out) and,
// inside qt_geom / qt_parse, the header value and the leaf size.

// Budget form's side of h_stage: the first leaves take its first kDecodeBatchMax words, the allowed splits (int64) and the
// qt_err head (the leaf total, a spare word and a double per image) follow.
constexpr size_t kQtStageSplits = sizeof(uint32_t) * kDecodeBatchMax, kQtStageHead = kQtStageSplits + sizeof(int64_t) * kDecodeBatchMax;
static_assert(kQtStageHead + sizeof(uint32_t) * (2 + 2 * kDecodeBatchMax) <= kStageBytes, "a group's budget words fit h_stage");

// Images go up and their streams come down in groups; a group is at most the smallest group any level's plan allows (so
// every level's run fits its engine's bounds) and at most kDecodeBatchMax images (one grid row and one leaf start of
// h_stage each).  Per group: one upload, then every level's ordinary grey or RGB batch run (the engine fic_encode_batch_u8
// would pick, into that level's [n][NR_L] code table; the direct engine image by image), one decimation of the sources for
// the collage errors, and the stream bodies built on the device (launch_qt_stream).  The leaf counts come down in one
// small copy, then the bodies in one copy with the caller's stride as pitch.  A single image is the group of one.
// Budget form (max_bytes non-NULL, one per image): every image's allowed splits go up with its pixels, its max_mse is
// chosen on the device (launch_qt_stream) and comes down with the leaf total into out_mse[i]; an infeasible budget fails
// the call before any device work.
static int encode_quadtree(fic_handle *h, int mode, const uint8_t *planes, int n_images, int W, int H, int b_max, int b_min,
                           int wk, double max_mse, uint8_t *streams, size_t stride, size_t *stream_bytes,
                           const size_t *max_bytes = nullptr, double *out_mse = nullptr)
{
    const bool budget = max_bytes != nullptr;
    if (!budget && max_mse != max_mse) return set_err(h, FIC_E_ARG, "max_mse is NaN");
    QtGeom q;
    const char *why = "";
    int rc = qt_geom(mode, W, H, b_max, b_min, wk, &q, &why);
    if (rc) return set_err(h, rc, "%s", why);
    if (budget) {
        int low = -1;  // the lowest image whose budget is below the unsplit tree
        for (int i = 0; i < n_images; i++)
            if (qt_budget_splits(q, max_bytes[i]) < 0 && low < 0) low = i;
        if (low >= 0) {
            const size_t least = kQtHeaderBytes + (size_t)q.flag_bytes + qt_leaf_bytes(q) * (size_t)q.g[0].NR;
            for (int i = 0; i < n_images; i++) {
                stream_bytes[i] = least;
                out_mse[i] = INFINITY;
            }
            if (n_images == 1) return set_err(h, FIC_E_ARG, "max_bytes = %zu is below the unsplit tree's %zu bytes", max_bytes[0], least);
            return set_err(h, FIC_E_ARG, "image %d: max_bytes = %zu is below the unsplit tree's %zu bytes", low, max_bytes[low], least);
        }
    }
    const Geom &fine = q.g[q.nl - 1];
    const size_t C = (size_t)fine.C, S = (size_t)code_stride(fine), image_bytes = C * W * H, body = qt_body_bytes(q);
    size_t bytes;
    if (__builtin_mul_overflow((size_t)n_images, image_bytes, &bytes) || __builtin_mul_overflow((size_t)n_images, stride, &bytes))
        return set_err(h, FIC_E_ARG, "n_images = %d images of %d x %d overflow a byte count", n_images, W, H);
    CU(cudaSetDevice(h->device));
    reset_timings(h);
    Work &w = h->w;
    cudaStream_t s = h->stream;
    EncodePlan plan[kQtMaxLevels];
    int group = n_images < kDecodeBatchMax ? n_images : kDecodeBatchMax;
    for (int L = 0; L < q.nl; L++) {
        if ((rc = status_err(h, plan_encode(h->enc, q.g[L], 0, q.g[L].NR, n_images, false, s, &plan[L])))) return rc;
        if (plan[L].group < group) group = plan[L].group;
    }
    ENSURE(w.src, S_SRC, image_bytes * group);
    ENSURE(w.dec, S_DEC, C * fine.sw * fine.sh * group);
    ENSURE(w.info, S_INFO, sizeof(float) * S * fine.NR * group);
    ENSURE(w.qt_codes, S_QT_CODES, sizeof(int32_t) * S * q.codes * group);
    ENSURE(w.qt_err, S_QT_ERR, sizeof(uint32_t) * qt_err_words(q, group));
    ENSURE(w.qt_stream, S_QT_STREAM, body * group);
    if (budget) ENSURE(w.qt_keys, S_QT_KEYS, (sizeof(int64_t) + sizeof(uint32_t) * qt_nodes(q)) * group);
    const uint32_t *starts = (const uint32_t *)h->h_stage;
    // budget form: the allowed splits go up from, and the qt_err head comes down to, h_stage past the first leaves
    int64_t *h_splits = (int64_t *)(h->h_stage + kQtStageSplits);
    const uint32_t *head = budget ? (const uint32_t *)(h->h_stage + kQtStageHead) : (const uint32_t *)h->h_acc;
    int too_long = -1;  // the lowest image whose stream does not fit
    DrainOnExit drain(s);
    CU(cudaEventRecord(h->call_begin, s));
    for (int i0 = 0; i0 < n_images; i0 += group) {
        const int gn = n_images - i0 < group ? n_images - i0 : group;
        CU(cudaMemcpyAsync(w.src, planes + i0 * image_bytes, image_bytes * gn, cudaMemcpyHostToDevice, s));
        if (budget) {
            for (int i = 0; i < gn; i++) h_splits[i] = qt_budget_splits(q, max_bytes[i0 + i]);
            CU(cudaMemcpyAsync(w.qt_keys, h_splits, sizeof(int64_t) * gn, cudaMemcpyHostToDevice, s));
        }
        for (int L = 0; L < q.nl; L++) {
            const Geom &g = q.g[L];
            const int per_run = plan[L].engine == FIC_ENGINE_DIRECT ? 1 : gn;
            for (int i = 0; i < gn; i += per_run) {
                rc = status_err(h, run_encode(h->enc, w, g, plan[L], w.src + i * image_bytes, false, 0, g.NR, per_run, w.info,
                                              w.qt_codes + S * (q.first[L] * gn + i * g.NR), &h->tm, s));
                if (rc) return rc;
                CU(cudaStreamSynchronize(s));  // the run's stage events, before the next run records them again
                read_stages(h->enc, &h->tm, nullptr, nullptr);
            }
        }
        h->tm.launches += launch_decimate(w.src, w.dec, fine, s, gn);  // the fused engine leaves no decimated plane behind
        h->tm.launches += launch_qt_stream(w, q, gn, max_mse, budget, s);
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync((void *)head, w.qt_err, sizeof(uint32_t) * (budget ? qt_head_words(gn) : 1), cudaMemcpyDeviceToHost, s));
        if (gn > 1)  // every image's first leaf: the first of its warp totals after the group's scan
            CU(cudaMemcpy2DAsync(h->h_stage, sizeof(uint32_t), w.qt_err + qt_starts_at(q, gn), sizeof(uint32_t) * ((q.flag_bytes + 31) / 32),
                                 sizeof(uint32_t), gn, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        const uint32_t total = head[0];
        if (budget) memcpy(out_mse + i0, head + 2, sizeof(double) * gn);
        size_t longest = 0;
        for (int i = 0; i < gn; i++) {
            const int64_t leaves = (i + 1 < gn ? starts[i + 1] : total) - (gn > 1 ? starts[i] : 0);
            const size_t need = kQtHeaderBytes + (size_t)q.flag_bytes + qt_leaf_bytes(q) * (size_t)leaves;
            stream_bytes[i0 + i] = need;
            if ((!streams || need > stride) && too_long < 0) too_long = i0 + i;
            if (need > longest) longest = need;
            if (too_long < 0) {
                const int32_t hd[8] = {mode, W, H, 0, wk, b_max, b_min, (int32_t)leaves};
                for (int k = 0; k < 8; k++) put_be32(streams + (i0 + i) * stride + 4 * k, hd[k]);
            }
        }
        if (too_long >= 0) continue;
        if (gn == 1) CU(cudaMemcpyAsync(streams + i0 * stride + kQtHeaderBytes, w.qt_stream, longest - kQtHeaderBytes, cudaMemcpyDeviceToHost, s));
        else CU(cudaMemcpy2DAsync(streams + i0 * stride + kQtHeaderBytes, stride, w.qt_stream, body, longest - kQtHeaderBytes, gn,
                                  cudaMemcpyDeviceToHost, s));
    }
    CU(cudaEventRecord(h->call_end, s));
    CU(cudaStreamSynchronize(s));
    float ms = 0;
    h->tm.total_ms = cudaEventElapsedTime(&ms, h->call_begin, h->call_end) == cudaSuccess ? ms : 0.0f;  // the whole call
    if (too_long >= 0) {
        if (n_images == 1) return set_err(h, FIC_E_ARG, "the stream needs %zu bytes, capacity is %zu", stream_bytes[0], stride);
        return set_err(h, FIC_E_ARG, "image %d: the stream needs %zu bytes, stride is %zu", too_long, stream_bytes[too_long], stride);
    }
    return FIC_OK;
}

static int quadtree_stream_info(int mode, const uint8_t *stream, size_t nbytes, int *W, int *H, int *b_max, int *b_min,
                                int *wk, int64_t *n_leaves)
{
    QtGeom q;
    const char *why = "";
    int rc = qt_parse(mode, stream, nbytes, &q, nullptr, true, &why);
    if (rc) return rc;
    if (W) *W = q.g[0].W;
    if (H) *H = q.g[0].H;
    if (b_max) *b_max = q.g[0].B;
    if (b_min) *b_min = q.g[q.nl - 1].B;
    if (wk) *wk = q.wk;
    if (n_leaves) *n_leaves = q.leaves;
    return FIC_OK;
}

// Image and plane workspace (img, dec, dec2) one decode group holds at most; a group is also at most kDecodeBatchMax
// images (their state blocks come back through h_stage).
constexpr size_t kQtDecodeGroupBytes = (size_t)256 << 20;

// Every stream is parsed (the lowest bad image is named) and must share stream 0's geometry.  Per group of images: the
// flag bytes and then the leaves of every image packed into one upload (a single image's body as it is), the first-leaf
// tables (counted over the group) in another, then decode_quadtree_run.
static int decode_quadtree(fic_handle *h, int mode, int n_images, const uint8_t *streams, size_t stride, const size_t *nbytes,
                           int max_iters, uint8_t *planes_out, float *avg_error, int *iterations)
{
    if (max_iters < 1) return set_err(h, FIC_E_ARG, "max_iters must be >= 1");
    const bool one = n_images == 1;
    QtGeom q;
    const char *why = "";
    std::vector<int64_t> leaves((size_t)n_images);
    for (int i = 0; i < n_images; i++) {
        QtGeom qi;
        const int rc = qt_parse(mode, streams + i * stride, nbytes[i], &qi, nullptr, false, &why);
        if (rc) return one ? set_err(h, rc, "%s", why) : set_err(h, rc, "image %d: %s", i, why);
        if (i == 0) q = qi;
        else if (qi.g[0].W != q.g[0].W || qi.g[0].H != q.g[0].H || qi.g[0].B != q.g[0].B || qi.nl != q.nl || qi.wk != q.wk)
            return set_err(h, FIC_E_STREAM, "image %d: W, H, b_max, b_min or wk differ from image 0's", i);
        leaves[i] = qi.leaves;
    }
    const Geom &g = q.g[0];
    const size_t C = (size_t)g.C, plane = (size_t)g.W * g.H, bmin = (size_t)q.g[q.nl - 1].B, leaf_bytes = qt_leaf_bytes(q);
    const size_t cells = plane / (bmin * bmin), ntop = (size_t)g.NR, flags = (size_t)q.flag_bytes;
    const size_t per_image = C * (plane + 2 * (size_t)g.sw * g.sh);
    size_t bytes;
    if (__builtin_mul_overflow((size_t)n_images, C * plane, &bytes))
        return set_err(h, FIC_E_ARG, "n_images = %d images of %d x %d overflow a byte count", n_images, g.W, g.H);
    size_t fit = kQtDecodeGroupBytes / per_image;
    fit = fit < 1 ? 1 : (fit > (size_t)kDecodeBatchMax ? (size_t)kDecodeBatchMax : fit);
    const int group = (size_t)n_images < fit ? n_images : (int)fit;
    int64_t most = 0;  // the most leaves of a group
    for (int i0 = 0; i0 < n_images; i0 += group) {
        int64_t sum = 0;
        for (int i = i0; i < n_images && i < i0 + group; i++) sum += leaves[i];
        if (sum > most) most = sum;
    }
    CU(cudaSetDevice(h->device));
    reset_timings(h);
    Work &w = h->w;
    cudaStream_t s = h->stream;
    ENSURE(w.img, S_IMG, C * plane * group);
    ENSURE(w.dec, S_DEC, C * g.sw * g.sh * group);
    ENSURE(w.dec2, S_DEC2, C * g.sw * g.sh * group);
    ENSURE(w.state, S_STATE, sizeof(DecodeState) * group);
    ENSURE(w.qt_stream, S_QT_STREAM, flags * group + leaf_bytes * most);
    ENSURE(w.qt_leaf, S_QT_LEAF, sizeof(int4) * (C == 3 ? 2 : 1) * most);  // k_qt_dequant's records
    ENSURE(w.qt_map, S_QT_MAP, sizeof(int32_t) * (cells + ntop) * group);
    std::vector<int32_t> base(ntop * group);  // every image's first leaf of each top block, counted over its group
    std::vector<uint8_t> pack(one ? 0 : flags * group + leaf_bytes * most);
    DrainOnExit drain(s);
    CU(cudaEventRecord(h->call_begin, s));
    for (int i0 = 0; i0 < n_images; i0 += group) {
        const int gn = n_images - i0 < group ? n_images - i0 : group;
        int64_t first = 0;
        for (int i = 0; i < gn; i++) {
            const uint8_t *si = streams + (i0 + i) * stride;
            QtGeom qi;
            qt_parse(mode, si, nbytes[i0 + i], &qi, base.data() + i * ntop, false, &why);
            for (size_t t = 0; t < ntop; t++) base[i * ntop + t] += (int32_t)first;
            if (!one) {
                memcpy(pack.data() + i * flags, si + kQtHeaderBytes, flags);
                memcpy(pack.data() + gn * flags + leaf_bytes * first, si + kQtHeaderBytes + flags, leaf_bytes * qi.leaves);
            }
            first += qi.leaves;
        }
        const uint8_t *body = one ? streams + kQtHeaderBytes : pack.data();
        CU(cudaMemcpyAsync(w.qt_stream, body, flags * gn + leaf_bytes * first, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(w.qt_map + cells * gn, base.data(), sizeof(int32_t) * ntop * gn, cudaMemcpyHostToDevice, s));
        int bad = 0;
        const Status st = decode_quadtree_run(w, q, gn, max_iters, planes_out + i0 * C * plane, avg_error ? avg_error + i0 : nullptr,
                                              iterations ? iterations + i0 : nullptr, h->h_stage, h->call_begin, h->call_end, &h->tm, &bad, s);
        if (st.rc == FIC_E_STREAM && !one)
            return set_err(h, FIC_E_STREAM, "image %d: a leaf indexes outside its level's domain pool", i0 + bad);
        if (st.rc) return status_err(h, st, "a leaf indexes outside its level's domain pool");
    }
    return FIC_OK;
}

size_t fic_quadtree_stream_bound(int W, int H, int b_max, int b_min) { return qt_stream_bound(FIC_MODE_GREY_QT, W, H, b_max, b_min); }

int fic_encode_quadtree(fic_handle *h, const uint8_t *plane, int W, int H, int b_max, int b_min, int wk, double max_mse,
                        uint8_t *stream, size_t capacity, size_t *stream_bytes)
{
    if (!h) return FIC_E_ARG;
    if (!plane || !stream_bytes) return set_err(h, FIC_E_ARG, "plane and stream_bytes must be non-NULL");
    return encode_quadtree(h, FIC_MODE_GREY_QT, plane, 1, W, H, b_max, b_min, wk, max_mse, stream, capacity, stream_bytes);
}

int fic_quadtree_stream_info(const uint8_t *stream, size_t nbytes, int *W, int *H, int *b_max, int *b_min, int *wk,
                             int64_t *n_leaves)
{
    return quadtree_stream_info(FIC_MODE_GREY_QT, stream, nbytes, W, H, b_max, b_min, wk, n_leaves);
}

int fic_decode_quadtree(fic_handle *h, const uint8_t *stream, size_t nbytes, int max_iters, uint8_t *plane_out,
                        float *avg_error, int *iterations)
{
    if (!h) return FIC_E_ARG;
    if (!stream || !plane_out) return set_err(h, FIC_E_ARG, "stream and plane_out must be non-NULL");
    return decode_quadtree(h, FIC_MODE_GREY_QT, 1, stream, 0, &nbytes, max_iters, plane_out, avg_error, iterations);
}

size_t fic_quadtree_rgb_stream_bound(int W, int H, int b_max, int b_min) { return qt_stream_bound(FIC_MODE_RGB_QT, W, H, b_max, b_min); }

int fic_encode_quadtree_rgb(fic_handle *h, const uint8_t *planes, int W, int H, int b_max, int b_min, int wk,
                            double max_mse, uint8_t *stream, size_t capacity, size_t *stream_bytes)
{
    if (!h) return FIC_E_ARG;
    if (!planes || !stream_bytes) return set_err(h, FIC_E_ARG, "planes and stream_bytes must be non-NULL");
    return encode_quadtree(h, FIC_MODE_RGB_QT, planes, 1, W, H, b_max, b_min, wk, max_mse, stream, capacity, stream_bytes);
}

int fic_quadtree_rgb_stream_info(const uint8_t *stream, size_t nbytes, int *W, int *H, int *b_max, int *b_min, int *wk,
                                 int64_t *n_leaves)
{
    return quadtree_stream_info(FIC_MODE_RGB_QT, stream, nbytes, W, H, b_max, b_min, wk, n_leaves);
}

int fic_decode_quadtree_rgb(fic_handle *h, const uint8_t *stream, size_t nbytes, int max_iters, uint8_t *planes_out,
                            float *avg_error, int *iterations)
{
    if (!h) return FIC_E_ARG;
    if (!stream || !planes_out) return set_err(h, FIC_E_ARG, "stream and planes_out must be non-NULL");
    return decode_quadtree(h, FIC_MODE_RGB_QT, 1, stream, 0, &nbytes, max_iters, planes_out, avg_error, iterations);
}

int fic_encode_quadtree_batch(fic_handle *h, int mode, const uint8_t *planes, int n_images, int W, int H, int b_max, int b_min,
                              int wk, double max_mse, uint8_t *streams, size_t stride, size_t *stream_bytes)
{
    if (!h) return FIC_E_ARG;
    if (n_images < 1) return set_err(h, FIC_E_ARG, "n_images must be >= 1");
    if (!planes || !streams || !stream_bytes) return set_err(h, FIC_E_ARG, "planes, streams and stream_bytes must be non-NULL");
    return encode_quadtree(h, mode, planes, n_images, W, H, b_max, b_min, wk, max_mse, streams, stride, stream_bytes);
}

int fic_encode_quadtree_budget(fic_handle *h, int mode, const uint8_t *planes, int W, int H, int b_max, int b_min, int wk,
                               size_t max_bytes, uint8_t *stream, size_t capacity, size_t *stream_bytes, double *max_mse)
{
    if (!h) return FIC_E_ARG;
    if (!planes || !stream_bytes || !max_mse) return set_err(h, FIC_E_ARG, "planes, stream_bytes and max_mse must be non-NULL");
    return encode_quadtree(h, mode, planes, 1, W, H, b_max, b_min, wk, 0.0, stream, capacity, stream_bytes, &max_bytes, max_mse);
}

int fic_encode_quadtree_budget_batch(fic_handle *h, int mode, const uint8_t *planes, int n_images, int W, int H, int b_max,
                                     int b_min, int wk, const size_t *max_bytes, uint8_t *streams, size_t stride,
                                     size_t *stream_bytes, double *max_mse)
{
    if (!h) return FIC_E_ARG;
    if (n_images < 1) return set_err(h, FIC_E_ARG, "n_images must be >= 1");
    if (!planes || !max_bytes || !streams || !stream_bytes || !max_mse)
        return set_err(h, FIC_E_ARG, "planes, max_bytes, streams, stream_bytes and max_mse must be non-NULL");
    return encode_quadtree(h, mode, planes, n_images, W, H, b_max, b_min, wk, 0.0, streams, stride, stream_bytes, max_bytes, max_mse);
}

int fic_decode_quadtree_batch(fic_handle *h, int mode, int n_images, const uint8_t *streams, size_t stride, const size_t *nbytes,
                              int max_iters, uint8_t *planes_out, float *avg_error, int *iterations)
{
    if (!h) return FIC_E_ARG;
    if (mode != FIC_MODE_GREY_QT && mode != FIC_MODE_RGB_QT) return set_err(h, FIC_E_ARG, "mode must be FIC_MODE_GREY_QT or FIC_MODE_RGB_QT");
    if (n_images < 1) return set_err(h, FIC_E_ARG, "n_images must be >= 1");
    if (!streams || !nbytes || !planes_out) return set_err(h, FIC_E_ARG, "streams, nbytes and planes_out must be non-NULL");
    size_t bytes;
    if (__builtin_mul_overflow((size_t)n_images, stride, &bytes)) return set_err(h, FIC_E_ARG, "n_images * stride overflows");
    return decode_quadtree(h, mode, n_images, streams, stride, nbytes, max_iters, planes_out, avg_error, iterations);
}

}  // extern "C"
