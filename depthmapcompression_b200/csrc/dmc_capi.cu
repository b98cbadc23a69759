// dmc_capi.cu -- the C ABI of libdmc_b200.so (include/dmc_c.h): context, host<->device staging, the dispatch
// rules of the reference's operators (which (type, method) pairs run, which are silent no-ops), the four
// PostFilterSet chains, and the frame-batch streaming executor.  No CPU fallback exists anywhere in this file.
#include "../../include/dmc_c.h"
#include "dmc_common.cuh"
#include "dmc_jpeg_enc_core.h"
#include "dmc_kernels.cuh"

#include <limits.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <thread>
#include <vector>

using namespace dmc;

namespace {

constexpr int kSlots = 4;        // streaming pipeline depth (H2D / kernels / D2H of different chunks overlap)

// Device buffers of a slot: the chain's staged input and output, ping-pong frames and float scratch (single-image operators
// stage extra images there too); JPEG bitstreams, metadata block (JpegGroup), de-stuffed scans, restart-stream coefficients.
enum { SB_IN, SB_OUT, SB_PING, SB_PONG, SB_FLOAT, SB_BITS, SB_META, SB_SCANS, SB_COEF, SB_COUNT };
// Device buffers of dmc_jpeg_decode_gray_batch.
enum { JD_BITS, JD_META, JD_SCANS, JD_COEF, JD_OUT, JD_COUNT };

struct Buf { void* p = nullptr; size_t cap = 0; };

struct Slot {
    Buf buf[SB_COUNT];
    cudaStream_t stream = nullptr;
    // pinned host staging for per-chunk metadata that is built on the host (JPEG descriptors and tables), and the event
    // after which the chunk that used it last is completely done
    void* hstage = nullptr; size_t hcap = 0; cudaEvent_t done = nullptr; bool done_pending = false;
};

}  // namespace

struct dmc_ctx {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    Slot slot[kSlots];
    std::string err;
    uint64_t launches = 0;
    float* xtab = nullptr; int xtab_w = 0; double xtab_f = 0;    // reprojectXYZ column table cache
    // host-link gateway (dmc_set_gateway): host traffic of the batch entry points runs over another device's link; that
    // device holds the staging buffers, this context's kernels reach them through NVLink peer access
    struct Gateway { int device = -1; cudaStream_t stream[kSlots] = {}; Buf in[kSlots], out[kSlots]; cudaEvent_t ev_in[kSlots] = {}, ev_out[kSlots] = {}, ev_done[kSlots] = {}; } gw;
    Buf render[2]; int* render_flag = nullptr;      // point-cloud render: attempt lists etc., device flag; pinned host flag
    Buf jpeg[JD_COUNT];
    Buf jpeg_enc[9];             // JPEG encode: tables, staged frames, coefficients, block records, scan words, slots, lengths + offsets, staged output, decoder tables + descriptors
    // optional per-stage CUDA-event timing of the chain (bench.py's live roofline measurement)
    int lanes = 1;               // concurrent frame groups in the device-resident batch path
    int profile_mask = 0;
    struct ProfRec { cudaEvent_t a, b; int stage; uint64_t pixels; };
    std::vector<ProfRec> prof_pending;
    std::vector<cudaEvent_t> prof_free;
    // CUDA graph of the single-frame chain for repeated identical device-resident calls (batch-1 latency, SURVEY 7.1-6):
    // captured the second time a (pointers, shape, parameters, stream) key is seen, replayed afterwards; dropped whenever
    // a scratch buffer is reallocated (alloc_epoch) because the kernels' scratch pointers are baked into the graph.
    struct GraphKey { const void* in; void* out; int rows, cols; dmc_chain_params p; cudaStream_t stream; };
    GraphKey graph_key, graph_seen; bool graph_valid = false, graph_seen_valid = false, graphs_off = false;
    cudaGraphExec_t graph_exec = nullptr; uint64_t graph_epoch = 0, alloc_epoch = 0, graph_launches = 0, graph_replays = 0;
    double prof_ms[DMC_STAGE_COUNT] = {0, 0, 0, 0};
    uint64_t prof_launches[DMC_STAGE_COUNT] = {0, 0, 0, 0}, prof_pixels[DMC_STAGE_COUNT] = {0, 0, 0, 0};
};

static thread_local std::string g_err;

namespace {

int fail(dmc_ctx* ctx, int code, const std::string& msg) {
    if (ctx) ctx->err = msg; else g_err = msg;
    return code;
}
#define CUDA_TRY(ctx, expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) return fail(ctx, DMC_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); } while (0)

size_t depth_size(int depth) { static const size_t s[8] = {1, 1, 2, 2, 4, 4, 8, 2}; return s[depth & 7]; }
int cv_depth(int t) { return t & 7; }
int cv_cn(int t) { return ((t >> 3) & 511) + 1; }
size_t elem_size(int t) { return depth_size(cv_depth(t)) * cv_cn(t); }
size_t dense_step(const dmc_image* im) { return (size_t)im->cols * elem_size(im->cvtype); }
size_t step_of(const dmc_image* im) { return im->step ? im->step : dense_step(im); }
size_t image_bytes(const dmc_image* im) { return dense_step(im) * (size_t)im->rows; }

int check_image(dmc_ctx* ctx, const dmc_image* im, const char* what) {
    if (!im || !im->data) return fail(ctx, DMC_ERR_SIZE, std::string(what) + ": null image");
    if (im->rows <= 0 || im->cols <= 0) return fail(ctx, DMC_ERR_SIZE, std::string(what) + ": empty image");
    if (im->step && im->step < dense_step(im)) return fail(ctx, DMC_ERR_SIZE, std::string(what) + ": step smaller than a row");
    if (im->mem != DMC_MEM_HOST && im->mem != DMC_MEM_DEVICE) return fail(ctx, DMC_ERR_ARG, std::string(what) + ": bad mem");
    return DMC_OK;
}

int reserve(dmc_ctx* ctx, Buf& b, size_t bytes) {
    if (b.cap >= bytes && b.p) return DMC_OK;
    ctx->alloc_epoch++;
    if (b.p) {      // growing means synchronising and freeing: not allowed while the caller captures its stream into a graph
        cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
        if (ctx->stream && ctx->stream != cudaStreamLegacy && cudaStreamIsCapturing(ctx->stream, &st) == cudaSuccess && st != cudaStreamCaptureStatusNone)
            return fail(ctx, DMC_ERR_ARG, "scratch memory must grow while the stream is being captured; run the call once outside the capture first");
        cudaGetLastError();
    }
    if (b.p) { CUDA_TRY(ctx, cudaDeviceSynchronize()); CUDA_TRY(ctx, cudaFree(b.p)); b.p = nullptr; b.cap = 0; }
    size_t cap = (bytes + 4095) & ~(size_t)4095;
    CUDA_TRY(ctx, cudaMalloc(&b.p, cap));
    b.cap = cap;
    return DMC_OK;
}

int after_launch(dmc_ctx* ctx, int nk) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ctx, DMC_ERR_CUDA, std::string("kernel launch: ") + cudaGetErrorString(e));
    ctx->launches += (uint64_t)nk;
    return DMC_OK;
}
#define LAUNCH(ctx, call) do { int _nk = (call); int _rc = after_launch(ctx, _nk); if (_rc) return _rc; } while (0)
#define TRY(expr) do { int _rc = (expr); if (_rc < 0) return _rc; } while (0)

// Small dense HOST images in pinned, device-mapped memory (dmc_host_alloc, dmc_host_register, cudaMallocHost, cudaHostRegister)
// are not copied: the kernels read and write them in place over the host link.  For a 640x480 frame that saves two DMA
// set-ups and lets the last kernel's stores overlap its arithmetic (BASELINE config 2, batch-1 latency).  Larger frames
// keep the copies: a tile's halo would cross the link once per neighbouring tile.  DMC_ZERO_COPY_MAX=<bytes> overrides.
void* mapped_ptr(const dmc_image* im) {
    static const size_t max_bytes = getenv("DMC_ZERO_COPY_MAX") ? (size_t)atoll(getenv("DMC_ZERO_COPY_MAX")) : ((size_t)2 << 20);
    if (im->mem != DMC_MEM_HOST || step_of(im) != dense_step(im) || image_bytes(im) > max_bytes) return nullptr;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, im->data) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return a.type == cudaMemoryTypeHost ? a.devicePointer : nullptr;
}

// Brings `im` into a dense device buffer.  Device-resident dense images are used in place.
int stage_in(dmc_ctx* ctx, const dmc_image* im, Buf& scratch, cudaStream_t s, const void** out) {
    size_t row = dense_step(im), st = step_of(im);
    if (im->mem == DMC_MEM_DEVICE && st == row) { *out = im->data; return DMC_OK; }
    if (void* z = mapped_ptr(im)) { *out = z; return DMC_OK; }
    TRY(reserve(ctx, scratch, image_bytes(im)));
    CUDA_TRY(ctx, cudaMemcpy2DAsync(scratch.p, row, im->data, st, row, im->rows,
                                    im->mem == DMC_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, s));
    *out = scratch.p;
    return DMC_OK;
}

bool overlaps(const void* a, size_t na, const void* b, size_t nb) {
    const uintptr_t x = (uintptr_t)a, y = (uintptr_t)b;
    return a && b && x < y + nb && y < x + na;
}

// Chooses where the kernels write: straight into a dense device dst unless its bytes overlap the source's (in-place calls
// and offset views of one buffer alike: the kernels read halos from src while other CTAs write dst).
int stage_out_begin(dmc_ctx* ctx, const dmc_image* dst, const void* src_dev, size_t src_bytes, Buf& scratch, void** out) {
    if (dst->mem == DMC_MEM_DEVICE && step_of(dst) == dense_step(dst) && !overlaps(dst->data, image_bytes(dst), src_dev, src_bytes)) { *out = dst->data; return DMC_OK; }
    if (void* z = mapped_ptr(dst)) if (!overlaps(z, image_bytes(dst), src_dev, src_bytes)) { *out = z; return DMC_OK; }
    TRY(reserve(ctx, scratch, image_bytes(dst)));
    *out = scratch.p;
    return DMC_OK;
}

int stage_out_end(dmc_ctx* ctx, const dmc_image* dst, void* dev, cudaStream_t s) {
    if (dev != dst->data && (dst->mem != DMC_MEM_HOST || dev != mapped_ptr(dst))) {
        size_t row = dense_step(dst);
        CUDA_TRY(ctx, cudaMemcpy2DAsync(dst->data, step_of(dst), dev, row, row, dst->rows,
                                        dst->mem == DMC_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, s));
    }
    if (dst->mem == DMC_MEM_HOST) CUDA_TRY(ctx, cudaStreamSynchronize(s));   // reference semantics: dst valid on return
    return DMC_OK;
}

// Prologue of a single-image operator: it runs on slot 0, which follows the context's stream; `in` is src on the device,
// `out` where the kernels write dst (stage_out_end delivers it).
int stage_op(dmc_ctx* ctx, const dmc_image* src, const dmc_image* dst, const void** in, void** out) {
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    Slot& sl = ctx->slot[0]; sl.stream = ctx->stream;
    TRY(stage_in(ctx, src, sl.buf[SB_IN], sl.stream, in));
    return stage_out_begin(ctx, dst, *in, image_bytes(src), sl.buf[SB_OUT], out);
}

// The identity cases of the operators: dst becomes a copy of src.
int copy_unless_same(dmc_ctx* ctx, void* dst, const void* src, size_t bytes, cudaStream_t s) {
    if (dst != src) CUDA_TRY(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s));
    return DMC_OK;
}

int check_radius(dmc_ctx* ctx, int r, const char* what) {
    if (r < 0 || r > DMC_MAX_RADIUS) return fail(ctx, DMC_ERR_ARG, std::string(what) + " out of range [0, 10]");
    return DMC_OK;
}

// ---- per-stage event timing ------------------------------------------------------------------------------
cudaEvent_t prof_event(dmc_ctx* ctx) {
    if (!ctx->prof_free.empty()) { cudaEvent_t e = ctx->prof_free.back(); ctx->prof_free.pop_back(); return e; }
    cudaEvent_t e = nullptr; cudaEventCreate(&e); return e;
}
struct ProfScope {          // records an event pair around the launches issued while it is alive
    dmc_ctx* ctx; cudaStream_t s; int idx = -1;
    ProfScope(dmc_ctx* c, cudaStream_t st, int stage, uint64_t pixels) : ctx(c), s(st) {
        if (!(c->profile_mask & (1 << stage))) return;
        dmc_ctx::ProfRec r; r.a = prof_event(c); r.b = prof_event(c); r.stage = stage; r.pixels = pixels;
        cudaEventRecord(r.a, s); c->prof_pending.push_back(r); idx = (int)c->prof_pending.size() - 1;
    }
    ~ProfScope() { if (idx >= 0) cudaEventRecord(ctx->prof_pending[idx].b, s); }
};

// ---- the range filter dispatcher (binalyWeightedRangeFilter.cpp:1106-1178) on dense device buffers ---------
// load_op / store_op / maf describe fused conversions around the 32f kernel.  `tmp` is a float scratch for
// the separable variant.  Returns DMC_UNSUPPORTED for the reference's silent no-ops.
int range_filter_8u(dmc_ctx* ctx, const uint8_t* src, uint8_t* dst, Buf& tmp, int n, int H, int W, int cn, int kw, int kh,
                    float threshold, int method, cudaStream_t s) {
    size_t bytes = (size_t)n * H * W * cn;
    const int th = (int)(uint8_t)(int)threshold;                                   // (uchar)threshold :1113
    if (method == DMC_FULL_KERNEL) {
        if (kw == 0 || kh == 0) return copy_unless_same(ctx, dst, src, bytes, s);   // :1033
        RowSpan rs = make_rowspan(kw, kh);
        if (cn == 1 && kw == kh && (kw & 1)) {                                     // square odd window: packed-half fast path when exact
            int nk = launch_bwrf8u_h2(src, dst, n, H, W, kw >> 1, th, rs.ntaps, s);
            if (nk) return after_launch(ctx, nk);
        }
        if (cn == 3 && kw == kh && (kw & 1)) {
            int nk = launch_bwrf8u_c3_h2(src, dst, n, H, W, kw >> 1, th, rs.ntaps, s);
            if (nk) return after_launch(ctx, nk);
        }
        LAUNCH(ctx, launch_bwrf8u(src, dst, n, H, W, cn, rs, th, s));
        return DMC_OK;
    }
    if (method == DMC_SEPARABLE_KERNEL) {                                          // :1084-1091 (both guards test .width)
        if (kw <= 1) return copy_unless_same(ctx, dst, src, bytes, s);
        TRY(reserve(ctx, tmp, bytes));
        RowSpan rh = make_rowspan(kw, 1), rv = make_rowspan(1, kh);
        LAUNCH(ctx, launch_bwrf8u(src, (uint8_t*)tmp.p, n, H, W, cn, rh, th, s));
        if (kh == 0) { CUDA_TRY(ctx, cudaMemcpyAsync(dst, tmp.p, bytes, cudaMemcpyDeviceToDevice, s)); return DMC_OK; }
        LAUNCH(ctx, launch_bwrf8u((const uint8_t*)tmp.p, dst, n, H, W, cn, rv, th, s));
        return DMC_OK;
    }
    return DMC_UNSUPPORTED;                                                        // 8U + FULL_KERNEL_PAIR: body commented out :1140-1143
}

int range_filter_32f(dmc_ctx* ctx, const void* src, void* dst, Buf& tmp, int n, int H, int W, int cn, int kw, int kh,
                     float threshold, int method, int load_op, float maf, int store_op, cudaStream_t s) {
    size_t count = (size_t)n * H * W * cn;
    if (method == DMC_FULL_KERNEL || method == DMC_FULL_KERNEL_PAIR) {
        // FULL_KERNEL_PAIR has no deterministic reference output (racy scatter, unwritten tail columns); it computes
        // the FULL_KERNEL result that it approximates.  No bit-parity claim for that method (DESIGN.md).
        if (kw == 0 || kh == 0) { kw = 1; kh = 1; if (load_op == LOAD_F32 && store_op == STORE_F32) return copy_unless_same(ctx, dst, src, count * sizeof(float), s); }
        RowSpan rs = make_rowspan(kw, kh);
        LAUNCH(ctx, launch_bwrf32f(src, dst, n, H, W, cn, rs, threshold, load_op, maf, store_op, s));
        return DMC_OK;
    }
    if (method == DMC_SEPARABLE_KERNEL) {                                          // :1092-1099
        TRY(reserve(ctx, tmp, count * sizeof(float)));
        if (kw <= 1) return DMC_ERR_ARG;   // handled by the callers (plain copy / conversion)
        RowSpan rh = make_rowspan(kw, 1), rv = make_rowspan(1, kh);
        LAUNCH(ctx, launch_bwrf32f(src, tmp.p, n, H, W, cn, rh, threshold, load_op, maf, STORE_F32, s));
        LAUNCH(ctx, launch_bwrf32f(tmp.p, dst, n, H, W, cn, rv, threshold, LOAD_F32, 0.f, store_op, s));
        return DMC_OK;
    }
    return DMC_UNSUPPORTED;
}

// ---- the chain on dense device buffers (postFilterSet.cpp:21-63) ------------------------------------------
int run_chain(dmc_ctx* ctx, Slot& sl, const uint8_t* src, void* dst, int n, int H, int W, const dmc_chain_params& p) {
    cudaStream_t s = sl.stream;
    const size_t px = (size_t)n * H * W;
    Buf& ping = sl.buf[SB_PING]; Buf& pong = sl.buf[SB_PONG]; Buf& ftmp = sl.buf[SB_FLOAT];
    TRY(reserve(ctx, ping, px)); TRY(reserve(ctx, pong, px));
    const uint8_t* cur = src;
    uint8_t* nxt = (uint8_t*)ping.p;
    auto advance = [&]() { cur = nxt; nxt = (nxt == (uint8_t*)ping.p) ? (uint8_t*)pong.p : (uint8_t*)ping.p; };
    if (p.median_r > 0) { ProfScope ps(ctx, s, DMC_STAGE_MEDIAN, px); LAUNCH(ctx, launch_median8u(cur, nxt, n, H, W, p.median_r, s)); advance(); }              // :23/:36/:47/:59 (k = 1: copy)
    if (p.gaussian_r > 0) {                                                                                            // :24 (d = 1: identity)
        GaussTaps t;
        if (!make_gauss_taps(2 * p.gaussian_r + 1, p.gaussian_r + 0.5, H, W, &t)) return fail(ctx, DMC_ERR_ARG, "gaussian radius");
        if (t.rx > 0 || t.ry > 0) { ProfScope ps(ctx, s, DMC_STAGE_GAUSS, px); LAUNCH(ctx, launch_gauss8u(cur, nxt, n, H, W, t, s)); advance(); }
    }
    if (p.minmax_r > 0) { ProfScope ps(ctx, s, DMC_STAGE_MINMAX, px); LAUNCH(ctx, launch_minmax(cur, nxt, n, H, W, DMC_8U, 1, p.minmax_r, s)); advance(); }     // :25 (r = 0: identity)
    const int k = 2 * p.brange_r + 1;
    ProfScope ps_range(ctx, s, DMC_STAGE_RANGE, px);
    if (p.chain == DMC_CHAIN_DISP8U) {                                                                                 // :57-63
        int rc = range_filter_8u(ctx, cur, (uint8_t*)dst, ftmp, n, H, W, 1, k, k, p.brange_th, p.brange_method, s);
        return rc;
    }
    const bool depth = p.chain != DMC_CHAIN_DISP32F;
    const int load_op = depth ? LOAD_U8_DISP2DEPTH : LOAD_U8;                                                          // :27/:40 vs :51
    const float maf = depth ? (float)p.amp * (float)(p.focus * p.baseline) : 0.f;                                      // a * focal_baseline in FP32, depthmapUtil.cpp:935
    const int store_op = p.chain == DMC_CHAIN_DEPTH32F ? STORE_F32 : STORE_U16;                                        // :31/:54 convertTo(CV_16U)
    bool filtered = true;
    if (p.brange_method == DMC_SEPARABLE_KERNEL && k <= 1) filtered = false;                                           // SP with width <= 1: src.copyTo(dst)
    else if (p.brange_method != DMC_FULL_KERNEL && p.brange_method != DMC_FULL_KERNEL_PAIR && p.brange_method != DMC_SEPARABLE_KERNEL) {
        if (p.chain == DMC_CHAIN_DEPTH32F) return DMC_UNSUPPORTED;     // dest never written by the reference
        filtered = false;                                              // bufff converted to 16U unfiltered
    }
    if (filtered) return range_filter_32f(ctx, cur, dst, ftmp, n, H, W, 1, k, k, p.brange_th, p.brange_method, load_op, maf, store_op, s);
    // unfiltered: disparity -> (depth | float) -> store
    TRY(reserve(ctx, ftmp, px * sizeof(float)));
    float* f = store_op == STORE_F32 ? (float*)dst : (float*)ftmp.p;
    if (depth) LAUNCH(ctx, launch_convert(0, cur, f, (long)px, (float)(p.focus * p.baseline), (float)p.amp, 0.f, s));
    else { RowSpan one = make_rowspan(1, 1); LAUNCH(ctx, launch_bwrf32f(cur, f, n, H, W, 1, one, FLT_MAX, LOAD_U8, 0.f, STORE_F32, s)); }
    if (store_op == STORE_U16) LAUNCH(ctx, launch_f32_to_u16(f, (uint16_t*)dst, (long)px, s));
    return DMC_OK;
}

int chain_out_type(int chain) { return chain == DMC_CHAIN_DISP8U ? DMC_8U : chain == DMC_CHAIN_DEPTH32F ? DMC_32F : DMC_16U; }

int check_chain_params(dmc_ctx* ctx, const dmc_chain_params& p) {
    TRY(check_radius(ctx, p.median_r, "median_r")); TRY(check_radius(ctx, p.gaussian_r, "gaussian_r"));
    TRY(check_radius(ctx, p.minmax_r, "minmax_r")); TRY(check_radius(ctx, p.brange_r, "brange_r"));
    if (p.chain < DMC_CHAIN_DISP8U || p.chain > DMC_CHAIN_DISP32F) return fail(ctx, DMC_ERR_ARG, "unknown chain");
    return DMC_OK;
}

bool graph_eligible(dmc_ctx* ctx, cudaStream_t s) {
    static const bool env_off = getenv("DMC_NO_GRAPH") != nullptr;
    // the legacy default stream cannot be captured; with stage profiling on, events are recorded between the kernels
    if (env_off || ctx->graphs_off || ctx->profile_mask != 0 || s == nullptr || s == cudaStreamLegacy) return false;
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;      // the caller may be capturing this stream into a graph of its own
    if (cudaStreamIsCapturing(s, &st) != cudaSuccess) { cudaGetLastError(); return false; }
    return st == cudaStreamCaptureStatusNone;
}

void drop_graph(dmc_ctx* ctx) {
    if (ctx->graph_exec) cudaGraphExecDestroy(ctx->graph_exec);
    ctx->graph_exec = nullptr; ctx->graph_valid = false;
}

// Captures run_chain for one frame into a graph, instantiates and launches it.  DMC_UNSUPPORTED: could not capture (the
// caller then launches the kernels directly and graphs stay off for this context).
int capture_chain(dmc_ctx* ctx, Slot& sl, const dmc_ctx::GraphKey& key, const uint8_t* in, void* out, int rows, int cols, const dmc_chain_params& p) {
    drop_graph(ctx);
    const uint64_t epoch = ctx->alloc_epoch, before = ctx->launches;
    if (cudaStreamBeginCapture(sl.stream, cudaStreamCaptureModeRelaxed) != cudaSuccess) { cudaGetLastError(); ctx->graphs_off = true; return DMC_UNSUPPORTED; }
    int rc = run_chain(ctx, sl, in, out, 1, rows, cols, p);
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamEndCapture(sl.stream, &g);
    const uint64_t nk = ctx->launches - before; ctx->launches = before;
    if (rc != DMC_OK || e != cudaSuccess || !g || epoch != ctx->alloc_epoch) {      // (a reallocation inside the capture: pointers stale)
        if (g) cudaGraphDestroy(g);
        cudaGetLastError(); ctx->graphs_off = true;
        return rc != DMC_OK && rc != DMC_UNSUPPORTED ? rc : DMC_UNSUPPORTED;
    }
    e = cudaGraphInstantiate(&ctx->graph_exec, g, 0);
    cudaGraphDestroy(g);
    if (e != cudaSuccess) { cudaGetLastError(); ctx->graph_exec = nullptr; ctx->graphs_off = true; return DMC_UNSUPPORTED; }
    ctx->graph_key = key; ctx->graph_epoch = epoch; ctx->graph_launches = nk; ctx->graph_valid = true;
    CUDA_TRY(ctx, cudaGraphLaunch(ctx->graph_exec, sl.stream));
    ctx->launches += nk;
    return DMC_OK;
}

int chain_single(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, const dmc_chain_params& p) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, src, "src")); TRY(check_image(ctx, dst, "dst")); TRY(check_chain_params(ctx, p));
    if (src->cvtype != DMC_8U) return fail(ctx, DMC_ERR_TYPE, "PostFilterSet: src must be CV_8UC1");
    if (dst->cvtype != chain_out_type(p.chain)) return fail(ctx, DMC_ERR_TYPE, "PostFilterSet: dst has the wrong type for this entry point");
    if (dst->rows != src->rows || dst->cols != src->cols) return fail(ctx, DMC_ERR_SIZE, "PostFilterSet: dst size != src size");
    const void* in; void* out;
    TRY(stage_op(ctx, src, dst, &in, &out));
    Slot& sl = ctx->slot[0];
    int rc = DMC_OK;
    const bool direct = in != sl.buf[SB_IN].p && out != sl.buf[SB_OUT].p;  // device-resident (or mapped host memory), dense, not aliased: nothing but kernels
    if (direct && graph_eligible(ctx, sl.stream)) {
        dmc_ctx::GraphKey key; memset(&key, 0, sizeof key);
        key.in = in; key.out = out; key.rows = src->rows; key.cols = src->cols; key.stream = sl.stream;
        key.p.chain = p.chain; key.p.median_r = p.median_r; key.p.gaussian_r = p.gaussian_r; key.p.minmax_r = p.minmax_r; key.p.brange_r = p.brange_r;
        key.p.brange_th = p.brange_th; key.p.brange_method = p.brange_method; key.p.focus = p.focus; key.p.baseline = p.baseline; key.p.amp = p.amp;   // (field by field: padding stays zero)
        if (ctx->graph_valid && ctx->graph_epoch == ctx->alloc_epoch && memcmp(&key, &ctx->graph_key, sizeof key) == 0) {
            CUDA_TRY(ctx, cudaGraphLaunch(ctx->graph_exec, sl.stream));
            ctx->launches += ctx->graph_launches; ctx->graph_replays++;
            return stage_out_end(ctx, dst, out, sl.stream);        // (nothing to copy; waits if dst is host memory)
        }
        if (ctx->graph_seen_valid && memcmp(&key, &ctx->graph_seen, sizeof key) == 0) {
            rc = capture_chain(ctx, sl, key, (const uint8_t*)in, out, src->rows, src->cols, p);      // launches it as well
            if (rc == DMC_OK) return stage_out_end(ctx, dst, out, sl.stream);
            if (rc != DMC_UNSUPPORTED) return rc;
            rc = DMC_OK;                                           // capture not possible here: plain launches below
        }
        ctx->graph_seen = key; ctx->graph_seen_valid = true;
    }
    rc = run_chain(ctx, sl, (const uint8_t*)in, out, 1, src->rows, src->cols, p);
    if (rc != DMC_OK) { if (dst->mem == DMC_MEM_HOST || rc < 0) cudaStreamSynchronize(sl.stream); return rc; }
    return stage_out_end(ctx, dst, out, sl.stream);
}

void drop_gateway(dmc_ctx* ctx) {
    if (ctx->gw.device < 0) return;
    cudaSetDevice(ctx->gw.device);
    for (int i = 0; i < kSlots; i++) {
        if (ctx->gw.stream[i]) { cudaStreamSynchronize(ctx->gw.stream[i]); cudaStreamDestroy(ctx->gw.stream[i]); ctx->gw.stream[i] = nullptr; }
        if (ctx->gw.ev_in[i]) { cudaEventDestroy(ctx->gw.ev_in[i]); ctx->gw.ev_in[i] = nullptr; }
        if (ctx->gw.ev_done[i]) { cudaEventDestroy(ctx->gw.ev_done[i]); ctx->gw.ev_done[i] = nullptr; }
        if (ctx->gw.in[i].p) { cudaFree(ctx->gw.in[i].p); ctx->gw.in[i] = Buf(); }
        if (ctx->gw.out[i].p) { cudaFree(ctx->gw.out[i].p); ctx->gw.out[i] = Buf(); }
    }
    cudaSetDevice(ctx->device);
    for (int i = 0; i < kSlots; i++) if (ctx->gw.ev_out[i]) { cudaEventDestroy(ctx->gw.ev_out[i]); ctx->gw.ev_out[i] = nullptr; }
    ctx->gw.device = -1;
}

// A tuning knob of the batch entry points: `name` in MiB when it is set to a positive number, else `dflt` bytes.
size_t env_mib(const char* name, size_t dflt) {
    if (const char* e = getenv(name)) { long v = atol(e); if (v > 0) return (size_t)v << 20; }
    return dflt;
}

// Frames per group or chunk of a batch: `target` bytes of `frame_bytes` each, at least one frame, at most `cap` (a grid
// dimension limit) and n_frames.  spread: at least kSlots chunks when there are that many frames, so every slot has work.
int chunk_frames(size_t target, size_t frame_bytes, int n_frames, int cap, bool spread) {
    size_t c = target / frame_bytes;
    if (c > (size_t)cap) c = cap;
    if (c > (size_t)n_frames) c = n_frames;
    const int chunk = c < 1 ? 1 : (int)c;
    return spread && n_frames / chunk < kSlots && n_frames >= kSlots ? (n_frames + kSlots - 1) / kSlots : chunk;
}

// Frames [f0, f0 + nf) of a streamed batch on slot `si`.  routed: its host traffic runs over the gateway's link; `copy` is
// the stream that carries it (the gateway's copy stream of the slot, or the slot's own).
struct Chunk { int f0, nf, si; Slot* sl; bool routed; cudaStream_t copy; };

// Staging buffers of a chunk's host traffic: `local_in` / `local_out` of its slot, or when routed the slot's buffers on
// the gateway's device (allocated there).  out_bytes == 0: no output staging.
int reserve_io(dmc_ctx* ctx, const Chunk& c, size_t in_bytes, size_t out_bytes, Buf& local_in, Buf& local_out, void** in, void** out) {
    Buf& bi = c.routed ? ctx->gw.in[c.si] : local_in;
    Buf& bo = c.routed ? ctx->gw.out[c.si] : local_out;
    if (!c.routed) {
        TRY(reserve(ctx, bi, in_bytes));
        if (out_bytes) TRY(reserve(ctx, bo, out_bytes));
    } else if (bi.cap < in_bytes || bo.cap < out_bytes) {
        CUDA_TRY(ctx, cudaDeviceSynchronize());                  // this device's kernels may still be reading the old buffers
        CUDA_TRY(ctx, cudaSetDevice(ctx->gw.device));
        int rc = reserve(ctx, bi, in_bytes); if (rc == DMC_OK && out_bytes) rc = reserve(ctx, bo, out_bytes);
        cudaSetDevice(ctx->device);
        if (rc != DMC_OK) return rc;
    }
    *in = bi.p; *out = bo.p;
    return DMC_OK;
}

// Streams n_frames through the kSlots slots in chunks of `chunk` frames, so that the copies in, the kernels and the copies
// out of different chunks overlap.  Chunk i runs on slot i % kSlots (slot 0 follows ctx->stream); a slot's first chunk
// waits for the work queued on ctx->stream before the call.  Per chunk the caller's prepare (host work, reservations),
// copy_in (on c.copy), kernels (on the slot's stream) and copy_out (on c.copy) run in turn.  routed: the copies run on the
// gateway's device (dmc_set_gateway), fenced against the kernels with events.  staged: prepare refills the slot's pinned
// hstage, so it first waits until the slot's previous chunk is done.  Stops at the first error; drains every stream it used.
template <class Prepare, class CopyIn, class Kernels, class CopyOut>
int stream_chunks(dmc_ctx* ctx, int n_frames, int chunk, bool routed, bool staged, Prepare prepare, CopyIn copy_in, Kernels kernels, CopyOut copy_out) {
    dmc_ctx::Gateway& gw = ctx->gw;
    cudaEvent_t ready;
    CUDA_TRY(ctx, cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
    CUDA_TRY(ctx, cudaEventRecord(ready, ctx->stream));
    int rc = DMC_OK;
    for (int f0 = 0, ci = 0; f0 < n_frames && rc == DMC_OK; f0 += chunk, ci++) {
        const int si = ci % kSlots;
        Slot& sl = ctx->slot[si]; if (si == 0) sl.stream = ctx->stream;
        const Chunk c = {f0, n_frames - f0 < chunk ? n_frames - f0 : chunk, si, &sl, routed, routed ? gw.stream[si] : sl.stream};
        if (ci < kSlots && sl.stream != ctx->stream) cudaStreamWaitEvent(sl.stream, ready, 0);
        if (sl.done_pending) { cudaError_t e = cudaEventSynchronize(routed ? gw.ev_done[si] : sl.done); sl.done_pending = false; if (e != cudaSuccess) { rc = fail(ctx, DMC_ERR_CUDA, cudaGetErrorString(e)); break; } }
        if (staged && !sl.done && cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming) != cudaSuccess) { rc = fail(ctx, DMC_ERR_CUDA, "cudaEventCreate"); break; }
        if ((rc = prepare(c)) != DMC_OK) break;
        if (routed) { cudaSetDevice(gw.device); if (ci < kSlots) cudaStreamWaitEvent(c.copy, ready, 0); }
        cudaError_t e = copy_in(c);
        if (e == cudaSuccess && routed) { e = cudaEventRecord(gw.ev_in[si], c.copy); cudaSetDevice(ctx->device); if (e == cudaSuccess) e = cudaStreamWaitEvent(sl.stream, gw.ev_in[si], 0); }
        if (e != cudaSuccess) { cudaSetDevice(ctx->device); rc = fail(ctx, DMC_ERR_CUDA, cudaGetErrorString(e)); break; }
        if ((rc = kernels(c)) != DMC_OK) break;
        if (routed) { e = cudaEventRecord(gw.ev_out[si], sl.stream); cudaSetDevice(gw.device); if (e == cudaSuccess) e = cudaStreamWaitEvent(c.copy, gw.ev_out[si], 0); }
        if (e == cudaSuccess) e = copy_out(c);
        if (e == cudaSuccess && staged) { e = cudaEventRecord(routed ? gw.ev_done[si] : sl.done, c.copy); sl.done_pending = e == cudaSuccess; }   // (an event lives on its stream's device)
        if (routed) cudaSetDevice(ctx->device);
        if (e != cudaSuccess) { rc = fail(ctx, DMC_ERR_CUDA, cudaGetErrorString(e)); break; }
    }
    for (int i = 0; i < kSlots; i++) {
        cudaError_t e = cudaStreamSynchronize(ctx->slot[i].stream);
        if (e == cudaSuccess && routed) e = cudaStreamSynchronize(gw.stream[i]);
        ctx->slot[i].done_pending = false;
        if (e != cudaSuccess && rc == DMC_OK) rc = fail(ctx, DMC_ERR_CUDA, cudaGetErrorString(e));
    }
    cudaEventDestroy(ready);
    return rc;
}

}  // namespace

// ==============================================================================================================
extern "C" {

int dmc_get_gateway(const dmc_ctx* ctx) { return ctx ? ctx->gw.device : -1; }

int dmc_set_gateway(dmc_ctx* ctx, int gateway_device) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    for (int i = 0; i < kSlots; i++) CUDA_TRY(ctx, cudaStreamSynchronize(ctx->slot[i].stream));
    drop_gateway(ctx);
    if (gateway_device < 0 || gateway_device == ctx->device) return DMC_OK;
    int n = 0; CUDA_TRY(ctx, cudaGetDeviceCount(&n));
    if (gateway_device >= n) return fail(ctx, DMC_ERR_ARG, "dmc_set_gateway: device index out of range");
    int can = 0; CUDA_TRY(ctx, cudaDeviceCanAccessPeer(&can, ctx->device, gateway_device));
    if (!can) return fail(ctx, DMC_ERR_ARG, "dmc_set_gateway: no peer access from this context's device to the gateway");
    cudaError_t e = cudaDeviceEnablePeerAccess(gateway_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
    else if (e != cudaSuccess) return fail(ctx, DMC_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
    for (int i = 0; i < kSlots; i++) CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->gw.ev_out[i], cudaEventDisableTiming));
    ctx->gw.device = gateway_device;
    e = cudaSetDevice(gateway_device);
    for (int i = 0; i < kSlots && e == cudaSuccess; i++) {
        e = cudaStreamCreateWithFlags(&ctx->gw.stream[i], cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->gw.ev_in[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->gw.ev_done[i], cudaEventDisableTiming);
    }
    cudaSetDevice(ctx->device);
    if (e != cudaSuccess) { drop_gateway(ctx); return fail(ctx, DMC_ERR_CUDA, std::string("dmc_set_gateway: ") + cudaGetErrorString(e)); }
    return DMC_OK;
}

int dmc_version(void) { return 100; }

int dmc_device_count(void) { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) return 0; return n; }

int dmc_create(int device, dmc_ctx** out) {
    if (!out) return fail(nullptr, DMC_ERR_ARG, "dmc_create: null out");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) return fail(nullptr, DMC_ERR_CUDA, std::string("dmc_create: no CUDA device (") + cudaGetErrorString(e) + "); libdmc_b200 has no CPU fallback");
    if (device < 0 || device >= n) return fail(nullptr, DMC_ERR_ARG, "dmc_create: device index out of range");
    if ((e = cudaSetDevice(device)) != cudaSuccess) return fail(nullptr, DMC_ERR_CUDA, cudaGetErrorString(e));
    dmc_ctx* ctx = new dmc_ctx();
    ctx->device = device;
    if ((e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess) { delete ctx; return fail(nullptr, DMC_ERR_CUDA, cudaGetErrorString(e)); }
    ctx->stream = ctx->own_stream;
    for (int i = 0; i < kSlots; i++) {
        if (i == 0) ctx->slot[i].stream = ctx->stream;
        else if ((e = cudaStreamCreateWithFlags(&ctx->slot[i].stream, cudaStreamNonBlocking)) != cudaSuccess) { dmc_destroy(ctx); return fail(nullptr, DMC_ERR_CUDA, cudaGetErrorString(e)); }
    }
    *out = ctx;
    return DMC_OK;
}

void dmc_destroy(dmc_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (int i = 0; i < kSlots; i++) {
        for (int b = 0; b < SB_COUNT; b++) if (ctx->slot[i].buf[b].p) cudaFree(ctx->slot[i].buf[b].p);
        if (ctx->slot[i].hstage) cudaFreeHost(ctx->slot[i].hstage);
        if (ctx->slot[i].done) cudaEventDestroy(ctx->slot[i].done);
        if (i > 0 && ctx->slot[i].stream) cudaStreamDestroy(ctx->slot[i].stream);
    }
    if (ctx->xtab) cudaFree(ctx->xtab);
    drop_gateway(ctx);
    drop_graph(ctx);
    for (auto& b : ctx->jpeg) if (b.p) cudaFree(b.p);
    for (auto& b : ctx->jpeg_enc) if (b.p) cudaFree(b.p);
    for (auto& b : ctx->render) if (b.p) cudaFree(b.p);
    if (ctx->render_flag) cudaFreeHost(ctx->render_flag);
    for (auto& r : ctx->prof_pending) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (auto e : ctx->prof_free) cudaEventDestroy(e);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

const char* dmc_last_error(const dmc_ctx* ctx) { return ctx ? ctx->err.c_str() : g_err.c_str(); }

int dmc_set_stream(dmc_ctx* ctx, void* cuda_stream) {
    if (!ctx) return DMC_ERR_ARG;
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    ctx->slot[0].stream = ctx->stream;
    return DMC_OK;
}
void* dmc_get_stream(dmc_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int dmc_synchronize(dmc_ctx* ctx) {
    if (!ctx) return DMC_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    for (int i = 0; i < kSlots; i++) CUDA_TRY(ctx, cudaStreamSynchronize(ctx->slot[i].stream));
    return DMC_OK;
}

uint64_t dmc_kernel_launches(const dmc_ctx* ctx) { return ctx ? ctx->launches : 0; }

void* dmc_host_alloc(size_t bytes) { void* p = nullptr; if (cudaMallocHost(&p, bytes) != cudaSuccess) return nullptr; return p; }
void dmc_host_free(void* p) { if (p) cudaFreeHost(p); }
int dmc_host_register(void* p, size_t bytes) {
    if (!p || !bytes) return DMC_ERR_ARG;
    if (cudaHostRegister(p, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped) != cudaSuccess) { cudaGetLastError(); return DMC_ERR_CUDA; }
    return DMC_OK;
}
int dmc_host_unregister(void* p) {
    if (!p) return DMC_ERR_ARG;
    if (cudaHostUnregister(p) != cudaSuccess) { cudaGetLastError(); return DMC_ERR_CUDA; }
    return DMC_OK;
}

int dmc_set_lanes(dmc_ctx* ctx, int lanes) {
    if (!ctx || lanes < 1 || lanes > kSlots) return DMC_ERR_ARG;
    ctx->lanes = lanes;
    return DMC_OK;
}

int dmc_profile_enable(dmc_ctx* ctx, int stage_mask) {
    if (!ctx) return DMC_ERR_ARG;
    ctx->profile_mask = stage_mask;
    return DMC_OK;
}

int dmc_profile_read(dmc_ctx* ctx, int stage, double* total_ms, uint64_t* launches, uint64_t* pixels, int reset) {
    if (!ctx || stage < 0 || stage >= DMC_STAGE_COUNT) return DMC_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    for (int i = 0; i < kSlots; i++) CUDA_TRY(ctx, cudaStreamSynchronize(ctx->slot[i].stream));
    for (auto& r : ctx->prof_pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) { ctx->prof_ms[r.stage] += ms; ctx->prof_launches[r.stage]++; ctx->prof_pixels[r.stage] += r.pixels; }
        ctx->prof_free.push_back(r.a); ctx->prof_free.push_back(r.b);
    }
    ctx->prof_pending.clear();
    if (total_ms) *total_ms = ctx->prof_ms[stage];
    if (launches) *launches = ctx->prof_launches[stage];
    if (pixels) *pixels = ctx->prof_pixels[stage];
    if (reset) { ctx->prof_ms[stage] = 0; ctx->prof_launches[stage] = 0; ctx->prof_pixels[stage] = 0; }
    return DMC_OK;
}

// ---- PostFilterSet ---------------------------------------------------------------------------------------------
int dmc_post_filter_set(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int median_r, int gaussian_r, int minmax_r,
                        int brange_r, int brange_th, int brange_method) {
    dmc_chain_params p = {DMC_CHAIN_DISP8U, median_r, gaussian_r, minmax_r, brange_r, (float)brange_th, brange_method, 0, 0, 0};
    return chain_single(ctx, src, dst, p);
}
int dmc_filter_disp8u_depth32f(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, double focus, double baseline, double amp,
                               int median_r, int gaussian_r, int minmax_r, int brange_r, float brange_th, int brange_method) {
    dmc_chain_params p = {DMC_CHAIN_DEPTH32F, median_r, gaussian_r, minmax_r, brange_r, brange_th, brange_method, focus, baseline, amp};
    return chain_single(ctx, src, dst, p);
}
int dmc_filter_disp8u_depth16u(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, double focus, double baseline, double amp,
                               int median_r, int gaussian_r, int minmax_r, int brange_r, float brange_th, int brange_method) {
    dmc_chain_params p = {DMC_CHAIN_DEPTH16U, median_r, gaussian_r, minmax_r, brange_r, brange_th, brange_method, focus, baseline, amp};
    return chain_single(ctx, src, dst, p);
}
int dmc_filter_disp8u_disp32f(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int median_r, int gaussian_r, int minmax_r,
                              int brange_r, float brange_th, int brange_method) {
    dmc_chain_params p = {DMC_CHAIN_DISP32F, median_r, gaussian_r, minmax_r, brange_r, brange_th, brange_method, 0, 0, 0};
    return chain_single(ctx, src, dst, p);
}

int dmc_shard_frames(int n_frames, int rank, int world, int* begin, int* count) {
    if (n_frames < 0 || world <= 0 || rank < 0 || rank >= world || !begin || !count) return DMC_ERR_ARG;
    int base = n_frames / world, rem = n_frames % world;
    *begin = rank * base + (rank < rem ? rank : rem);
    *count = base + (rank < rem ? 1 : 0);
    return DMC_OK;
}

// Frame batches.  Device memory: one launch sequence over all frames.  Host memory: chunks of frames flow through
// kSlots independent (stream, buffers) slots so that the H2D copy of chunk i+1, the kernels of chunk i and the D2H
// copy of chunk i-1 overlap on the copy engines and the SMs.
int dmc_chain_batch(dmc_ctx* ctx, const void* src, void* dst, int n_frames, int rows, int cols, const dmc_chain_params* pp, int mem) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    if (!src || !dst || !pp || n_frames < 0 || rows <= 0 || cols <= 0) return fail(ctx, DMC_ERR_SIZE, "dmc_chain_batch: bad arguments");
    const dmc_chain_params& p = *pp;
    TRY(check_chain_params(ctx, p));
    if (n_frames == 0) return DMC_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t fpx = (size_t)rows * cols, obytes = fpx * depth_size(chain_out_type(p.chain));
    if (mem == DMC_MEM_DEVICE) {
        // Frames are processed in groups of ~256 MB: large enough that the launch gaps and the partially filled last
        // wave of every kernel are a small share of the launch (per 1000 1080p frames: 32 MB groups 24.7 ms, 64 MB 23.6,
        // 128 MB 23.0, 256 MB 22.7, 512 MB 22.6; L2 residency between stages does not matter, every kernel is
        // instruction-bound), small enough that scratch stays modest (two group-sized buffers).
        uint8_t* out = (uint8_t*)dst;
        ctx->slot[0].stream = ctx->stream;
        if (overlaps(dst, obytes * n_frames, src, fpx * n_frames)) { TRY(reserve(ctx, ctx->slot[0].buf[SB_OUT], obytes * n_frames)); out = (uint8_t*)ctx->slot[0].buf[SB_OUT].p; }
        const int lanes = ctx->lanes < 1 ? 1 : (ctx->lanes > kSlots ? kSlots : ctx->lanes);
        const int group = chunk_frames(env_mib("DMC_GROUP_MB", (size_t)256 << 20) / lanes, fpx, n_frames, 65535, false);
        // lanes > 1: consecutive groups run on different streams so that the tail of one kernel (partially filled last
        // wave) overlaps the head of another group's kernel.  The extra streams are fenced against ctx->stream.
        cudaEvent_t fence = nullptr;
        if (lanes > 1) {
            CUDA_TRY(ctx, cudaEventCreateWithFlags(&fence, cudaEventDisableTiming));
            CUDA_TRY(ctx, cudaEventRecord(fence, ctx->stream));
            for (int l = 1; l < lanes; l++) CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->slot[l].stream, fence, 0));
        }
        int rc = DMC_OK, gi = 0;
        for (int f0 = 0; f0 < n_frames && rc == DMC_OK; f0 += group, gi++) {
            int nf = n_frames - f0 < group ? n_frames - f0 : group;
            rc = run_chain(ctx, ctx->slot[gi % lanes], (const uint8_t*)src + fpx * f0, out + obytes * f0, nf, rows, cols, p);
        }
        if (lanes > 1) {
            for (int l = 1; l < lanes; l++) { cudaEventRecord(fence, ctx->slot[l].stream); cudaStreamWaitEvent(ctx->stream, fence, 0); }
            cudaEventDestroy(fence);
        }
        if (rc != DMC_OK) return rc;
        if ((void*)out != dst) CUDA_TRY(ctx, cudaMemcpyAsync(dst, out, obytes * n_frames, cudaMemcpyDeviceToDevice, ctx->stream));
        return DMC_OK;
    }
    // host: chunked streaming
    const int chunk = chunk_frames(env_mib("DMC_CHUNK_MB", (size_t)48 << 20), fpx, n_frames, 65535, true);   // input bytes per chunk; per 1000 1080p frames host-to-host: 16 MB 42.0, 32 MB 42.5, 48 MB 45.5, 64 MB 45.0, 128 MB 43.5 Gpx/s
    void *din = nullptr, *dout = nullptr;
    return stream_chunks(ctx, n_frames, chunk, ctx->gw.device >= 0, false,
        [&](const Chunk& c) { return reserve_io(ctx, c, fpx * c.nf, obytes * c.nf, c.sl->buf[SB_IN], c.sl->buf[SB_OUT], &din, &dout); },
        [&](const Chunk& c) { return cudaMemcpyAsync(din, (const uint8_t*)src + fpx * c.f0, fpx * c.nf, cudaMemcpyHostToDevice, c.copy); },
        [&](const Chunk& c) { return run_chain(ctx, *c.sl, (const uint8_t*)din, dout, c.nf, rows, cols, p); },
        [&](const Chunk& c) { return cudaMemcpyAsync((uint8_t*)dst + obytes * c.f0, dout, obytes * c.nf, cudaMemcpyDeviceToHost, c.copy); });
}

// The same chain on a batch given as ARRAYS OF IMAGE DESCRIPTORS (frames anywhere in host or device memory, any row step):
// every frame is packed into the slot's dense buffer (H2D or D2D), chunks of frames run through run_chain and are
// unpacked into their own dst -- the slot pipeline of the dense host path, always on this context's own device (frames
// may be device-resident).  Returns when every dst is valid.
int dmc_chain_batch_images(dmc_ctx* ctx, const dmc_image* srcs, dmc_image* dsts, int n_frames, const dmc_chain_params* pp) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    if (!srcs || !dsts || !pp || n_frames < 0) return fail(ctx, DMC_ERR_ARG, "dmc_chain_batch_images: bad arguments");
    const dmc_chain_params& p = *pp;
    TRY(check_chain_params(ctx, p));
    if (n_frames == 0) return DMC_OK;
    const int rows = srcs[0].rows, cols = srcs[0].cols, otype = chain_out_type(p.chain);
    for (int i = 0; i < n_frames; i++) {
        TRY(check_image(ctx, &srcs[i], "src")); TRY(check_image(ctx, &dsts[i], "dst"));
        if (srcs[i].cvtype != DMC_8U) return fail(ctx, DMC_ERR_TYPE, "PostFilterSet: src must be CV_8UC1");
        if (dsts[i].cvtype != otype) return fail(ctx, DMC_ERR_TYPE, "PostFilterSet: dst has the wrong type for this entry point");
        if (srcs[i].rows != rows || srcs[i].cols != cols || dsts[i].rows != rows || dsts[i].cols != cols) return fail(ctx, DMC_ERR_SIZE, "dmc_chain_batch_images: all frames must have one size");
    }
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t fpx = (size_t)rows * cols, obytes = fpx * depth_size(otype), orow = (size_t)cols * depth_size(otype);
    const int chunk = chunk_frames((size_t)48 << 20, fpx, n_frames, 65535, true);
    void *din = nullptr, *dout = nullptr;
    return stream_chunks(ctx, n_frames, chunk, false, false,
        [&](const Chunk& c) { return reserve_io(ctx, c, fpx * c.nf, obytes * c.nf, c.sl->buf[SB_IN], c.sl->buf[SB_OUT], &din, &dout); },
        [&](const Chunk& c) {
            cudaError_t e = cudaSuccess;
            for (int i = 0; i < c.nf && e == cudaSuccess; i++) {
                const dmc_image& im = srcs[c.f0 + i];
                e = cudaMemcpy2DAsync((uint8_t*)din + fpx * i, cols, im.data, step_of(&im), cols, rows,
                                      im.mem == DMC_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, c.copy);
            }
            return e;
        },
        [&](const Chunk& c) { return run_chain(ctx, *c.sl, (const uint8_t*)din, dout, c.nf, rows, cols, p); },
        [&](const Chunk& c) {
            cudaError_t e = cudaSuccess;
            for (int i = 0; i < c.nf && e == cudaSuccess; i++) {
                const dmc_image& im = dsts[c.f0 + i];
                e = cudaMemcpy2DAsync(im.data, step_of(&im), (uint8_t*)dout + obytes * i, orow, orow, rows,
                                      im.mem == DMC_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, c.copy);
            }
            return e;
        });
}

// ---- frame-batch scheduler across the GPUs of one box ---------------------------------------------------------------
// One context per listed device, kept alive between runs (device buffers, streams); every run cuts the batch into
// contiguous shards (dmc_shard_frames) and streams each shard through its device on its own host thread with
// dmc_chain_batch (its slot pipeline of H2D / kernels / D2H).  Frames are independent: no exchange between devices.
struct dmc_sched {
    std::vector<dmc_ctx*> ctxs;
    std::string err;
    dmc_hostlink_info link;        // measured at creation (n_devices == 0: not probed)
};

int dmc_sched_create(const int* devices, int n_devices, dmc_sched** out) {
    if (!out) return DMC_ERR_ARG;
    DeviceGuard keep_device;
    *out = nullptr;
    if (!devices || n_devices <= 0) return fail(nullptr, DMC_ERR_ARG, "dmc_sched_create: no devices");
    if (n_devices > DMC_MAX_DEVICES) return fail(nullptr, DMC_ERR_ARG, "dmc_sched_create: too many devices");
    dmc_sched* sc = new dmc_sched();
    memset(&sc->link, 0, sizeof sc->link);
    // Which links are worth using?  Measured once, here, while the devices are idle (see dmc_hostlink_probe).
    if (n_devices > 1 && !getenv("DMC_NO_TOPOLOGY") && dmc_hostlink_probe(devices, n_devices, &sc->link) != DMC_OK) memset(&sc->link, 0, sizeof sc->link);
    for (int i = 0; i < n_devices; i++) {
        dmc_ctx* c = nullptr;
        int rc = dmc_create(devices[i], &c);
        if (rc != DMC_OK) { for (auto x : sc->ctxs) dmc_destroy(x); delete sc; return rc; }
        sc->ctxs.push_back(c);
        if (sc->link.n_devices == n_devices && sc->link.gateway[i] != devices[i] && dmc_set_gateway(c, sc->link.gateway[i]) != DMC_OK) sc->link.gateway[i] = devices[i];
    }
    *out = sc;
    return DMC_OK;
}

int dmc_sched_get_routing(const dmc_sched* sc, int* gateways, double* all_gbs, double* best_gbs) {
    if (!sc) return DMC_ERR_ARG;
    for (size_t i = 0; i < sc->ctxs.size(); i++) if (gateways) gateways[i] = sc->ctxs[i]->gw.device;
    if (all_gbs) *all_gbs = sc->link.all_gbs;
    if (best_gbs) *best_gbs = sc->link.best_gbs;
    return DMC_OK;
}

void dmc_sched_destroy(dmc_sched* sc) {
    if (!sc) return;
    DeviceGuard keep_device;
    for (auto c : sc->ctxs) dmc_destroy(c);
    delete sc;
}

const char* dmc_sched_last_error(const dmc_sched* sc) { return sc ? sc->err.c_str() : g_err.c_str(); }
int dmc_sched_device_count(const dmc_sched* sc) { return sc ? (int)sc->ctxs.size() : 0; }

int dmc_sched_chain_batch(dmc_sched* sc, const void* src, void* dst, int n_frames, int rows, int cols, const dmc_chain_params* p) {
    if (!sc) return fail(nullptr, DMC_ERR_ARG, "null scheduler");
    if (!src || !dst || !p || n_frames < 0 || rows <= 0 || cols <= 0) { sc->err = "dmc_sched_chain_batch: bad arguments"; return DMC_ERR_ARG; }
    const int nd = (int)sc->ctxs.size();
    const size_t fpx = (size_t)rows * cols, obytes = fpx * depth_size(chain_out_type(p->chain));
    std::vector<int> rcs(nd, DMC_OK);
    std::vector<std::thread> workers;
    for (int i = 0; i < nd; i++)
        workers.emplace_back([&, i]() {
            int begin = 0, count = 0;
            dmc_shard_frames(n_frames, i, nd, &begin, &count);
            if (count > 0) rcs[i] = dmc_chain_batch(sc->ctxs[i], (const uint8_t*)src + fpx * begin, (uint8_t*)dst + obytes * begin, count, rows, cols, p, DMC_MEM_HOST);
        });
    for (auto& w : workers) w.join();
    for (int i = 0; i < nd; i++) if (rcs[i] != DMC_OK) { sc->err = dmc_last_error(sc->ctxs[i]); return rcs[i]; }
    return DMC_OK;
}

// Convenience: create the scheduler, run once, destroy it.
int dmc_multi_chain_batch(const int* devices, int n_devices, const void* src, void* dst, int n_frames, int rows, int cols,
                          const dmc_chain_params* p, char* err, size_t err_len) {
    auto set_err = [&](const std::string& m) { if (err && err_len) { strncpy(err, m.c_str(), err_len - 1); err[err_len - 1] = 0; } };
    dmc_sched* sc = nullptr;
    int rc = dmc_sched_create(devices, n_devices, &sc);
    if (rc != DMC_OK) { set_err(dmc_last_error(nullptr)); return rc; }
    rc = dmc_sched_chain_batch(sc, src, dst, n_frames, rows, cols, p);
    if (rc != DMC_OK) set_err(sc->err);
    dmc_sched_destroy(sc);
    return rc;
}

// ---- JPEG decode feeding the chain (SURVEY.md 8f-1) -----------------------------------------------------------------
namespace {

// Host side of one group of streams: parsed descriptors + de-duplicated tables, packed into ONE metadata block so that a
// single H2D copy brings everything the kernels need besides the bitstreams themselves.  The block is
// [FrameDesc...][HuffTable...][QuantTable...] with 16-byte aligned parts; o_huff and o_quant are the tables' offsets.
struct JpegGroup {
    std::vector<dmcjpeg::FrameDesc> desc; std::vector<dmcjpeg::QuantTable> qpool; std::vector<dmcjpeg::HuffTable> hpool;
    size_t scratch_bytes = 0; int n_restart = 0;
    size_t o_huff = 0, o_quant = 0, meta_bytes = 0;
};

void jpeg_write_meta(const JpegGroup& g, void* block) {
    memcpy(block, g.desc.data(), g.desc.size() * sizeof(dmcjpeg::FrameDesc));
    memcpy((char*)block + g.o_huff, g.hpool.data(), g.hpool.size() * sizeof(dmcjpeg::HuffTable));
    memcpy((char*)block + g.o_quant, g.qpool.data(), g.qpool.size() * sizeof(dmcjpeg::QuantTable));
}

// Parses streams [f0, f0 + nf) of the blob; scan offsets are relative to `blob_base` (the first byte that will be copied).
int jpeg_parse_group(dmc_ctx* ctx, const uint8_t* blob, const uint64_t* offsets, int f0, int nf, uint64_t blob_base, int rows, int cols, JpegGroup* g) {
    g->desc.resize(nf); g->qpool.clear(); g->hpool.clear(); g->scratch_bytes = 0; g->n_restart = 0;
    for (int i = 0; i < nf; i++) {
        const uint64_t o = offsets[f0 + i], e = offsets[f0 + i + 1];
        if (e < o || o < blob_base) return fail(ctx, DMC_ERR_ARG, "JPEG batch: offsets must be non-decreasing");
        std::string why = jpeg_parse_frame(blob + o, e - o, o - blob_base, rows, cols, g->qpool, g->hpool, &g->desc[i]);
        if (!why.empty()) return fail(ctx, DMC_ERR_TYPE, "JPEG frame " + std::to_string(f0 + i) + ": " + why);
        if (g->desc[i].scan_end - g->desc[i].scan_offset >= (1ull << 28)) return fail(ctx, DMC_ERR_SIZE, "JPEG frame " + std::to_string(f0 + i) + ": scan larger than 256 MB");
        g->desc[i].ds_offset = g->scratch_bytes;
        g->scratch_bytes += jpeg_scratch_bytes(g->desc[i].scan_end - g->desc[i].scan_offset);
        if (g->desc[i].restart_interval) g->n_restart++;
    }
    g->o_huff = (g->desc.size() * sizeof(dmcjpeg::FrameDesc) + 15) & ~(size_t)15;
    g->o_quant = (g->o_huff + g->hpool.size() * sizeof(dmcjpeg::HuffTable) + 15) & ~(size_t)15;
    g->meta_bytes = g->o_quant + g->qpool.size() * sizeof(dmcjpeg::QuantTable);
    return DMC_OK;
}

}  // namespace

// Streamed bitstream -> chain: the reference's pointcloudTest loop (main.cpp:276-303: JPEG decode, then the filter set) for
// a whole batch.  Chunks of frames flow through the kSlots pipeline slots: the host parses the chunk's headers into the
// slot's pinned staging block, the bitstreams go H2D straight from the caller's blob (about 1/30 of the decoded bytes), one
// launch decodes every frame of the chunk (one CTA per frame), the chain runs on the decoded frames without leaving the
// device and the result is copied out; no host synchronisation except when a slot comes round again.  With a gateway
// (dmc_set_gateway) the bitstreams and the results travel over the gateway's link, as in dmc_chain_batch.
int dmc_chain_batch_jpeg(dmc_ctx* ctx, const void* blob, const uint64_t* offsets, int n_frames, int rows, int cols, void* dst, int dst_mem,
                         const dmc_chain_params* pp) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    if (!blob || !offsets || !dst || !pp || n_frames < 0 || rows <= 0 || cols <= 0 || rows > 65535 || cols > 65535) return fail(ctx, DMC_ERR_SIZE, "dmc_chain_batch_jpeg: bad arguments");
    const dmc_chain_params& p = *pp;
    TRY(check_chain_params(ctx, p));
    if (n_frames == 0) return DMC_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t fpx = (size_t)rows * cols, obytes = fpx * depth_size(chain_out_type(p.chain)), blocks = (size_t)((rows + 7) / 8) * ((cols + 7) / 8);
    const int chunk = chunk_frames(env_mib("DMC_CHUNK_MB", (size_t)128 << 20), fpx, n_frames, 4096, true);   // decoded bytes per chunk: enough frames (one CTA each) to fill the SMs together with the neighbouring slots
    const bool host_out = dst_mem == DMC_MEM_HOST;
    JpegGroup g;
    uint64_t b0 = 0, b1 = 0;
    void *dblob = nullptr, *dout = nullptr;
    return stream_chunks(ctx, n_frames, chunk, ctx->gw.device >= 0, true,
        [&](const Chunk& c) -> int {
            Slot& sl = *c.sl;
            b0 = offsets[c.f0]; b1 = offsets[c.f0 + c.nf];
            if (b1 < b0) return fail(ctx, DMC_ERR_ARG, "dmc_chain_batch_jpeg: offsets must be non-decreasing");
            TRY(jpeg_parse_group(ctx, (const uint8_t*)blob, offsets, c.f0, c.nf, b0, rows, cols, &g));
            if (sl.hcap < g.meta_bytes) {
                if (sl.hstage) cudaFreeHost(sl.hstage);
                sl.hstage = nullptr; sl.hcap = 0;
                const size_t cap = (g.meta_bytes * 2 + 65535) & ~(size_t)65535;
                if (cudaHostAlloc(&sl.hstage, cap, cudaHostAllocDefault) != cudaSuccess) return fail(ctx, DMC_ERR_CUDA, "cudaHostAlloc (JPEG metadata staging)");
                sl.hcap = cap;
            }
            jpeg_write_meta(g, sl.hstage);
            // bitstreams and results on the device whose link carries them, everything else local
            TRY(reserve_io(ctx, c, (size_t)(b1 - b0) + 16, host_out ? obytes * c.nf : 0, sl.buf[SB_BITS], sl.buf[SB_OUT], &dblob, &dout));
            if (!host_out) dout = (uint8_t*)dst + obytes * c.f0;
            TRY(reserve(ctx, sl.buf[SB_IN], fpx * c.nf));
            TRY(reserve(ctx, sl.buf[SB_META], g.meta_bytes));
            TRY(reserve(ctx, sl.buf[SB_SCANS], g.scratch_bytes + 16));
            if (g.n_restart) TRY(reserve(ctx, sl.buf[SB_COEF], (size_t)c.nf * blocks * 64 * sizeof(int16_t)));
            return DMC_OK;
        },
        [&](const Chunk& c) { return cudaMemcpyAsync(dblob, (const uint8_t*)blob + b0, (size_t)(b1 - b0), cudaMemcpyHostToDevice, c.copy); },
        [&](const Chunk& c) -> int {
            Slot& sl = *c.sl;
            cudaError_t e = cudaMemcpyAsync(sl.buf[SB_META].p, sl.hstage, g.meta_bytes, cudaMemcpyHostToDevice, sl.stream);
            if (e != cudaSuccess) return fail(ctx, DMC_ERR_CUDA, cudaGetErrorString(e));
            const char* dm = (const char*)sl.buf[SB_META].p;
            LAUNCH(ctx, launch_jpeg_decode((const uint8_t*)dblob, dm, dm + g.o_huff, dm + g.o_quant, (uint8_t*)sl.buf[SB_SCANS].p, (int16_t*)sl.buf[SB_COEF].p,
                                           (uint8_t*)sl.buf[SB_IN].p, c.nf, g.n_restart, rows, cols, sl.stream));
            return run_chain(ctx, sl, (const uint8_t*)sl.buf[SB_IN].p, dout, c.nf, rows, cols, p);
        },
        [&](const Chunk& c) { return host_out ? cudaMemcpyAsync((uint8_t*)dst + obytes * c.f0, dout, obytes * c.nf, cudaMemcpyDeviceToHost, c.copy) : cudaSuccess; });
}

int dmc_jpeg_probe(const void* stream, size_t len, int* rows, int* cols, char* err, size_t err_len) {
    std::vector<dmcjpeg::QuantTable> qp; std::vector<dmcjpeg::HuffTable> hp; dmcjpeg::FrameDesc d;
    int r = 0, c = 0;
    std::string why = stream ? jpeg_parse_frame((const uint8_t*)stream, len, 0, -1, -1, qp, hp, &d, &r, &c) : std::string("null stream");
    if (rows) *rows = r;
    if (cols) *cols = c;
    if (err && err_len) { strncpy(err, why.c_str(), err_len - 1); err[err_len - 1] = 0; }
    return why.empty() ? DMC_OK : DMC_ERR_TYPE;
}

int dmc_jpeg_decode_gray_batch(dmc_ctx* ctx, const void* blob, const uint64_t* offsets, int n_frames, int rows, int cols, void* dst, int dst_mem) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    if (!blob || !offsets || !dst || n_frames < 0 || rows <= 0 || cols <= 0 || rows > 65535 || cols > 65535) return fail(ctx, DMC_ERR_SIZE, "dmc_jpeg_decode_gray_batch: bad arguments");
    if (n_frames == 0) return DMC_OK;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const size_t fpx = (size_t)rows * cols, blocks = (size_t)((rows + 7) / 8) * ((cols + 7) / 8);
    const int group_max = 2048;
    JpegGroup g;
    std::vector<char> meta;
    for (int f0 = 0; f0 < n_frames; f0 += group_max) {
        const int nf = n_frames - f0 < group_max ? n_frames - f0 : group_max;
        const uint64_t b0 = offsets[f0], b1 = offsets[f0 + nf];
        if (b1 < b0) return fail(ctx, DMC_ERR_ARG, "dmc_jpeg_decode_gray_batch: offsets must be non-decreasing");
        TRY(jpeg_parse_group(ctx, (const uint8_t*)blob, offsets, f0, nf, b0, rows, cols, &g));
        TRY(reserve(ctx, ctx->jpeg[JD_BITS], (size_t)(b1 - b0) + 16));
        TRY(reserve(ctx, ctx->jpeg[JD_META], g.meta_bytes));
        if (g.n_restart) TRY(reserve(ctx, ctx->jpeg[JD_COEF], (size_t)nf * blocks * 64 * sizeof(int16_t)));
        TRY(reserve(ctx, ctx->jpeg[JD_SCANS], g.scratch_bytes + 16));
        uint8_t* out = (uint8_t*)dst + fpx * f0;
        if (dst_mem == DMC_MEM_HOST) { TRY(reserve(ctx, ctx->jpeg[JD_OUT], fpx * nf)); out = (uint8_t*)ctx->jpeg[JD_OUT].p; }
        meta.resize(g.meta_bytes);
        jpeg_write_meta(g, meta.data());
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->jpeg[JD_BITS].p, (const uint8_t*)blob + b0, (size_t)(b1 - b0), cudaMemcpyHostToDevice, s));
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->jpeg[JD_META].p, meta.data(), g.meta_bytes, cudaMemcpyHostToDevice, s));
        const char* dm = (const char*)ctx->jpeg[JD_META].p;
        LAUNCH(ctx, launch_jpeg_decode((const uint8_t*)ctx->jpeg[JD_BITS].p, dm, dm + g.o_huff, dm + g.o_quant, (uint8_t*)ctx->jpeg[JD_SCANS].p, (int16_t*)ctx->jpeg[JD_COEF].p,
                                       out, nf, g.n_restart, rows, cols, s));
        if (dst_mem == DMC_MEM_HOST) CUDA_TRY(ctx, cudaMemcpyAsync((uint8_t*)dst + fpx * f0, out, fpx * nf, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(ctx, cudaStreamSynchronize(s));     // the pageable metadata block is reused by the next group
    }
    return DMC_OK;
}

// ---- JPEG encode (SURVEY.md 8f-5) ------------------------------------------------------------------------------------
int dmc_jpeg_encode_bound(int rows, int cols, uint64_t* bytes) {
    if (!bytes) return fail(nullptr, DMC_ERR_ARG, "dmc_jpeg_encode_bound: null bytes");
    if (rows <= 0 || cols <= 0 || rows > 65535 || cols > 65535) return fail(nullptr, DMC_ERR_SIZE, "JPEG encode: frame size must be 1..65535 x 1..65535");
    *bytes = dmcjpeg::jpeg_encode_bound(rows, cols);
    if (*bytes > dmcjpeg::kEncMaxStreamBytes) return fail(nullptr, DMC_ERR_SIZE, "JPEG encode: the worst-case stream of a " + std::to_string(rows) + " x " + std::to_string(cols) + " frame exceeds 256 MB");
    return DMC_OK;
}

namespace {

// Scratch of all frames of one group; the group is as large as this allows (at least one frame, at most 2048).  A 1080p
// frame needs about 26 MB (slot 13.4 MB, scan words 6.7 MB, coefficients 4.1 MB, staged frame).
constexpr size_t kEncGroupBytes = (size_t)4 << 30;

enum { JE_TABS, JE_SRC, JE_COEF, JE_INFO, JE_WORDS, JE_SLOTS, JE_LENS, JE_OUT, JE_DEC };

// Checks the arguments shared by the encode entry points, uploads the encoder tables and returns the group size.
int jpeg_enc_prepare(dmc_ctx* ctx, const char* what, int rows, int cols, int quality, int mem_a, int mem_b, int* group) {
    if (quality < 0 || quality > 100) return fail(ctx, DMC_ERR_ARG, std::string(what) + ": quality must be in 0..100");
    if ((mem_a != DMC_MEM_HOST && mem_a != DMC_MEM_DEVICE) || (mem_b != DMC_MEM_HOST && mem_b != DMC_MEM_DEVICE)) return fail(ctx, DMC_ERR_ARG, std::string(what) + ": bad mem");
    uint64_t bound;
    if (dmc_jpeg_encode_bound(rows, cols, &bound) != DMC_OK) return fail(ctx, DMC_ERR_SIZE, std::string(what) + ": " + g_err);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const JpegEncLayout l = jpeg_enc_layout(rows, cols);
    const size_t per = l.coef_bytes + l.info_bytes + l.word_bytes + l.slot_bytes + 2 * (size_t)rows * cols;
    *group = chunk_frames(kEncGroupBytes, per, INT_MAX, 2048, false);
    dmcjpeg::EncTables t;
    dmcjpeg::make_enc_tables(quality, rows, cols, &t);
    TRY(reserve(ctx, ctx->jpeg_enc[JE_TABS], sizeof t));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->jpeg_enc[JE_TABS].p, &t, sizeof t, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));          // (t lives on this stack frame)
    return DMC_OK;
}

// Encodes frames [f0, f0 + nf) of src into the slots (lengths in JE_LENS); desc: also write the decoder's FrameDescs there.
int jpeg_enc_group(dmc_ctx* ctx, const uint8_t* src, int src_mem, int f0, int nf, int rows, int cols, void* desc) {
    cudaStream_t s = ctx->stream;
    const size_t fpx = (size_t)rows * cols;
    const JpegEncLayout l = jpeg_enc_layout(rows, cols);
    const uint8_t* dsrc = src + fpx * f0;
    if (src_mem == DMC_MEM_HOST) {
        TRY(reserve(ctx, ctx->jpeg_enc[JE_SRC], fpx * nf));
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->jpeg_enc[JE_SRC].p, dsrc, fpx * nf, cudaMemcpyHostToDevice, s));
        dsrc = (const uint8_t*)ctx->jpeg_enc[JE_SRC].p;
    }
    TRY(reserve(ctx, ctx->jpeg_enc[JE_COEF], l.coef_bytes * nf));
    TRY(reserve(ctx, ctx->jpeg_enc[JE_INFO], l.info_bytes * nf));
    TRY(reserve(ctx, ctx->jpeg_enc[JE_WORDS], l.word_bytes * nf));
    TRY(reserve(ctx, ctx->jpeg_enc[JE_SLOTS], l.slot_bytes * nf));
    TRY(reserve(ctx, ctx->jpeg_enc[JE_LENS], (size_t)nf * (sizeof(uint32_t) + sizeof(uint64_t)) + 16));
    LAUNCH(ctx, launch_jpeg_encode(dsrc, ctx->jpeg_enc[JE_TABS].p, ctx->jpeg_enc[JE_COEF].p, ctx->jpeg_enc[JE_INFO].p, ctx->jpeg_enc[JE_WORDS].p,
                                   (uint8_t*)ctx->jpeg_enc[JE_SLOTS].p, (uint32_t*)ctx->jpeg_enc[JE_LENS].p, desc, nf, rows, cols, s));
    return DMC_OK;
}

uint64_t* enc_offs(dmc_ctx* ctx, int nf) { return (uint64_t*)((char*)ctx->jpeg_enc[JE_LENS].p + (((size_t)nf * sizeof(uint32_t) + 15) & ~(size_t)15)); }

}  // namespace

// Streams are encoded group by group into per-frame slots on the device; the host reads the group's lengths back, places
// the streams back to back after the previous group's and a gather kernel copies them there (through a device staging
// buffer and one copy for a host blob).
int dmc_jpeg_encode_gray_batch(dmc_ctx* ctx, const void* src, int src_mem, int n_frames, int rows, int cols, int quality, void* blob, int blob_mem,
                               uint64_t capacity, uint64_t* offsets) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    if (!offsets || n_frames < 0 || (n_frames > 0 && (!src || !blob))) return fail(ctx, DMC_ERR_SIZE, "dmc_jpeg_encode_gray_batch: bad arguments");
    int group;
    TRY(jpeg_enc_prepare(ctx, "dmc_jpeg_encode_gray_batch", rows, cols, quality, src_mem, blob_mem, &group));
    offsets[0] = 0;
    cudaStream_t s = ctx->stream;
    const JpegEncLayout l = jpeg_enc_layout(rows, cols);
    std::vector<uint32_t> lens; std::vector<uint64_t> offs;
    for (int f0 = 0; f0 < n_frames; f0 += group) {
        const int nf = n_frames - f0 < group ? n_frames - f0 : group;
        TRY(jpeg_enc_group(ctx, (const uint8_t*)src, src_mem, f0, nf, rows, cols, nullptr));
        lens.resize(nf); offs.resize(nf);
        CUDA_TRY(ctx, cudaMemcpyAsync(lens.data(), ctx->jpeg_enc[JE_LENS].p, nf * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(ctx, cudaStreamSynchronize(s));
        const uint64_t base = offsets[f0];
        uint64_t end = base, longest = 0;
        for (int i = 0; i < nf; i++) { offs[i] = end - base; end += lens[i]; if (lens[i] > longest) longest = lens[i]; }
        if (end > capacity)
            return fail(ctx, DMC_ERR_SIZE, "dmc_jpeg_encode_gray_batch: the streams of frames 0.." + std::to_string(f0 + nf - 1) + " need " + std::to_string(end) +
                                               " bytes, capacity is " + std::to_string(capacity));
        for (int i = 0; i < nf; i++) offsets[f0 + i + 1] = base + offs[i] + lens[i];
        uint64_t* d_offs = enc_offs(ctx, nf);
        CUDA_TRY(ctx, cudaMemcpyAsync(d_offs, offs.data(), nf * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
        uint8_t* dst = (uint8_t*)blob + base;
        if (blob_mem == DMC_MEM_HOST) { TRY(reserve(ctx, ctx->jpeg_enc[JE_OUT], end - base)); dst = (uint8_t*)ctx->jpeg_enc[JE_OUT].p; }
        LAUNCH(ctx, launch_jpeg_enc_gather((const uint8_t*)ctx->jpeg_enc[JE_SLOTS].p, l.slot_bytes, (const uint32_t*)ctx->jpeg_enc[JE_LENS].p, d_offs, dst, nf, longest, s));
        if (blob_mem == DMC_MEM_HOST) CUDA_TRY(ctx, cudaMemcpyAsync((uint8_t*)blob + base, dst, end - base, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(ctx, cudaStreamSynchronize(s));     // offs is reused by the next group
    }
    return DMC_OK;
}

// The reference's degradeJPEG on the device: encode into the slots, then decode every slot in place with the decoder of
// dmc_jpeg_decode_gray_batch.  The decoder's tables come from parsing the encoder's header once; the encoder writes each
// frame's FrameDesc itself, so the streams never leave the device.
int dmc_jpeg_degrade_gray_batch(dmc_ctx* ctx, const void* src, void* dst, int n_frames, int rows, int cols, int quality, int mem, uint64_t* bytes) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    if (n_frames < 0 || (n_frames > 0 && (!src || !dst))) return fail(ctx, DMC_ERR_SIZE, "dmc_jpeg_degrade_gray_batch: bad arguments");
    int group;
    TRY(jpeg_enc_prepare(ctx, "dmc_jpeg_degrade_gray_batch", rows, cols, quality, mem, mem, &group));
    if (n_frames == 0) return DMC_OK;
    cudaStream_t s = ctx->stream;
    const size_t fpx = (size_t)rows * cols;
    // decoder tables: [DC, AC Huffman tables][quantisation table][FrameDesc per frame]
    dmcjpeg::EncTables t;
    dmcjpeg::make_enc_tables(quality, rows, cols, &t);
    std::vector<dmcjpeg::QuantTable> qpool; std::vector<dmcjpeg::HuffTable> hpool; dmcjpeg::FrameDesc hd;
    const std::string why = jpeg_parse_frame(t.header, dmcjpeg::kEncHeaderBytes, 0, rows, cols, qpool, hpool, &hd);
    if (!why.empty() || hpool.size() != 2 || qpool.size() != 1 || hd.dc != 0 || hd.ac != 1 || hd.qt != 0)
        return fail(ctx, DMC_ERR_TYPE, "dmc_jpeg_degrade_gray_batch: encoder header does not parse: " + why);
    const size_t o_q = 2 * sizeof(dmcjpeg::HuffTable), o_desc = (o_q + sizeof(dmcjpeg::QuantTable) + 15) & ~(size_t)15;
    TRY(reserve(ctx, ctx->jpeg_enc[JE_DEC], o_desc + (size_t)group * sizeof(dmcjpeg::FrameDesc)));
    char* dm = (char*)ctx->jpeg_enc[JE_DEC].p;
    CUDA_TRY(ctx, cudaMemcpyAsync(dm, hpool.data(), 2 * sizeof(dmcjpeg::HuffTable), cudaMemcpyHostToDevice, s));
    CUDA_TRY(ctx, cudaMemcpyAsync(dm + o_q, qpool.data(), sizeof(dmcjpeg::QuantTable), cudaMemcpyHostToDevice, s));
    std::vector<uint32_t> lens;
    for (int f0 = 0; f0 < n_frames; f0 += group) {
        const int nf = n_frames - f0 < group ? n_frames - f0 : group;
        TRY(jpeg_enc_group(ctx, (const uint8_t*)src, mem, f0, nf, rows, cols, dm + o_desc));
        uint8_t* out = (uint8_t*)dst + fpx * f0;
        if (mem == DMC_MEM_HOST) { TRY(reserve(ctx, ctx->jpeg_enc[JE_OUT], fpx * nf)); out = (uint8_t*)ctx->jpeg_enc[JE_OUT].p; }
        LAUNCH(ctx, launch_jpeg_decode((const uint8_t*)ctx->jpeg_enc[JE_SLOTS].p, dm + o_desc, dm, dm + o_q, (uint8_t*)ctx->jpeg_enc[JE_WORDS].p, nullptr, out,
                                       nf, 0, rows, cols, s));
        if (mem == DMC_MEM_HOST) CUDA_TRY(ctx, cudaMemcpyAsync((uint8_t*)dst + fpx * f0, out, fpx * nf, cudaMemcpyDeviceToHost, s));
        if (bytes) {
            lens.resize(nf);
            CUDA_TRY(ctx, cudaMemcpyAsync(lens.data(), ctx->jpeg_enc[JE_LENS].p, nf * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        }
        CUDA_TRY(ctx, cudaStreamSynchronize(s));
        if (bytes) for (int i = 0; i < nf; i++) bytes[f0 + i] = lens[i];
    }
    return DMC_OK;
}

// ---- stand-alone operators ---------------------------------------------------------------------------------------
int dmc_bwrf(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int kw, int kh, float threshold, int method, int border_type) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, src, "src")); TRY(check_image(ctx, dst, "dst"));
    if (border_type != DMC_BORDER_REPLICATE) return fail(ctx, DMC_ERR_ARG, "binalyWeightedRangeFilter: only BORDER_REPLICATE is supported");
    if (kw < 0 || kh < 0 || (kw >> 1) > DMC_MAX_RADIUS || (kh >> 1) > DMC_MAX_RADIUS) return fail(ctx, DMC_ERR_ARG, "binalyWeightedRangeFilter: kernel size out of range");
    const int depth = cv_depth(src->cvtype), cn = cv_cn(src->cvtype);
    // dispatcher :1106-1178: which (type, method) pairs do anything at all
    bool runs = false;
    if (method == DMC_FULL_KERNEL) runs = depth == DMC_8U || depth == DMC_16S || depth == DMC_16U || depth == DMC_32F;
    else if (method == DMC_FULL_KERNEL_PAIR) runs = depth == DMC_16S || depth == DMC_16U || depth == DMC_32F;
    else if (method == DMC_SEPARABLE_KERNEL) runs = depth == DMC_8U || depth == DMC_32F;
    if (!runs) return DMC_UNSUPPORTED;
    if (cn != 1 && cn != 3) return fail(ctx, DMC_ERR_TYPE, "binalyWeightedRangeFilter: CV_Assert(type is C1 or C3)");   // :1038 / :985
    if (dst->cvtype != src->cvtype || dst->rows != src->rows || dst->cols != src->cols) return fail(ctx, DMC_ERR_TYPE, "binalyWeightedRangeFilter: CV_Assert(src.type()==dst.type() && src.size()==dst.size())");
    const void* in; void* out;
    TRY(stage_op(ctx, src, dst, &in, &out));
    const cudaStream_t s = ctx->stream;
    Buf& ftmp = ctx->slot[0].buf[SB_FLOAT];
    const int H = src->rows, W = src->cols;
    int rc;
    if (depth == DMC_8U) rc = range_filter_8u(ctx, (const uint8_t*)in, (uint8_t*)out, ftmp, 1, H, W, cn, kw, kh, threshold, method, s);
    else {
        int lop = depth == DMC_32F ? LOAD_F32 : depth == DMC_16U ? LOAD_U16 : LOAD_S16;
        int sop = depth == DMC_32F ? STORE_F32 : depth == DMC_16U ? STORE_U16 : STORE_S16;
        if (method == DMC_SEPARABLE_KERNEL && kw <= 1) {          // SP_32f: src.copyTo(dst) and nothing else
            TRY(copy_unless_same(ctx, out, in, image_bytes(src), s));
            rc = DMC_OK;
        } else if (method == DMC_SEPARABLE_KERNEL && kh == 0) {  // vertical pass with height 0 copies
            RowSpan rh = make_rowspan(kw, 1);
            rc = DMC_OK; LAUNCH(ctx, launch_bwrf32f(in, out, 1, H, W, cn, rh, threshold, lop, 0.f, sop, s));
        } else rc = range_filter_32f(ctx, in, out, ftmp, 1, H, W, cn, kw, kh, threshold, method, lop, 0.f, sop, s);
    }
    if (rc != DMC_OK) { cudaStreamSynchronize(s); return rc; }
    return stage_out_end(ctx, dst, out, s);
}

int dmc_joint_bwrf(dmc_ctx* ctx, const dmc_image* src, const dmc_image* guide, dmc_image* dst, int kw, int kh, float threshold, int method) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, src, "src")); TRY(check_image(ctx, guide, "guide")); TRY(check_image(ctx, dst, "dst"));
    if (method != DMC_FULL_KERNEL) return fail(ctx, DMC_ERR_ARG, "jointBinalyWeightedRangeFilter: only FULL_KERNEL is defined");
    if (kw < 0 || kh < 0 || (kw >> 1) > DMC_MAX_RADIUS || (kh >> 1) > DMC_MAX_RADIUS) return fail(ctx, DMC_ERR_ARG, "jointBinalyWeightedRangeFilter: kernel size out of range");
    if (src->cvtype != DMC_8U) return fail(ctx, DMC_ERR_TYPE, "jointBinalyWeightedRangeFilter: src must be CV_8UC1");
    const int gcn = cv_cn(guide->cvtype);
    if (cv_depth(guide->cvtype) != DMC_8U || (gcn != 1 && gcn != 3)) return fail(ctx, DMC_ERR_TYPE, "jointBinalyWeightedRangeFilter: guide must be CV_8UC1 or CV_8UC3");
    if (guide->rows != src->rows || guide->cols != src->cols) return fail(ctx, DMC_ERR_SIZE, "jointBinalyWeightedRangeFilter: guide size != src size");
    if (dst->cvtype != src->cvtype || dst->rows != src->rows || dst->cols != src->cols) return fail(ctx, DMC_ERR_TYPE, "jointBinalyWeightedRangeFilter: dst must match src");
    const void* in; const void* gd; void* out;
    TRY(stage_op(ctx, src, dst, &in, &out));
    const cudaStream_t s = ctx->stream;
    Buf& bout = ctx->slot[0].buf[SB_OUT];
    TRY(stage_in(ctx, guide, ctx->slot[0].buf[SB_PING], s, &gd));
    if (out != bout.p && overlaps(out, image_bytes(dst), gd, image_bytes(guide))) { TRY(reserve(ctx, bout, image_bytes(dst))); out = bout.p; }      // dst aliases the guide
    const int H = src->rows, W = src->cols;
    int rc = DMC_OK;
    if (kw == 0 || kh == 0) TRY(copy_unless_same(ctx, out, in, image_bytes(src), s));
    else {
        RowSpan rs = make_rowspan(kw, kh);
        int nk = launch_joint_bwrf8u((const uint8_t*)in, (const uint8_t*)gd, (uint8_t*)out, 1, H, W, gcn, rs, (int)(uint8_t)(int)threshold, s);
        if (!nk) rc = fail(ctx, DMC_ERR_ARG, "jointBinalyWeightedRangeFilter: unsupported configuration"); else rc = after_launch(ctx, nk);
    }
    if (rc != DMC_OK) { cudaStreamSynchronize(s); return rc; }
    return stage_out_end(ctx, dst, out, s);
}

int dmc_blur_remove_minmax(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int r) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, src, "src")); TRY(check_image(ctx, dst, "dst")); TRY(check_radius(ctx, r, "r"));
    const int depth = cv_depth(src->cvtype), cn = cv_cn(src->cvtype);
    if (dst->cvtype != src->cvtype || dst->rows != src->rows || dst->cols != src->cols) return fail(ctx, DMC_ERR_SIZE, "blurRemoveMinMax: dst must match src");
    const void* in; void* out;
    TRY(stage_op(ctx, src, dst, &in, &out));
    const cudaStream_t s = ctx->stream;
    const bool known = depth == DMC_8U || depth == DMC_16S || depth == DMC_16U || depth == DMC_32F || depth == DMC_64F;
    if (!known || r == 0) TRY(copy_unless_same(ctx, out, in, image_bytes(src), s));     // other depths: only src.copyTo(dest) happens (:52); r == 0 is the identity
    else LAUNCH(ctx, launch_minmax(in, out, 1, src->rows, src->cols, depth, cn, r, s));
    return stage_out_end(ctx, dst, out, s);
}

static int minmax_filter(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int kw, int kh, int border_type, int is_max) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, src, "src")); TRY(check_image(ctx, dst, "dst"));
    if (border_type != DMC_BORDER_REPLICATE) return fail(ctx, DMC_ERR_ARG, "maxFilter/minFilter: only BORDER_REPLICATE is supported");
    if (kw < 1 || kh < 1 || kw / 2 > DMC_MAX_RADIUS || kh / 2 > DMC_MAX_RADIUS) return fail(ctx, DMC_ERR_ARG, "maxFilter/minFilter: kernel size out of range");
    const int t = src->cvtype;
    if (t != DMC_8U && t != DMC_16S && t != DMC_16U && t != DMC_32F) return DMC_UNSUPPORTED;    // `src.type()==CV_8U` ... :316-333
    if (dst->cvtype != t || dst->rows != src->rows || dst->cols != src->cols) return fail(ctx, DMC_ERR_SIZE, "maxFilter/minFilter: dst must match src");
    const void* in; void* out;
    TRY(stage_op(ctx, src, dst, &in, &out));
    const cudaStream_t s = ctx->stream;
    if (t == DMC_32F) {
        Buf& ftmp = ctx->slot[0].buf[SB_FLOAT];
        TRY(reserve(ctx, ftmp, image_bytes(src)));
        LAUNCH(ctx, launch_minmax_filter_f32_seeded((const float*)in, (float*)out, (float*)ftmp.p, src->rows, src->cols, kw, kh, is_max, s));
    } else LAUNCH(ctx, launch_morph(in, out, 1, src->rows, src->cols, t, kw, kh, is_max, s));
    return stage_out_end(ctx, dst, out, s);
}
int dmc_max_filter(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int kw, int kh, int border_type) { return minmax_filter(ctx, src, dst, kw, kh, border_type, 1); }
int dmc_min_filter(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int kw, int kh, int border_type) { return minmax_filter(ctx, src, dst, kw, kh, border_type, 0); }

int dmc_boundary_reconstruction(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int kw, int kh, float frec, float color, float space) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, src, "src")); TRY(check_image(ctx, dst, "dst"));
    if (kw < 1 || kh < 1 || kw / 2 > DMC_MAX_RADIUS || kh / 2 > DMC_MAX_RADIUS) return fail(ctx, DMC_ERR_ARG, "boundaryReconstructionFilter: kernel size out of range");
    const int t = src->cvtype;
    if (t != DMC_8U && t != DMC_16S && t != DMC_16U && t != DMC_32F && t != DMC_64F) return DMC_UNSUPPORTED;   // :133-155 single channel only
    if (dst->cvtype != t || dst->rows != src->rows || dst->cols != src->cols) return fail(ctx, DMC_ERR_SIZE, "boundaryReconstructionFilter: dst must match src");
    const void* in; void* out;
    TRY(stage_op(ctx, src, dst, &in, &out));
    const cudaStream_t s = ctx->stream;
    int nk = launch_brf(in, out, src->rows, src->cols, t, kw, kh, frec, color, space, s);
    if (nk == 0) return fail(ctx, DMC_ERR_ARG, "boundaryReconstructionFilter: window too large");
    TRY(after_launch(ctx, nk));
    return stage_out_end(ctx, dst, out, s);
}

int dmc_minmax_boundary_reconstruction(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int minmax_r, int kw, int kh, float frec, float color, float space) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, src, "src")); TRY(check_image(ctx, dst, "dst"));
    if (kw < 1 || kh < 1 || kw / 2 > DMC_MAX_RADIUS || kh / 2 > DMC_MAX_RADIUS) return fail(ctx, DMC_ERR_ARG, "minmaxBoundaryReconstructionFilter: kernel size out of range");
    if (minmax_r < 0 || minmax_r > DMC_MAX_RADIUS) return fail(ctx, DMC_ERR_ARG, "minmaxBoundaryReconstructionFilter: min-max radius out of range");
    const int t = src->cvtype;
    if (t != DMC_8U && t != DMC_16S && t != DMC_16U) return fail(ctx, DMC_ERR_TYPE, "minmaxBoundaryReconstructionFilter: single channel 8U / 16U / 16S only");
    if (dst->cvtype != t || dst->rows != src->rows || dst->cols != src->cols) return fail(ctx, DMC_ERR_SIZE, "minmaxBoundaryReconstructionFilter: dst must match src");
    const void* in; void* out;
    TRY(stage_op(ctx, src, dst, &in, &out));
    const cudaStream_t s = ctx->stream;
    int nk = launch_minmax_brf(in, out, src->rows, src->cols, t, minmax_r, kw, kh, frec, color, space, s);
    if (nk == 0) return fail(ctx, DMC_ERR_ARG, "minmaxBoundaryReconstructionFilter: window too large");
    TRY(after_launch(ctx, nk));
    return stage_out_end(ctx, dst, out, s);
}

int dmc_small_gaussian(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int d, double sigma) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, src, "src")); TRY(check_image(ctx, dst, "dst"));
    if (src->cvtype != DMC_8U || dst->cvtype != DMC_8U) return fail(ctx, DMC_ERR_TYPE, "smallGaussianBlur: CV_8UC1 only");
    if (dst->rows != src->rows || dst->cols != src->cols) return fail(ctx, DMC_ERR_SIZE, "smallGaussianBlur: dst must match src");
    if (d < 0 || (d > 0 && (d & 1) == 0) || d / 2 > DMC_MAX_RADIUS) return fail(ctx, DMC_ERR_ARG, "smallGaussianBlur: d must be 0 or odd, <= 21");
    const void* in; void* out;
    TRY(stage_op(ctx, src, dst, &in, &out));
    const cudaStream_t s = ctx->stream;
    GaussTaps t; t.rx = t.ry = 0;
    if (d > 1 && !make_gauss_taps(d, sigma, src->rows, src->cols, &t)) return fail(ctx, DMC_ERR_ARG, "smallGaussianBlur: bad kernel");
    if (d <= 1 || (t.rx == 0 && t.ry == 0)) TRY(copy_unless_same(ctx, out, in, image_bytes(src), s));
    else LAUNCH(ctx, launch_gauss8u((const uint8_t*)in, (uint8_t*)out, 1, src->rows, src->cols, t, s));
    return stage_out_end(ctx, dst, out, s);
}

int dmc_median_blur(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, int ksize) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, src, "src")); TRY(check_image(ctx, dst, "dst"));
    if (src->cvtype != DMC_8U || dst->cvtype != DMC_8U) return fail(ctx, DMC_ERR_TYPE, "medianBlur: CV_8UC1 only");
    if (dst->rows != src->rows || dst->cols != src->cols) return fail(ctx, DMC_ERR_SIZE, "medianBlur: dst must match src");
    if (ksize < 1 || (ksize & 1) == 0 || ksize / 2 > DMC_MAX_RADIUS) return fail(ctx, DMC_ERR_ARG, "medianBlur: ksize must be odd, <= 21");
    const void* in; void* out;
    TRY(stage_op(ctx, src, dst, &in, &out));
    const cudaStream_t s = ctx->stream;
    if (ksize == 1) TRY(copy_unless_same(ctx, out, in, image_bytes(src), s));
    else LAUNCH(ctx, launch_median8u((const uint8_t*)in, (uint8_t*)out, 1, src->rows, src->cols, ksize / 2, s));
    return stage_out_end(ctx, dst, out, s);
}

// ---- converters ---------------------------------------------------------------------------------------------------
static int convert_op(dmc_ctx* ctx, int kind, int stype, int dtype, const dmc_image* src, dmc_image* dst, float fb, float a, float b) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, src, "src")); TRY(check_image(ctx, dst, "dst"));
    if (src->cvtype != stype || dst->cvtype != dtype) return fail(ctx, DMC_ERR_TYPE, "converter: wrong src/dst type");
    if (dst->rows != src->rows || dst->cols != src->cols) return fail(ctx, DMC_ERR_SIZE, "converter: dst must match src");
    const void* in; void* out;
    TRY(stage_op(ctx, src, dst, &in, &out));
    const cudaStream_t s = ctx->stream;
    // disp8U2depth32F with b != 0 leaves most of dst untouched, so dst's previous contents are staged too
    if (kind == 0 && b != 0.f) { const void* prev; TRY(stage_in(ctx, dst, ctx->slot[0].buf[SB_OUT], s, &prev)); out = (void*)prev; }
    LAUNCH(ctx, launch_convert(kind, in, out, (long)src->rows * src->cols, fb, a, b, s));
    return stage_out_end(ctx, dst, out, s);
}
int dmc_disp8u2depth32f(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, float fb, float a, float b) { return convert_op(ctx, 0, DMC_8U, DMC_32F, src, dst, fb, a, b); }
int dmc_depth32f2disp8u(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, float fb, float a, float b) { return convert_op(ctx, 1, DMC_32F, DMC_8U, src, dst, fb, a, b); }
int dmc_depth16u2disp8u(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, float fb, float a, float b) { return convert_op(ctx, 2, DMC_16U, DMC_8U, src, dst, fb, a, b); }
int dmc_disp16s2depth16u(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst, float fb, float a, float b) { return convert_op(ctx, 3, DMC_16S, DMC_16U, src, dst, fb, a, b); }

int dmc_fill_occlusion(dmc_ctx* ctx, dmc_image* img, int invalid_value, int disp_or_depth) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, img, "img"));
    const int t = img->cvtype;
    if (t != DMC_8U && t != DMC_16S && t != DMC_16U && t != DMC_32F) return DMC_UNSUPPORTED;   // depthmapUtil.cpp:645-682
    if (img->cols < 2) return fail(ctx, DMC_ERR_SIZE, "fillOcclusion: needs at least 2 columns");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    Slot& sl = ctx->slot[0]; sl.stream = ctx->stream; cudaStream_t s = sl.stream;
    size_t row = dense_step(img), bytes = image_bytes(img);
    TRY(reserve(ctx, sl.buf[SB_IN], bytes)); TRY(reserve(ctx, sl.buf[SB_OUT], bytes));
    cudaMemcpyKind in_kind = img->mem == DMC_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    CUDA_TRY(ctx, cudaMemcpy2DAsync(sl.buf[SB_IN].p, row, img->data, step_of(img), row, img->rows, in_kind, s));
    CUDA_TRY(ctx, cudaMemcpyAsync(sl.buf[SB_OUT].p, sl.buf[SB_IN].p, bytes, cudaMemcpyDeviceToDevice, s));
    LAUNCH(ctx, launch_fill_occlusion(sl.buf[SB_OUT].p, sl.buf[SB_IN].p, img->rows, img->cols, t, (double)invalid_value, disp_or_depth == DMC_FILL_DEPTH, s));
    return stage_out_end(ctx, img, sl.buf[SB_OUT].p, s);
}

int dmc_transpose(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, src, "src")); TRY(check_image(ctx, dst, "dst"));
    if (cv_cn(src->cvtype) != 1) return fail(ctx, DMC_ERR_TYPE, "transpose: single-channel images only");
    if (dst->cvtype != src->cvtype || dst->rows != src->cols || dst->cols != src->rows) return fail(ctx, DMC_ERR_SIZE, "transpose: dst must be cols x rows of the same type");
    const void* in; void* out;
    TRY(stage_op(ctx, src, dst, &in, &out));
    const cudaStream_t s = ctx->stream;
    LAUNCH(ctx, launch_transpose(in, out, src->rows, src->cols, (int)elem_size(src->cvtype), s));
    return stage_out_end(ctx, dst, out, s);
}

int dmc_reproject_xyz(dmc_ctx* ctx, const dmc_image* depth, dmc_image* xyz, double f) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, depth, "depth")); TRY(check_image(ctx, xyz, "xyz"));
    const int t = depth->cvtype;
    if (t != DMC_8U && t != DMC_16S && t != DMC_16U && t != DMC_32F) return DMC_UNSUPPORTED;   // depthmapUtil.cpp:483-501
    const int H = depth->rows, W = depth->cols;
    if (xyz->cvtype != DMC_MAKETYPE(DMC_32F, 3) || (size_t)xyz->rows * xyz->cols != (size_t)H * W) return fail(ctx, DMC_ERR_TYPE, "reprojectXYZ: xyz must be 32FC3 with rows*cols == depth.total()");
    if (xyz->step && xyz->step != dense_step(xyz)) return fail(ctx, DMC_ERR_SIZE, "reprojectXYZ: xyz must be dense");
    const void* in; void* out;
    TRY(stage_op(ctx, depth, xyz, &in, &out));
    const cudaStream_t s = ctx->stream;
    const float fxinv = (float)(1.0 / f), fyinv = (float)(1.0 / f);
    const float cw = (W - 1) * 0.5f, ch = (H - 1) * 0.5f;
    if (!ctx->xtab || ctx->xtab_w != W || ctx->xtab_f != f) {       // x = (-cw)*fxinv; x += fxinv per column (:469, :478)
        std::vector<float> tab(W);
        volatile float x = (-cw) * fxinv;
        for (int i = 0; i < W; i++) { tab[i] = x; x = x + fxinv; }
        if (ctx->xtab) { CUDA_TRY(ctx, cudaStreamSynchronize(s)); CUDA_TRY(ctx, cudaFree(ctx->xtab)); ctx->xtab = nullptr; }
        CUDA_TRY(ctx, cudaMalloc(&ctx->xtab, W * sizeof(float)));
        CUDA_TRY(ctx, cudaMemcpy(ctx->xtab, tab.data(), W * sizeof(float), cudaMemcpyHostToDevice));
        ctx->xtab_w = W; ctx->xtab_f = f;
    }
    LAUNCH(ctx, launch_reproject(in, (float*)out, ctx->xtab, H, W, t, fyinv, ch, s));
    return stage_out_end(ctx, xyz, out, s);
}

// ---- point-cloud render (SURVEY.md 8f-3) ------------------------------------------------------------------------------
namespace {
void camera_floats(const double* R, const double* t, const double* K, float kr[9], float tt[3]) {      // Mat kr = K*R; (float)kr(i,j)  depthmapUtil.cpp:12-29
    for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) { double s = 0; for (int k = 0; k < 3; k++) s += K[3 * i + k] * R[3 * k + j]; kr[3 * i + j] = (float)s; }
    for (int i = 0; i < 3; i++) tt[i] = (float)t[i];
}
}  // namespace

int dmc_project_points(dmc_ctx* ctx, const dmc_image* xyz, const double* R, const double* t, const double* K, dmc_image* pt, int flags) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, xyz, "xyz")); TRY(check_image(ctx, pt, "pt"));
    if (!R || !t || !K) return fail(ctx, DMC_ERR_ARG, "projectPointsSimple: null camera");
    if (xyz->cvtype != DMC_MAKETYPE(DMC_32F, 3) || pt->cvtype != DMC_MAKETYPE(DMC_32F, 2)) return fail(ctx, DMC_ERR_TYPE, "projectPointsSimple: xyz must be 32FC3, pt 32FC2");
    const long n = (long)xyz->rows * xyz->cols;
    if ((long)pt->rows * pt->cols != n || (xyz->step && xyz->step != dense_step(xyz)) || (pt->step && pt->step != dense_step(pt))) return fail(ctx, DMC_ERR_SIZE, "projectPointsSimple: pt must hold one point per xyz entry, both dense");
    const void* in; void* out;
    TRY(stage_op(ctx, xyz, pt, &in, &out));
    const cudaStream_t s = ctx->stream;
    float kr[9], tt[3]; camera_floats(R, t, K, kr, tt);
    LAUNCH(ctx, launch_project_points((const float*)in, (float*)out, n, kr, tt, flags & DMC_RENDER_EXACT_DIVIDE, s));
    return stage_out_end(ctx, pt, out, s);
}

int dmc_project_image_from_xyz(dmc_ctx* ctx, const dmc_image* image, dmc_image* dest, const dmc_image* xyz, const double* R, const double* t, const double* K,
                               int is_sub, dmc_image* depth, dmc_image* pt, int flags) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, image, "image")); TRY(check_image(ctx, dest, "destimage")); TRY(check_image(ctx, xyz, "xyz"));
    if (!R || !t || !K) return fail(ctx, DMC_ERR_ARG, "projectImagefromXYZ: only support 64F matrix type");         // CV_Assert :290-294
    const int H = image->rows, W = image->cols; const long n = (long)H * W;
    if (image->cvtype != DMC_MAKETYPE(DMC_8U, 3) || dest->cvtype != image->cvtype) return fail(ctx, DMC_ERR_TYPE, "projectImagefromXYZ: image and destimage must be CV_8UC3");
    if (dest->rows != H || dest->cols != W) return fail(ctx, DMC_ERR_SIZE, "projectImagefromXYZ: destimage size != image size");
    if (xyz->cvtype != DMC_MAKETYPE(DMC_32F, 3) || (long)xyz->rows * xyz->cols != n || (xyz->step && xyz->step != dense_step(xyz))) return fail(ctx, DMC_ERR_TYPE, "projectImagefromXYZ: xyz must be dense 32FC3 with one point per pixel");
    if (depth) { TRY(check_image(ctx, depth, "depth")); if (depth->cvtype != DMC_32F || depth->rows != H || depth->cols != W) return fail(ctx, DMC_ERR_TYPE, "projectImagefromXYZ: depth must be 32FC1 of the image size"); }
    if (pt) { TRY(check_image(ctx, pt, "pt")); if (pt->cvtype != DMC_MAKETYPE(DMC_32F, 2) || (long)pt->rows * pt->cols != n || (pt->step && pt->step != dense_step(pt))) return fail(ctx, DMC_ERR_TYPE, "projectImagefromXYZ: pt must be dense 32FC2 with one entry per pixel"); }
    if (n >= (1l << 29)) return fail(ctx, DMC_ERR_SIZE, "projectImagefromXYZ: image too large");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    Slot& sl = ctx->slot[0]; sl.stream = ctx->stream; cudaStream_t s = sl.stream;
    const void *d_img, *d_xyz; void *d_dest, *d_depth = nullptr, *d_pt = nullptr;
    TRY(stage_in(ctx, image, sl.buf[SB_IN], s, &d_img));
    TRY(stage_in(ctx, xyz, sl.buf[SB_PING], s, &d_xyz));
    TRY(stage_out_begin(ctx, dest, d_img, image_bytes(image), sl.buf[SB_OUT], &d_dest));
    if (depth) { if (depth->mem == DMC_MEM_DEVICE && step_of(depth) == dense_step(depth)) d_depth = depth->data; else { TRY(reserve(ctx, sl.buf[SB_PONG], (size_t)n * 4)); d_depth = sl.buf[SB_PONG].p; } }
    if (pt && pt->mem == DMC_MEM_DEVICE) d_pt = pt->data; else { TRY(reserve(ctx, sl.buf[SB_FLOAT], (size_t)n * 8)); d_pt = sl.buf[SB_FLOAT].p; }
    TRY(reserve(ctx, ctx->render[0], render_scratch_bytes(H, W)));
    TRY(reserve(ctx, ctx->render[1], 64));
    if (!ctx->render_flag) CUDA_TRY(ctx, cudaHostAlloc((void**)&ctx->render_flag, 64, cudaHostAllocDefault));
    float kr[9], tt[3]; camera_floats(R, t, K, kr, tt);
    LAUNCH(ctx, launch_project_points((const float*)d_xyz, (float*)d_pt, n, kr, tt, flags & DMC_RENDER_EXACT_DIVIDE, s));
    int nk = launch_render((const uint8_t*)d_img, (const float*)d_xyz, (const float*)d_pt, H, W, is_sub, (uint8_t*)d_dest, (float*)d_depth,
                           ctx->render[0].p, (int*)ctx->render[1].p, ctx->render_flag, s);
    if (nk < 0) return fail(ctx, DMC_ERR_CUDA, std::string("projectImagefromXYZ: ") + cudaGetErrorString(cudaGetLastError()));
    TRY(after_launch(ctx, nk));
    if (depth && d_depth != depth->data) TRY(stage_out_end(ctx, depth, d_depth, s));
    if (pt && d_pt != pt->data) TRY(stage_out_end(ctx, pt, d_pt, s));
    return stage_out_end(ctx, dest, d_dest, s);
}

int dmc_fill_small_hole(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, src, "src")); TRY(check_image(ctx, dst, "dest"));
    if (src->cvtype != DMC_MAKETYPE(DMC_8U, 3) || dst->cvtype != src->cvtype) return fail(ctx, DMC_ERR_TYPE, "fillSmallHole: CV_8UC3 only");
    if (dst->rows != src->rows || dst->cols != src->cols) return fail(ctx, DMC_ERR_SIZE, "fillSmallHole: dest must match src");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    Slot& sl = ctx->slot[0]; sl.stream = ctx->stream; cudaStream_t s = sl.stream;
    const void* in; void* out;
    TRY(stage_in(ctx, src, sl.buf[SB_IN], s, &in));
    const bool same = dst->data == src->data;
    if (!same && dst->mem == DMC_MEM_DEVICE && step_of(dst) == dense_step(dst) && !overlaps(dst->data, image_bytes(dst), in, image_bytes(src))) out = dst->data;   // only holes are written: dest keeps the rest
    else {          // staged: dest's own previous content (or, in place, a copy of src -- `src.copyTo(src_)` :189-193) is the canvas
        TRY(reserve(ctx, sl.buf[SB_OUT], image_bytes(dst)));
        out = sl.buf[SB_OUT].p;
        const size_t row = dense_step(dst);
        if (same) CUDA_TRY(ctx, cudaMemcpyAsync(out, in, image_bytes(src), cudaMemcpyDeviceToDevice, s));
        else CUDA_TRY(ctx, cudaMemcpy2DAsync(out, row, dst->data, step_of(dst), row, dst->rows, dst->mem == DMC_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, s));
    }
    int nk = launch_fill_small_hole((const uint8_t*)in, (uint8_t*)out, src->rows, src->cols, s);
    TRY(after_launch(ctx, nk));
    return stage_out_end(ctx, dst, out, s);
}

// splitBGRLineInterleave filter.h:12 (split.cpp:167-177): 8UC3 / 32FC3 -> single channel, 3*rows x cols
int dmc_split_bgr_line_interleave(dmc_ctx* ctx, const dmc_image* src, dmc_image* dst) {
    if (!ctx) return fail(nullptr, DMC_ERR_ARG, "null context");
    TRY(check_image(ctx, src, "src")); TRY(check_image(ctx, dst, "dest"));
    const int depth = cv_depth(src->cvtype);
    if (cv_cn(src->cvtype) != 3 || (depth != DMC_8U && depth != DMC_32F)) return DMC_UNSUPPORTED;      // other types: nothing happens (:169-176)
    if (dst->cvtype != depth || dst->rows != 3 * src->rows || dst->cols != src->cols) return fail(ctx, DMC_ERR_SIZE, "splitBGRLineInterleave: dest must be single channel, 3*rows x cols");
    const void* in; void* out;
    TRY(stage_op(ctx, src, dst, &in, &out));
    const cudaStream_t s = ctx->stream;
    LAUNCH(ctx, launch_split_line_interleave(in, out, src->rows, src->cols, (int)depth_size(depth), s));
    return stage_out_end(ctx, dst, out, s);
}

}  // extern "C"
