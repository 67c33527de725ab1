// extern "C" surface of libsnn_b200.so for contexts, tensors, weights, single-operator launches and timers.
// (The whole-model engine entry points live in engine/model_capi.cpp.) See include/snnb.h for the reference
// interface each entry point replaces.
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <memory>

#include "snnb_internal.h"

namespace snnb {

static thread_local char g_err[1024] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
const char* get_error() { return g_err; }

bool pdl_enabled() {
    static const bool on = getenv("SNNB_NO_PDL") == nullptr;
    return on;
}

int ensure_stage(snnb_context* ctx, size_t bytes) {
    if (ctx->stage_dev_bytes < bytes) {
        if (ctx->stage_dev) cudaFree(ctx->stage_dev);
        ctx->stage_dev       = nullptr;
        ctx->stage_dev_bytes = 0;
        SNNB_CUDA_OK(cudaMalloc(&ctx->stage_dev, bytes));
        ctx->stage_dev_bytes = bytes;
    }
    return 0;
}
static int ensure_stage_host(snnb_context* ctx, size_t bytes) {
    if (ctx->stage_host_bytes < bytes) {
        if (ctx->stage_host) cudaFreeHost(ctx->stage_host);
        ctx->stage_host       = nullptr;
        ctx->stage_host_bytes = 0;
        SNNB_CUDA_OK(cudaMallocHost(&ctx->stage_host, bytes));
        ctx->stage_host_bytes = bytes;
    }
    return 0;
}

int tensor_alloc(snnb_context* ctx, int n, int h, int w, int c, snnb_tensor** out, bool lo_plane) {
    SNNB_REQUIRE(ctx && out, "tensor_alloc: null argument");
    SNNB_REQUIRE(n > 0 && h > 0 && w > 0 && c > 0, "tensor_alloc: bad dims %d %d %d %d", n, h, w, c);
    auto t   = std::make_unique<snnb_tensor>();
    t->ctx   = ctx;
    t->n = n, t->h = h, t->w = w, t->c = c, t->cp = round_up(c, 8);
    size_t elems   = (size_t) n * h * w * t->cp;
    t->plane_elems = (elems + 63) / 64 * 64;
    const size_t planes = lo_plane ? 2 : 1; // half-precision storage mode: the hi plane alone
    SNNB_CUDA_OK(cudaMalloc(&t->hi, t->plane_elems * planes * sizeof(__half)));
    t->lo = lo_plane ? t->hi + t->plane_elems : nullptr;
    SNNB_CUDA_OK(cudaMemsetAsync(t->hi, 0, t->plane_elems * planes * sizeof(__half), ctx->stream));
    *out = t.release();
    return 0;
}

// The compact 4-channel copy a stride-2 RGB stem reads (snnb_tensor::feed_*): zeroed once, the input kernels only ever write
// the image area, so the margins stay the constant padding.
int tensor_alloc_feed(snnb_tensor* t, int feed_h, int feed_w, int py, int px) {
    SNNB_REQUIRE(t && !t->feed_hi && t->c <= 4 && feed_h >= t->h + py && feed_w >= t->w + px && (feed_w & 1) == 0 && (px & 1) == 0, "tensor_alloc_feed: bad argument");
    const size_t plane  = ((size_t) t->n * feed_h * feed_w * 4 + 63) / 64 * 64;
    const size_t planes = t->lo ? 2 : 1;
    SNNB_CUDA_OK(cudaMalloc(&t->feed_hi, plane * planes * sizeof(__half)));
    SNNB_CUDA_OK(cudaMemsetAsync(t->feed_hi, 0, plane * planes * sizeof(__half), t->ctx->stream));
    t->feed_lo = t->lo ? t->feed_hi + plane : nullptr;
    t->feed_h = feed_h, t->feed_w = feed_w, t->feed_py = py, t->feed_px = px;
    return 0;
}

} // namespace snnb

using namespace snnb;

#define CHECK_DIMS_EQ(a, b, what) SNNB_REQUIRE((a)->n == (b)->n && (a)->h == (b)->h && (a)->w == (b)->w && (a)->c == (b)->c, what ": tensor dims differ")

extern "C" {

int snnb_version(void) { return SNNB_VERSION; }
int snnb_context_set_precision(snnb_context* ctx, int precision) {
    SNNB_REQUIRE(ctx && (precision == SNNB_PRECISION_FP32X3 || precision == SNNB_PRECISION_FP16W), "snnb_context_set_precision: FP32X3 or FP16W (FP16 storage is a model option)");
    ctx->precision = precision;
    return 0;
}
const char* snnb_last_error(void) { return get_error(); }

int snnb_context_create(int device, snnb_context** out) {
    SNNB_REQUIRE(out, "snnb_context_create: null out");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        set_error("snnb_context_create: no CUDA device available (%s). This library has no CPU fallback.", cudaGetErrorString(e));
        return 1;
    }
    SNNB_REQUIRE(device >= 0 && device < count, "snnb_context_create: device %d out of range (%d devices)", device, count);
    SNNB_CUDA_OK(cudaSetDevice(device));
    cudaDeviceProp prop;
    SNNB_CUDA_OK(cudaGetDeviceProperties(&prop, device));
    SNNB_REQUIRE(prop.major == 10, "snnb_context_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
    auto ctx      = std::make_unique<snnb_context>();
    ctx->device   = device;
    ctx->sm_count = prop.multiProcessorCount;
    SNNB_CUDA_OK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    *out = ctx.release();
    return 0;
}

int snnb_context_destroy(snnb_context* ctx) {
    if (!ctx) return 0;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->stage_dev) cudaFree(ctx->stage_dev);
    if (ctx->stage_host) cudaFreeHost(ctx->stage_host);
    for (void* b : ctx->scratch_blocks) cudaFree(b);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
    return 0;
}

int snnb_sync(snnb_context* ctx) {
    SNNB_REQUIRE(ctx, "snnb_sync: null context");
    SNNB_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    return 0;
}
void* snnb_context_stream(snnb_context* ctx) { return ctx ? (void*) ctx->stream : nullptr; }
uint64_t snnb_launch_count(snnb_context* ctx) { return ctx ? ctx->launches : 0; }

// ---- tensors ----
int snnb_tensor_alloc(snnb_context* ctx, int n, int h, int w, int c, snnb_tensor** out) { return tensor_alloc(ctx, n, h, w, c, out); }
int snnb_tensor_free(snnb_tensor* t) {
    if (!t) return 0;
    if (t->owns && t->hi) cudaFree(t->hi);
    if (t->feed_hi) cudaFree(t->feed_hi);
    delete t;
    return 0;
}
int snnb_debug_feed_plan(int k, int stride, int pad_x, int ic, int out[5]) {
    FeedPlan fp;
    if (!out || !make_feed_plan(k, stride, pad_x, ic, fp)) return 0;
    out[0] = fp.px, out[1] = fp.d, out[2] = fp.nch, out[3] = fp.ksteps, out[4] = fp.rows_per_panel;
    return 1;
}
int snnb_debug_streamk_schedule(int tiles, int num_kb, int sms, int* rows, int capacity) {
    SNNB_REQUIRE(rows || capacity == 0, "snnb_debug_streamk_schedule: null buffer");
    return streamk_schedule(tiles, num_kb, sms, rows, capacity);
}
int snnb_debug_kblock_schedule(int ksize, int cblocks, int icp, int sc_cblocks, int tiles, int ksplit, int sms, int* rows, int capacity) {
    SNNB_REQUIRE(rows || capacity == 0, "snnb_debug_kblock_schedule: null buffer");
    return kblock_schedule(ksize, cblocks, icp, sc_cblocks, tiles, ksplit, sms, rows, capacity);
}
int snnb_tensor_planes(const snnb_tensor* t, void** hi, void** lo, int* cp) {
    SNNB_REQUIRE(t && hi && lo && cp, "snnb_tensor_planes: null argument");
    *hi = t->hi, *lo = t->lo, *cp = t->cp;
    return 0;
}
int snnb_tensor_dims(const snnb_tensor* t, int* n, int* h, int* w, int* c) {
    SNNB_REQUIRE(t, "snnb_tensor_dims: null tensor");
    if (n) *n = t->n;
    if (h) *h = t->h;
    if (w) *w = t->w;
    if (c) *c = t->c;
    return 0;
}
int snnb_tensor_upload_nhwc(snnb_context* ctx, snnb_tensor* t, const float* host) {
    SNNB_REQUIRE(ctx && t && host, "snnb_tensor_upload_nhwc: null argument");
    const size_t bytes = t->pixels() * t->c * sizeof(float);
    if (ensure_stage(ctx, bytes)) return 1;
    SNNB_CUDA_OK(cudaMemcpyAsync(ctx->stage_dev, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (launch_split_f32(ctx, ctx->stage_dev, t)) return 1;
    SNNB_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    return 0;
}
int snnb_tensor_download_nhwc(snnb_context* ctx, const snnb_tensor* t, float* host) {
    SNNB_REQUIRE(ctx && t && host, "snnb_tensor_download_nhwc: null argument");
    const size_t bytes = t->pixels() * t->c * sizeof(float);
    if (ensure_stage(ctx, bytes)) return 1;
    if (launch_merge_f32(ctx, t, ctx->stage_dev)) return 1;
    SNNB_CUDA_OK(cudaMemcpyAsync(host, ctx->stage_dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    SNNB_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// C4HW4 <-> NHWC on the host (API-edge convenience for callers holding reference-layout textures).
static void c4_to_nhwc(const float* c4, int N, int H, int W, int C, float* nhwc) {
    const int D = (C + 3) / 4;
    for (int n = 0; n < N; ++n)
        for (int y = 0; y < H; ++y)
            for (int x = 0; x < W; ++x)
                for (int c = 0; c < C; ++c)
                    nhwc[(((size_t) n * H + y) * W + x) * C + c] = c4[((((size_t) n * D + c / 4) * H + y) * W + x) * 4 + (c % 4)];
}
static void nhwc_to_c4(const float* nhwc, int N, int H, int W, int C, float* c4) {
    const int D = (C + 3) / 4;
    memset(c4, 0, sizeof(float) * (size_t) N * D * H * W * 4);
    for (int n = 0; n < N; ++n)
        for (int y = 0; y < H; ++y)
            for (int x = 0; x < W; ++x)
                for (int c = 0; c < C; ++c)
                    c4[((((size_t) n * D + c / 4) * H + y) * W + x) * 4 + (c % 4)] = nhwc[(((size_t) n * H + y) * W + x) * C + c];
}
int snnb_tensor_upload_c4hw4(snnb_context* ctx, snnb_tensor* t, const float* host_c4) {
    SNNB_REQUIRE(ctx && t && host_c4, "snnb_tensor_upload_c4hw4: null argument");
    std::vector<float> tmp(t->pixels() * t->c);
    c4_to_nhwc(host_c4, t->n, t->h, t->w, t->c, tmp.data());
    return snnb_tensor_upload_nhwc(ctx, t, tmp.data());
}
int snnb_tensor_download_c4hw4(snnb_context* ctx, const snnb_tensor* t, float* host_c4) {
    SNNB_REQUIRE(ctx && t && host_c4, "snnb_tensor_download_c4hw4: null argument");
    std::vector<float> tmp(t->pixels() * t->c);
    if (snnb_tensor_download_nhwc(ctx, t, tmp.data())) return 1;
    nhwc_to_c4(tmp.data(), t->n, t->h, t->w, t->c, host_c4);
    return 0;
}
int snnb_tensor_dump(snnb_context* ctx, const snnb_tensor* t, const char* path) {
    SNNB_REQUIRE(ctx && t && path, "snnb_tensor_dump: null argument");
    const int D = (t->c + 3) / 4;
    std::vector<float> c4((size_t) t->n * D * t->h * t->w * 4);
    if (snnb_tensor_download_c4hw4(ctx, t, c4.data())) return 1;
    for (int n = 0; n < t->n; ++n) {
        std::string p = path;
        if (t->n > 1) p += ".n" + std::to_string(n);
        FILE* f = fopen(p.c_str(), "wb");
        SNNB_REQUIRE(f, "snnb_tensor_dump: cannot open %s", p.c_str());
        char header[32];
        memset(header, 0, sizeof(header));
        snprintf(header, sizeof(header), "%d %d %d %d", t->w, t->h, D, t->c); // image.cpp:216-245: "W H D C"
        fwrite(header, 1, sizeof(header), f);
        fwrite(c4.data() + (size_t) n * D * t->h * t->w * 4, sizeof(float), (size_t) D * t->h * t->w * 4, f);
        fclose(f);
    }
    return 0;
}

// ---- weights ----
static int make_weights(snnb_context* ctx, const PackedHost& p, snnb_weights** out) {
    auto w       = std::make_unique<snnb_weights>();
    size_t bytes = p.device_bytes();
    SNNB_CUDA_OK(cudaMalloc(&w->owned, bytes ? bytes : 256));
    if (place_weights(ctx, p, (char*) w->owned, w.get())) {
        cudaFree(w->owned);
        return 1;
    }
    *out = w.release();
    return 0;
}
int snnb_weights_pack_conv2d(snnb_context* ctx, const snnb_conv_desc* d, const float* w_oihw, const float* bias, const float* g, const float* b,
                             const float* m, const float* v, snnb_weights** out) {
    SNNB_REQUIRE(ctx && d && w_oihw && out, "snnb_weights_pack_conv2d: null argument");
    SNNB_REQUIRE(d->in_channels > 0 && d->out_channels > 0 && d->kernel > 0, "snnb_weights_pack_conv2d: bad desc");
    PackedHost p;
    pack_conv2d_host(d->in_channels, d->out_channels, d->kernel, w_oihw, bias, g, b, m, v, p);
    pack_rowwin_host(p, d->stride, d->pad_x);
    return make_weights(ctx, p, out);
}
int snnb_weights_pack_depthwise(snnb_context* ctx, const snnb_conv_desc* d, const float* w_chw, const float* bias, const float* g, const float* b,
                                const float* m, const float* v, snnb_weights** out) {
    SNNB_REQUIRE(ctx && d && w_chw && out, "snnb_weights_pack_depthwise: null argument");
    SNNB_REQUIRE(d->in_channels > 0 && d->in_channels == d->out_channels, "snnb_weights_pack_depthwise: depth multiplier != 1 is not supported "
                                                                           "(as in the reference, modelparser.cpp:821)");
    PackedHost p;
    pack_depthwise_host(d->in_channels, d->kernel, w_chw, bias, g, b, m, v, p);
    return make_weights(ctx, p, out);
}
int snnb_weights_pack_dense(snnb_context* ctx, int n_in, int n_out, const float* kernel, const float* bias, snnb_weights** out) {
    SNNB_REQUIRE(ctx && kernel && out && n_in > 0 && n_out > 0, "snnb_weights_pack_dense: bad argument");
    PackedHost p; // [out][in] row-major == OIHW with k = 1
    pack_conv2d_host(n_in, n_out, 1, kernel, bias, nullptr, nullptr, nullptr, nullptr, p);
    p.kind = 3;
    return make_weights(ctx, p, out);
}
int snnb_weights_pack_channels(snnb_context* ctx, int channels, const float* g, const float* b, const float* m, const float* v, snnb_weights** out) {
    SNNB_REQUIRE(ctx && out && channels > 0, "snnb_weights_pack_channels: bad argument");
    PackedHost p;
    pack_channels_host(channels, g, b, m, v, p);
    return make_weights(ctx, p, out);
}
int snnb_weights_free(snnb_weights* w) {
    if (!w) return 0;
    if (w->owned) cudaFree(w->owned);
    delete w;
    return 0;
}

// ---- operators ----
int snnb_conv2d_launch(snnb_context* ctx, const snnb_conv_desc* d, const snnb_weights* w, const snnb_tensor* in, const snnb_tensor* residual,
                       snnb_tensor* out) {
    SNNB_REQUIRE(ctx && d && w && in && out, "snnb_conv2d_launch: null argument");
    SNNB_REQUIRE(w->kind == 1 || w->kind == 3, "snnb_conv2d_launch: weights were not packed for conv2d");
    SNNB_REQUIRE(in->c == w->in_ch && out->c == w->out_ch && d->kernel == w->kernel, "snnb_conv2d_launch: tensor channels (%d -> %d, k%d) do not match the weights (%d -> %d, k%d)",
                 in->c, out->c, d->kernel, w->in_ch, w->out_ch, w->kernel);
    SNNB_REQUIRE(in->n == out->n, "snnb_conv2d_launch: batch mismatch");
    if (residual) CHECK_DIMS_EQ(residual, out, "snnb_conv2d_launch(residual)");
    ConvArgs a {in, residual, out, w, d->kernel, d->stride, d->pad_x, d->pad_y, d->pad_mode, d->activation, d->leaky_alpha};
    a.stream_k = d->algo == SNNB_ALGO_TCGEN05_STREAMK;
    if (d->algo == SNNB_ALGO_TCGEN05 || d->algo == SNNB_ALGO_TCGEN05_STREAMK) {
        SNNB_REQUIRE(conv2d_umma_supported(a), "snnb_conv2d_launch: the tcgen05 path does not support this shape (IC=%d OC=%d k=%d s=%d pad_mode=%d)", in->c, out->c,
                     d->kernel, d->stride, d->pad_mode);
        return launch_conv2d_umma(ctx, a);
    }
    if (d->algo == SNNB_ALGO_AUTO && conv2d_umma_supported(a)) return launch_conv2d_umma(ctx, a);
    return launch_conv2d_simt(ctx, a);
}
int snnb_depthwise_launch(snnb_context* ctx, const snnb_conv_desc* d, const snnb_weights* w, const snnb_tensor* in, snnb_tensor* out) {
    SNNB_REQUIRE(ctx && d && w && in && out, "snnb_depthwise_launch: null argument");
    SNNB_REQUIRE(w->kind == 2 && in->c == w->in_ch && out->c == in->c && d->kernel == w->kernel, "snnb_depthwise_launch: weights/tensor mismatch");
    SNNB_REQUIRE(in->n == out->n, "snnb_depthwise_launch: batch mismatch");
    ConvArgs a {in, nullptr, out, w, d->kernel, d->stride, d->pad_x, d->pad_y, SNNB_PAD_CONSTANT, d->activation, d->leaky_alpha};
    return launch_depthwise(ctx, a);
}
int snnb_maxpool_launch(snnb_context* ctx, int kernel, int stride, const snnb_tensor* in, snnb_tensor* out) {
    SNNB_REQUIRE(ctx && in && out && kernel > 0 && stride > 0 && in->c == out->c && in->n == out->n, "snnb_maxpool_launch: bad argument");
    // every window must START inside the input (pool windows are clipped at the bottom/right edge, never padded top/left)
    SNNB_REQUIRE((long long) (out->w - 1) * stride < in->w && (long long) (out->h - 1) * stride < in->h, "snnb_maxpool_launch: output %dx%d does not fit input %dx%d at stride %d", out->h, out->w, in->h, in->w, stride);
    return launch_pool(ctx, in, out, kernel, stride, false);
}
int snnb_avgpool_launch(snnb_context* ctx, int kernel, int stride, const snnb_tensor* in, snnb_tensor* out) {
    SNNB_REQUIRE(ctx && in && out && kernel > 0 && stride > 0 && in->c == out->c && in->n == out->n, "snnb_avgpool_launch: bad argument");
    // every window must START inside the input (pool windows are clipped at the bottom/right edge, never padded top/left)
    SNNB_REQUIRE((long long) (out->w - 1) * stride < in->w && (long long) (out->h - 1) * stride < in->h, "snnb_avgpool_launch: output %dx%d does not fit input %dx%d at stride %d", out->h, out->w, in->h, in->w, stride);
    return launch_pool(ctx, in, out, kernel, stride, true);
}
int snnb_add_launch(snnb_context* ctx, int act, float alpha, const snnb_tensor* a, const snnb_tensor* b, snnb_tensor* out) {
    SNNB_REQUIRE(ctx && a && b && out, "snnb_add_launch: null argument");
    CHECK_DIMS_EQ(a, b, "snnb_add_launch");
    CHECK_DIMS_EQ(a, out, "snnb_add_launch");
    return launch_add(ctx, a, b, out, act, alpha);
}
int snnb_batchnorm_launch(snnb_context* ctx, const snnb_weights* w, int act, float alpha, const snnb_tensor* in, snnb_tensor* out) {
    SNNB_REQUIRE(ctx && w && in && out && w->kind == 4 && w->in_ch == in->c, "snnb_batchnorm_launch: bad argument");
    CHECK_DIMS_EQ(in, out, "snnb_batchnorm_launch");
    return launch_batchnorm(ctx, in, out, w, act, alpha);
}
int snnb_activation_launch(snnb_context* ctx, int act, float alpha, const snnb_tensor* in, snnb_tensor* out) {
    SNNB_REQUIRE(ctx && in && out, "snnb_activation_launch: null argument");
    CHECK_DIMS_EQ(in, out, "snnb_activation_launch");
    return launch_activation(ctx, in, out, act, alpha);
}
int snnb_softmax_launch(snnb_context* ctx, const snnb_tensor* in, snnb_tensor* out) {
    SNNB_REQUIRE(ctx && in && out, "snnb_softmax_launch: null argument");
    CHECK_DIMS_EQ(in, out, "snnb_softmax_launch");
    return launch_softmax(ctx, in, out);
}
int snnb_flatten_launch(snnb_context* ctx, const snnb_tensor* in, snnb_tensor* out) {
    SNNB_REQUIRE(ctx && in && out && out->n == in->n && out->h == 1 && out->w == 1 && out->c == in->h * in->w * in->c, "snnb_flatten_launch: bad dims");
    return launch_flatten(ctx, in, out);
}
int snnb_dense_launch(snnb_context* ctx, const snnb_weights* w, int act, float alpha, const snnb_tensor* in, snnb_tensor* out) {
    SNNB_REQUIRE(ctx && w && in && out && (w->kind == 3 || w->kind == 1), "snnb_dense_launch: bad argument");
    SNNB_REQUIRE(in->h * in->w * in->c == w->in_ch && out->c == w->out_ch && out->h == 1 && out->w == 1 && in->n == out->n,
                 "snnb_dense_launch: dims do not match the weights (%d -> %d)", w->in_ch, w->out_ch);
    snnb_tensor* flat   = nullptr;
    const snnb_tensor* x = in;
    if (in->h * in->w != 1) {
        if (tensor_alloc(ctx, in->n, 1, 1, w->in_ch, &flat)) return 1;
        if (launch_flatten(ctx, in, flat)) return 1;
        x = flat;
    }
    const bool softmax = act == SNNB_ACT_SOFTMAX;
    ConvArgs a {x, nullptr, out, w, 1, 1, 0, 0, SNNB_PAD_NONE, softmax ? SNNB_ACT_NONE : act, alpha};
    int rc = conv2d_umma_supported(a) ? launch_conv2d_umma(ctx, a) : launch_conv2d_simt(ctx, a);
    if (!rc && softmax) rc = launch_softmax(ctx, out, out);
    if (flat) {
        cudaStreamSynchronize(ctx->stream);
        snnb_tensor_free(flat);
    }
    return rc;
}
int snnb_argmax1(snnb_context* ctx, const snnb_tensor* in, int* host_idx) {
    SNNB_REQUIRE(ctx && in && host_idx, "snnb_argmax1: null argument");
    if (ensure_stage(ctx, sizeof(int) * in->n)) return 1;
    int* dev = reinterpret_cast<int*>(ctx->stage_dev);
    if (launch_argmax(ctx, in, dev)) return 1;
    SNNB_CUDA_OK(cudaMemcpyAsync(host_idx, dev, sizeof(int) * in->n, cudaMemcpyDeviceToHost, ctx->stream));
    SNNB_CUDA_OK(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < in->n; ++i) host_idx[i] += 1; // core.cpp:228-233: 1-based
    return 0;
}
int snnb_concat_launch(snnb_context* ctx, const snnb_tensor* a, const snnb_tensor* b, snnb_tensor* out) {
    SNNB_REQUIRE(ctx && a && b && out, "snnb_concat_launch: null argument");
    SNNB_REQUIRE(a->n == b->n && a->h == b->h && a->w == b->w && out->n == a->n && out->h == a->h && out->w == a->w && out->c == a->c + b->c,
                 "snnb_concat_launch: bad dims");
    return launch_concat(ctx, a, b, out);
}
int snnb_upsample_launch(snnb_context* ctx, float scale, int bilinear, const snnb_tensor* in, snnb_tensor* out) {
    SNNB_REQUIRE(ctx && in && out && scale > 0 && in->c == out->c && in->n == out->n, "snnb_upsample_launch: bad argument");
    return launch_upsample(ctx, in, out, scale, bilinear != 0);
}
int snnb_pad_launch(snnb_context* ctx, int pad_x, int pad_y, int mode, const snnb_tensor* in, snnb_tensor* out) {
    SNNB_REQUIRE(ctx && in && out && in->c == out->c && in->n == out->n, "snnb_pad_launch: bad argument");
    return launch_pad(ctx, in, out, pad_x, pad_y, mode);
}
int snnb_instancenorm_launch(snnb_context* ctx, const snnb_weights* w, int act, float alpha, const snnb_tensor* in, snnb_tensor* out) {
    SNNB_REQUIRE(ctx && w && in && out && w->kind == 4 && w->in_ch == in->c, "snnb_instancenorm_launch: bad argument");
    CHECK_DIMS_EQ(in, out, "snnb_instancenorm_launch");
    return launch_instancenorm(ctx, in, out, w, act, alpha);
}
int snnb_subpixel_launch(snnb_context* ctx, int r, const snnb_tensor* in, snnb_tensor* out) {
    SNNB_REQUIRE(ctx && in && out && r > 0 && in->c == r * r && out->c == 1 && out->h == in->h * r && out->w == in->w * r && in->n == out->n,
                 "snnb_subpixel_launch: bad dims");
    return launch_subpixel(ctx, in, out, r);
}

// ---- timers ----
int snnb_timer_create(snnb_context* ctx, snnb_timer** out) {
    SNNB_REQUIRE(ctx && out, "snnb_timer_create: null argument");
    auto t = std::make_unique<snnb_timer>();
    t->ctx = ctx;
    SNNB_CUDA_OK(cudaEventCreate(&t->e0));
    SNNB_CUDA_OK(cudaEventCreate(&t->e1));
    *out = t.release();
    return 0;
}
int snnb_timer_start(snnb_timer* t) {
    SNNB_REQUIRE(t, "snnb_timer_start: null timer");
    SNNB_CUDA_OK(cudaEventRecord(t->e0, t->ctx->stream));
    return 0;
}
int snnb_timer_stop(snnb_timer* t) {
    SNNB_REQUIRE(t, "snnb_timer_stop: null timer");
    SNNB_CUDA_OK(cudaEventRecord(t->e1, t->ctx->stream));
    return 0;
}
int snnb_timer_elapsed_ms(snnb_timer* t, float* ms) {
    SNNB_REQUIRE(t && ms, "snnb_timer_elapsed_ms: null argument");
    SNNB_CUDA_OK(cudaEventSynchronize(t->e1));
    SNNB_CUDA_OK(cudaEventElapsedTime(ms, t->e0, t->e1));
    return 0;
}
int snnb_timer_destroy(snnb_timer* t) {
    if (!t) return 0;
    cudaEventDestroy(t->e0);
    cudaEventDestroy(t->e1);
    delete t;
    return 0;
}

// ---- launch capture -----------------------------------------------------------------------------------------
int snnb_graph_capture_begin(snnb_context* ctx) {
    SNNB_REQUIRE(ctx, "snnb_graph_capture_begin: null context");
    SNNB_CUDA_OK(cudaSetDevice(ctx->device));
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    SNNB_CUDA_OK(cudaStreamIsCapturing(ctx->stream, &st));
    SNNB_REQUIRE(st == cudaStreamCaptureStatusNone, "snnb_graph_capture_begin: the context is already capturing");
    SNNB_CUDA_OK(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
    return 0;
}
int snnb_graph_capture_end(snnb_context* ctx, snnb_graph** out) {
    SNNB_REQUIRE(ctx && out, "snnb_graph_capture_end: null argument");
    cudaGraph_t g = nullptr;
    const cudaError_t e = cudaStreamEndCapture(ctx->stream, &g);
    if (e != cudaSuccess || !g) {
        cudaGetLastError();
        set_error("snnb_graph_capture_end: capture failed (%s); a launch inside the region reported an error or allocated memory", cudaGetErrorString(e));
        return 1;
    }
    cudaGraphExec_t ex = nullptr;
    const cudaError_t e2 = cudaGraphInstantiate(&ex, g, 0);
    if (e2 != cudaSuccess) {
        cudaGraphDestroy(g);
        set_error("snnb_graph_capture_end: cudaGraphInstantiate failed (%s)", cudaGetErrorString(e2));
        return 1;
    }
    auto* h = new snnb_graph();
    h->ctx = ctx, h->graph = g, h->exec = ex;
    *out = h;
    return 0;
}
int snnb_graph_launch(snnb_graph* g) {
    SNNB_REQUIRE(g && g->exec, "snnb_graph_launch: null graph");
    SNNB_CUDA_OK(cudaSetDevice(g->ctx->device));
    SNNB_CUDA_OK(cudaGraphLaunch(g->exec, g->ctx->stream));
    return 0;
}
int snnb_graph_destroy(snnb_graph* g) {
    if (!g) return 0;
    if (g->exec) cudaGraphExecDestroy(g->exec);
    if (g->graph) cudaGraphDestroy(g->graph);
    delete g;
    return 0;
}

} // extern "C"
