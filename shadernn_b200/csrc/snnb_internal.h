// Internal types shared by the C-ABI layer (capi.cpp), the host engine (engine/*.cpp) and the CUDA
// kernels (kernels_*.cu). Not installed; the public surface is include/snnb.h.
#pragma once

#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cstdint>
#include <cstdio>
#include <string>
#include <utility>
#include <vector>

#include "snnb.h"

namespace snnb {

// ---- error plumbing: status codes + thread-local message (never abort across the C-ABI) ----------------------
void set_error(const char* fmt, ...);
const char* get_error();

#define SNNB_CUDA_OK(expr)                                                                              \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess) {                                                                        \
            ::snnb::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));    \
            return 1;                                                                                   \
        }                                                                                               \
    } while (0)

#define SNNB_REQUIRE(cond, ...)          \
    do {                                 \
        if (!(cond)) {                   \
            ::snnb::set_error(__VA_ARGS__); \
            return 2;                    \
        }                                \
    } while (0)

static inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

// ---- programmatic dependent launch (PDL) -----------------------------------------------------------------------
// The persistent TMA / tcgen05 kernels are launched with cudaLaunchAttributeProgrammaticStreamSerialization: their CTAs may
// be scheduled (and run their prologue: barrier init, TMEM allocation, tensor-map prefetch) while the previous kernel is
// still draining. pdl_wait() blocks until the previous grid has completed and its writes are visible; NOTHING before it
// may touch global memory that another kernel writes. pdl_trigger() lets the next grid start launching. ONLY the persistent
// kernels (grid <= SM count, every CTA resident from the start) call it, first thing: in a multi-wave kernel the early
// dependents would sit resident in griddepcontrol.wait and take SM slots from this grid's later waves (measured: the
// style-transfer graph ran 2.2x slower with triggers in the CUDA-core kernels). Set SNNB_NO_PDL=1 to launch plainly.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k_impl(bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim            = grid;
    cfg.blockDim           = block;
    cfg.dynamicSmemBytes   = smem;
    cfg.stream             = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id                                         = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs                                          = attr;
    cfg.numAttrs                                       = (pdl && pdl_enabled()) ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
// plain stream-ordered launch (the CUDA-core kernels: no prologue worth overlapping)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
    return launch_k_impl(false, kernel, grid, block, smem, stream, std::forward<Args>(args)...);
}
// programmatic dependent launch (the persistent TMA / tcgen05 kernels, which call pdl_trigger() and pdl_wait())
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
    return launch_k_impl(true, kernel, grid, block, smem, stream, std::forward<Args>(args)...);
}
#endif

} // namespace snnb

// ---- device storage -----------------------------------------------------------------------------------------
// Activations: NHWC, channel pitch Cp = round_up(C, 8), stored as TWO fp16 planes ("split-fp16"):
//     hi = fp16_rn(v),  lo = fp16_rn(v - hi)          (v = hi + lo to 2^-22 relative for |v| >= 2^-3; absolute 3e-8 below)
// Same 4 bytes/element of HBM traffic as fp32, but each plane is a K-major fp16 operand that TMA can drop into shared
// memory for tcgen05.mma (kind::f16) unmodified. Products accumulate in fp32 TMEM as
//     3-term  hi*Whi + lo*Whi + hi*Wlo   (weights as fp16 pairs too: ~22 bits per operand)          SNNB_PRECISION_FP32X3
//     2-term  hi*Whi + lo*Whi            (weights rounded once to fp16: <= 2^-12 relative per weight)  SNNB_PRECISION_FP16W
//     1-term  hi*Whi                     (half-precision storage mode: no lo planes at all)           SNNB_PRECISION_FP16->FP16
// Round 1 stored bf16 pairs (8+8 bits); tcgen05's kind::f16 refuses a bf16 A with an fp16 B operand ("illegal instruction",
// tools/umma_desc_probe.cu), so the pair format itself moved to fp16 to make the 2-term product possible. Range: values are
// saturated to +-65504 on store (cvt.rn.satfinite), the same range as the reference's own RGBA16F mode.
// Channels [C, Cp) are kept at zero.
struct snnb_tensor {
    snnb_context* ctx = nullptr;
    __half* hi = nullptr; // plane 0; plane 1 (lo) = hi + plane_elems
    __half* lo = nullptr;
    int n = 0, h = 0, w = 0, c = 0, cp = 0;
    size_t plane_elems = 0;      // n*h*w*cp rounded up to 64 elements (128 B)
    bool owns = true;
    // Optional "stem feed" (model input tensors consumed by a stride-2 convolution with <= 4 input channels, see FeedPlan and
    // conv_rowwin_kernel): a second, compact copy of the image with 4 channels per pixel, [n][feed_h][feed_w][4] fp16 per plane,
    // image pixel (y, x) at (y + feed_py, x + feed_px), zero margins. Written by the input kernels (split / normalise / resize)
    // together with the regular planes; the regular planes stay valid for every other consumer.
    __half* feed_hi = nullptr;
    __half* feed_lo = nullptr;
    int feed_h = 0, feed_w = 0, feed_py = 0, feed_px = 0;
    // Every consumer of this tensor reads the feed: the input kernels then skip the regular planes (51 of 87 MB written per ResNet-18
    // batch) and read-backs of the tensor (layer output, dumps) are served from the feed.
    bool feed_only = false;
    size_t pixels() const { return (size_t) n * h * w; }
};

// Packed weights of one layer (device pointers; owned unless carved from a model arena).
struct snnb_weights {
    snnb_context* ctx = nullptr;
    int kind = 0; // 1 conv, 2 depthwise, 3 dense(conv1x1), 4 channels
    int in_ch = 0, out_ch = 0, kernel = 1;
    // SIMT path: fp32 [K = k*k*IC][OCw], OCw = round_up(OC, 64); BN folded in.
    float* w_f32 = nullptr;
    int ocw = 0;
    // tcgen05 path: fp16 hi/lo [OCr][Kp] K-major (k index = (ky*k+kx)*IC + ic), Kp = round_up(K, 8), OCr = round_up(OC, 16).
    __half* w_hi = nullptr;
    __half* w_lo = nullptr;
    int kp = 0, ocr = 0;
    // small-input-channel "row window" variant (IC <= 8): fp16 hi/lo [kh][OCr][64], columns in RowPlan K order
    __half* w_row_hi = nullptr;
    __half* w_row_lo = nullptr;
    int row_stride = 0, row_pad = 0;
    __half* w_feed_hi = nullptr; // feed-mode operand [kh][OCr][64] (FeedPlan K order), or null
    __half* w_feed_lo = nullptr;
    int feed_pad = -1;           // the x padding it was packed for
    // depthwise: fp32 [k*k][Cp]
    // folded bias: fp32 [round_up(OC, 64)]
    float* bias = nullptr;
    // channel vectors (BatchNormalization / InstanceNorm): fp32 [Cp] each
    float *gamma = nullptr, *beta = nullptr, *mean = nullptr, *var = nullptr;
    void* owned = nullptr; // single allocation backing all of the above (nullptr when arena-backed)
    size_t bytes = 0;
};

struct snnb_context {
    int device          = 0;
    cudaStream_t stream = nullptr;
    int sm_count        = 148;
    uint64_t launches   = 0;
    // staging for upload/download (grown on demand)
    float* stage_dev    = nullptr;
    size_t stage_dev_bytes = 0;
    float* stage_host   = nullptr; // pinned
    size_t stage_host_bytes = 0;
    void* tmap_encode_fn = nullptr; // cuTensorMapEncodeTiled, resolved lazily
    // split-K scratch of the tensor-core convolution (kernels_umma.cu); blocks are freed with the context
    float* splitk_partials = nullptr;
    size_t splitk_bytes    = 0;
    int* splitk_counters   = nullptr;
    size_t splitk_counter_n = 0;
    int* sched_counter      = nullptr; // dynamic tile scheduler of conv_umma_kernel (self-resetting)
    // cudaFuncSetAttribute(MaxDynamicSharedMemorySize) applies to the CURRENT device only: one bit per kernel, per context
    // (= per device), not a process-wide flag
    uint32_t func_attr_mask = 0;
    const char* last_kernel = nullptr; // name of the kernel the most recent launcher chose (snnb_model_layer_kernel, bench.py's roofline)
    int precision = SNNB_PRECISION_FP32X3; // default product form of per-operator convolution launches (snnb_context_set_precision)
    std::vector<void*> scratch_blocks;
};

struct snnb_graph {
    snnb_context* ctx     = nullptr;
    cudaGraph_t graph     = nullptr;
    cudaGraphExec_t exec  = nullptr;
};

struct snnb_timer {
    snnb_context* ctx = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
};

namespace snnb {

int ensure_stage(snnb_context* ctx, size_t bytes);

// ---- kernel launchers (kernels_simt.cu) -------------------------------------------------------------------
struct ConvArgs {
    const snnb_tensor* in;
    const snnb_tensor* residual; // nullable
    snnb_tensor* out;
    const snnb_weights* w;
    int k, stride, pad_x, pad_y, pad_mode, act;
    float alpha;
    int precision = -1; // SNNB_PRECISION_* of this launch; -1 = the context's default
    bool stream_k = false; // the planner may choose the stream-K decomposition (SNNB_ALGO_TCGEN05_STREAMK)
    // Folded projection shortcut (tensor path only): out = conv(in) + conv1x1_stride(shortcut), the second product as extra K blocks
    // of the same GEMM. The weights then carry [k*k*ICp | ICp_shortcut] columns and one summed bias; `residual` must be null.
    const snnb_tensor* shortcut = nullptr;
    int sc_stride = 1;
};
int launch_conv2d_simt(snnb_context* ctx, const ConvArgs& a);
int launch_conv2d_umma(snnb_context* ctx, const ConvArgs& a); // kernels_umma.cu (tcgen05 + TMA)
bool conv2d_umma_supported(const ConvArgs& a);
// Would launch_conv2d_umma run `a` (shortcut set, weights may be a probe) in plain mode, the only mode that reads a shortcut? False for
// the row-window kernel, for layers the planner gives to the halo mode, and for shortcuts the TMA box cannot express.
bool conv2d_umma_fold_supported(const snnb_context* ctx, const ConvArgs& a);
// host walk of every K block of a (folded) launch's work items, as the producer visits them (tests); see kernels_umma.cu
int kblock_schedule(int ksize, int cblocks, int icp, int sc_cblocks, int tiles, int ksplit, int sms, int* rows, int capacity);
int streamk_schedule(int tiles, int num_kb, int sms, int* rows, int capacity); // host evaluation of the stream-K work decomposition (tests)
int launch_depthwise(snnb_context* ctx, const ConvArgs& a);
bool depthwise_tma_supported(const ConvArgs& a);          // 3x3 stride 1/2: TMA-staged, register-tiled (kernels_umma.cu)
int launch_depthwise_tma(snnb_context* ctx, const ConvArgs& a);
int launch_pool(snnb_context* ctx, const snnb_tensor* in, snnb_tensor* out, int k, int stride, bool avg);
// global average pool -> Dense (+ activation / softmax) in one launch (small classifier heads)
bool gap_dense_supported(const snnb_tensor* in, const snnb_tensor* out, const snnb_weights* w);
int launch_gap_dense(snnb_context* ctx, const snnb_tensor* in, snnb_tensor* out, const snnb_weights* w, int act, float alpha, bool softmax);
int launch_add(snnb_context* ctx, const snnb_tensor* a, const snnb_tensor* b, snnb_tensor* out, int act, float alpha);
int launch_batchnorm(snnb_context* ctx, const snnb_tensor* in, snnb_tensor* out, const snnb_weights* w, int act, float alpha);
int launch_activation(snnb_context* ctx, const snnb_tensor* in, snnb_tensor* out, int act, float alpha);
int launch_softmax(snnb_context* ctx, const snnb_tensor* in, snnb_tensor* out);
int launch_argmax(snnb_context* ctx, const snnb_tensor* in, int* dev_idx);
// YOLO decode, device part: cells whose score can pass `thresh` -> ONE candidate list [maxc][8] = {image, scan index, d0..d5}; counts[0] = its length
int launch_yolo_candidates(snnb_context* ctx, const snnb_tensor* h0, const snnb_tensor* h1, float thresh, int maxc, int* counts, float* cand);
int launch_flatten(snnb_context* ctx, const snnb_tensor* in, snnb_tensor* out);
int launch_concat(snnb_context* ctx, const snnb_tensor* a, const snnb_tensor* b, snnb_tensor* out);
int launch_upsample(snnb_context* ctx, const snnb_tensor* in, snnb_tensor* out, float scale, bool bilinear);
int launch_pad(snnb_context* ctx, const snnb_tensor* in, snnb_tensor* out, int pad_x, int pad_y, int mode);
// InstanceNorm scratch: (mean, rstd) per (n, c) followed by up to INSTNORM_MAX_CHUNKS x 16 partial sums per (n, 8-channel group)
constexpr int INSTNORM_MAX_CHUNKS = 64;
static inline size_t instnorm_scratch_floats(int n, int cp) { return (size_t) n * cp * 2 + (size_t) n * (cp >> 3) * INSTNORM_MAX_CHUNKS * 16; }
int launch_instancenorm(snnb_context* ctx, const snnb_tensor* in, snnb_tensor* out, const snnb_weights* w, int act, float alpha, float* scratch = nullptr);
int launch_subpixel(snnb_context* ctx, const snnb_tensor* in, snnb_tensor* out, int r);
int launch_split_f32(snnb_context* ctx, const float* dev_nhwc, snnb_tensor* t);       // fp32 NHWC (pitch C) -> hi/lo
int launch_split_u8(snnb_context* ctx, const uint8_t* dev_nhwc_u8, snnb_tensor* t, const float mean[4], const float norm[4]); // (u8 - mean[c&3]) * norm[c&3]
int launch_merge_f32(snnb_context* ctx, const snnb_tensor* t, float* dev_nhwc);       // hi/lo -> fp32 NHWC (pitch C)
int launch_result_small(snnb_context* ctx, const snnb_tensor* t, float* values, int* idx); // 1x1xC tensor -> fp32 values and/or arg-max per image (pointers may be mapped host memory)
// u8 NHWC image of size src_h x src_w -> resized (linear / nearest, vk_resize.comp) + normalised -> t
int launch_resize_u8(snnb_context* ctx, const uint8_t* dev_nhwc_u8, int src_h, int src_w, snnb_tensor* t, const float mean[4], const float norm[4], bool linear);
int launch_merge_u8(snnb_context* ctx, const snnb_tensor* t, uint8_t* dev_nhwc_u8, float scale, float offset); // clamp(round(v*scale+offset), 0, 255)

// ---- host-side weight folding/packing (pack.cpp) -----------------------------------------------------------
// K ordering of the row-window convolution kernel (kernels_umma.cu): for stride s the taps of one filter row fall
// into s column parities; within a parity consecutive taps read consecutive pixels of the de-interleaved row, so one
// tcgen05.mma K step (16 fp16 = 2 pixels x 8 channels) covers two taps of the same parity.
struct RowPlan {
    int parities = 0;
    int dmin[2]  = {0, 0}; // pixel offset (in de-interleaved index) of the first tap of each parity, relative to the output index
    int ntaps[2] = {0, 0};
    int ksteps   = 0;
    int ks_parity[8], ks_erel[8], ks_tap[8][2]; // up to 8 K steps = 2 weight panels of 64 K columns per filter row (9x9 taps)
    int span = 0; // pixels needed beyond the 128 of the tile
};
static inline bool make_row_plan(int k, int stride, int pad_x, RowPlan& rp) {
    if (k < 1 || k > 9 || !(stride == 1 || stride == 2)) return false;
    rp = RowPlan();
    rp.parities = stride;
    for (int par = 0; par < stride; ++par) {
        int js[9], t = 0;
        for (int j = 0; j < k; ++j)
            if ((((j - pad_x) % stride) + stride) % stride == par) js[t++] = j;
        rp.ntaps[par] = t;
        if (!t) continue;
        const int a  = js[0] - pad_x;
        rp.dmin[par] = a >= 0 ? a / stride : -((-a + stride - 1) / stride);
        for (int q = 0; q < (t + 1) / 2; ++q) {
            if (rp.ksteps >= 8) return false;
            rp.ks_parity[rp.ksteps] = par;
            rp.ks_erel[rp.ksteps]   = 2 * q;
            rp.ks_tap[rp.ksteps][0] = js[2 * q];
            rp.ks_tap[rp.ksteps][1] = (2 * q + 1 < t) ? js[2 * q + 1] : -1;
            rp.ksteps++;
        }
        rp.span = rp.span > 2 * ((t + 1) / 2) ? rp.span : 2 * ((t + 1) / 2);
    }
    return rp.ksteps > 0;
}

// K ordering of the row-window kernel's FEED mode (stride 2, <= 4 input channels: the RGB stems). With 4 channels per pixel one
// 16-byte K chunk holds TWO horizontally adjacent pixels, and for stride 2 the window of output pixel m starts at input pixel 2 m:
// chunk j of A row m is the pair (2 m + 2 j, 2 m + 2 j + 1) = 16 m + 16 j bytes into a plain dense pixel row - the canonical
// row pitch and LBO = 16 B again, but with NO parity de-interleave and half the K of the 8-channel form (7 taps x 4 ch + 1 pad
// tap = 32 K instead of 64). The feed copy is shifted right by px (even, >= pad_x) so that pairs start on even pixels; tap t of
// the filter sits at pixel offset d + t, d = px - pad_x in {0, 1}; offsets without a tap get zero weights.
struct FeedPlan {
    int px = 0, d = 0, nch = 0, ksteps = 0; // nch = 16-byte chunks per window (even), ksteps = nch / 2
    // A filter row needs only 16 * ksteps of the 64 K columns of a 128-byte weight row: rows_per_panel filter rows share one
    // (filter row ky -> panel row ky / rows_per_panel, columns (ky % rows_per_panel) * 64 / rows_per_panel ..), so the resident weight
    // panels of the 7x7 stem take 64 KB instead of 112 KB of shared memory.
    int rows_per_panel = 1;
};
static inline bool make_feed_plan(int k, int stride, int pad_x, int ic, FeedPlan& fp) {
    if (stride != 2 || ic > 4 || k < 2 || k > 9 || pad_x < 0 || pad_x > 8) return false;
    fp.px     = (pad_x + 1) & ~1;
    fp.d      = fp.px - pad_x;
    fp.nch    = ((fp.d + k + 1) / 2 + 1) & ~1;
    fp.ksteps = fp.nch / 2;
    fp.rows_per_panel = fp.ksteps == 1 ? 4 : (fp.ksteps == 2 ? 2 : 1);
    return fp.ksteps <= 4;
}

struct PackedHost {
    std::vector<float> w_f32;           // [K][OCw]
    std::vector<__half> w_hi, w_lo; // [OCr][Kp]
    std::vector<__half> w_row_hi, w_row_lo; // [kh][OCr][64] (row-window kernel), empty unless IC <= 8
    int row_stride = 0, row_pad = 0;
    std::vector<__half> w_feed_hi, w_feed_lo; // [ceil(kh / rows_per_panel)][OCr][64] in FeedPlan K order (stride-2 stems with <= 4 input channels)
    int feed_pad = -1;
    std::vector<float> bias;            // [round_up(OC,64)]
    std::vector<float> gamma, beta, mean, var;
    int kind = 0, in_ch = 0, out_ch = 0, kernel = 1, ocw = 0, kp = 0, ocr = 0;
    size_t device_bytes() const;
};
void pack_conv2d_host(int IC, int OC, int k, const float* w_oihw, const float* bias, const float* g, const float* b, const float* m, const float* v,
                      PackedHost& out);
// Appends a folded 1x1 projection shortcut (weights [OC][IC], bias and BatchNorm folded as in pack_conv2d_host) to the tensor-core
// operand of an already packed convolution: w_hi/lo become [OCr][k*k*ICp + round_up(IC, 8)], the bias becomes the sum of both biases.
void pack_shortcut_host(int IC, const float* w_oi, const float* bias, const float* g, const float* b, const float* m, const float* v, PackedHost& out);
// Adds the row-window operand (w_row_hi/lo) for small-IC convolutions; needs the layer's stride and x padding.
void pack_rowwin_host(PackedHost& p, int stride, int pad_x);
// Adds the feed-mode operand (w_feed_hi/lo) when make_feed_plan() accepts the layer.
void pack_feed_host(PackedHost& p, int stride, int pad_x);
void pack_depthwise_host(int C, int k, const float* w_chw, const float* bias, const float* g, const float* b, const float* m, const float* v,
                         PackedHost& out);
void pack_channels_host(int C, const float* g, const float* b, const float* m, const float* v, PackedHost& out);
// Copy a PackedHost into device memory at `base` (device, 256-B aligned) and point `w` at it. Returns bytes used.
int place_weights(snnb_context* ctx, const PackedHost& p, char* base, snnb_weights* w);

int tensor_alloc(snnb_context* ctx, int n, int h, int w, int c, snnb_tensor** out, bool lo_plane = true);
int tensor_alloc_feed(snnb_tensor* t, int feed_h, int feed_w, int py, int px); // see snnb_tensor::feed_hi

} // namespace snnb
