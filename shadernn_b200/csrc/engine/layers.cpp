// Per-layer output-dimension rules, weight packing and kernel dispatch. Each rule cites the reference code it
// restates; the arithmetic (float scale/translate then uint32 truncation) is kept exactly because it decides
// tensor shapes.
#include <algorithm>
#include <cmath>

#include <cstring>
#include <thread>

#include "engine.h"

using namespace snnb;

namespace snn {
namespace dp {

// genericlayer.cpp:64-90. The accumulators start at 0 and are combined with std::max, exactly as in the reference: a
// negative translation (e.g. a "valid" 3x3 stride-1 conv: 1 - 3 = -2) is therefore clamped to 0 and the layer keeps
// its input size. Kept on purpose - it decides tensor shapes a reference user's downstream code depends on.
void GenericModelLayer::getOutputDims(uint32_t& width, uint32_t& height, uint32_t& depth) const {
    width = height = depth = 0U;
    float accSW = 0, accSH = 0, accTW = 0, accTH = 0;
    const Transform t = getOutputScaleDimAdjustment();
    for (auto& dim : inputDims) {
        accSW  = std::max(accSW, t.scaleW * dim.width);
        accTW  = std::max(accTW, t.transW);
        accSH  = std::max(accSH, t.scaleH * dim.height);
        accTH  = std::max(accTH, t.transH);
        width  = (uint32_t) (accSW + accTW);
        height = (uint32_t) (accSH + accTH);
        depth  = std::max(depth, dim.depth);
    }
}

void InputLayerLayer::getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const {
    // real input dims come from ShaderGenOptions.desiredInput (dp.cpp:505-507); inputDims[0] is set by the graph builder
    w = inputDims.empty() ? _desc.inputWidth : inputDims[0].width;
    h = inputDims.empty() ? _desc.inputHeight : inputDims[0].height;
    d = _desc.inputChannels;
}

// ---- Conv2D ----------------------------------------------------------------------------------------------
GenericModelLayer::Transform Conv2DLayer::getOutputScaleDimAdjustment() const { // conv2d.cpp:102-113
    uint32_t offset[4];
    _desc.padding.offsets((int) _desc.kernelSize, true, offset);
    float scale       = 1 / static_cast<float>(_desc.stride);
    float translation = 0.0f;
    if (_desc.kernelSize % 2 != 0) {
        translation = 1 + (static_cast<float>(offset[0] + offset[1]) - static_cast<float>(_desc.kernelSize)) / static_cast<float>(_desc.stride);
    } else {
        translation = 1 + (static_cast<float>(offset[0] + offset[1] - 1) - static_cast<float>(_desc.kernelSize)) / static_cast<float>(_desc.stride);
    }
    return Transform {scale, scale, translation, translation};
}
void Conv2DLayer::getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const { // conv2d.cpp:34-37
    GenericModelLayer::getOutputDims(w, h, d);
    d = numOutputPlanes;
}
int padModeId(const std::string& m) { // conv2dVulkan.cpp:73-80
    if (m == "constant") return SNNB_PAD_CONSTANT;
    if (m == "replicate") return SNNB_PAD_REPLICATE;
    if (m == "reflect") return SNNB_PAD_REFLECT;
    return SNNB_PAD_NONE;
}
static const float* bnv(const std::map<std::string, std::vector<float>>& bn, const char* key) {
    auto it = bn.find(key);
    return (it == bn.end() || it->second.empty()) ? nullptr : it->second.data();
}
void Conv2DLayer::packWeights(PackedHost& p) {
    if (foldedInto) return; // packed as the extra columns of the convolution it was folded into (which frees the host copy)
    const auto& bn = _desc.batchNormalization;
    const bool use = _desc.useBatchNormalization;
    pack_conv2d_host((int) numInputPlanes, (int) numOutputPlanes, (int) _desc.kernelSize, _desc.weights.data(), _desc.biases.empty() ? nullptr : _desc.biases.data(),
                     use ? bnv(bn, "gamma") : nullptr, use ? bnv(bn, "beta") : nullptr, use ? bnv(bn, "movingMean") : nullptr,
                     use ? bnv(bn, "movingVariance") : nullptr, p);
    {
        uint32_t offs[4];
        _desc.padding.offsets((int) _desc.kernelSize, true, offs);
        const int mode = padModeId(_desc.padding.mode);
        // reflect / replicate convolutions run on a pre-padded copy of the input with pad 0 (wantsPrepad)
        if (mode == SNNB_PAD_NONE || mode == SNNB_PAD_CONSTANT) {
            pack_rowwin_host(p, (int) _desc.stride, _desc.kernelSize == 1 ? 0 : (int) offs[0]);
            if (feedInput) pack_feed_host(p, (int) _desc.stride, _desc.kernelSize == 1 ? 0 : (int) offs[0]);
        } else {
            pack_rowwin_host(p, (int) _desc.stride, 0);
        }
    }
    if (shortcut) {
        const auto& sd = shortcut->_desc;
        const bool sbn = sd.useBatchNormalization;
        pack_shortcut_host((int) shortcut->numInputPlanes, sd.weights.data(), sd.biases.empty() ? nullptr : sd.biases.data(),
                           sbn ? bnv(sd.batchNormalization, "gamma") : nullptr, sbn ? bnv(sd.batchNormalization, "beta") : nullptr,
                           sbn ? bnv(sd.batchNormalization, "movingMean") : nullptr, sbn ? bnv(sd.batchNormalization, "movingVariance") : nullptr, p);
        std::vector<float>().swap(shortcut->_desc.weights);
    }
    std::vector<float>().swap(_desc.weights); // host copy no longer needed
}
bool Conv2DLayer::wantsPrepad(const snnb_tensor* in, const snnb_tensor* out, int convAlgo, int& ph, int& pw) const {
    const int mode = padModeId(_desc.padding.mode);
    if (!(mode == SNNB_PAD_REPLICATE || mode == SNNB_PAD_REFLECT) || _desc.kernelSize <= 1 || convAlgo == SNNB_ALGO_SIMT) return false;
    ConvArgs probe {in, nullptr, const_cast<snnb_tensor*>(out), &weights, (int) _desc.kernelSize, (int) _desc.stride, 0, 0, SNNB_PAD_CONSTANT, 0, 0.0f};
    if (!conv2d_umma_supported(probe)) return false;
    // the window of the last output pixel ends at (O-1)*s + k - 1 in padded coordinates
    ph = (out->h - 1) * (int) _desc.stride + (int) _desc.kernelSize;
    pw = (out->w - 1) * (int) _desc.stride + (int) _desc.kernelSize;
    return true;
}

int Conv2DLayer::run(snnb_context* ctx, const ExecOptions& opt) {
    uint32_t offs[4];
    _desc.padding.offsets((int) _desc.kernelSize, true, offs);
    if (prepadded) {
        // padded[y][x] = in[reflect/replicate(y - pad_y)][..(x - pad_x)] with the conv's own (pad_x, pad_y) = (T, L) mapping
        if (launch_pad(ctx, inputs[0], prepadded, (int) offs[0], (int) offs[2], padModeId(_desc.padding.mode))) return 1;
        ConvArgs a {prepadded, residual, output, &weights, (int) _desc.kernelSize, (int) _desc.stride, 0, 0, SNNB_PAD_CONSTANT,
                    fusedAct >= 0 ? fusedAct : _desc.activation.id, fusedAct >= 0 ? fusedAlpha : _desc.activation.alpha};
        a.precision = opt.precision;
        return launch_conv2d_umma(ctx, a);
    }
    ConvArgs a;
    a.in = inputs[0], a.residual = residual, a.out = output, a.w = &weights;
    a.k = (int) _desc.kernelSize, a.stride = (int) _desc.stride;
    // uPadx <- offsets[0] (top), uPady <- offsets[2] (left): conv2dVulkan.cpp:183-184 (SURVEY Q5). The 1x1 shader has no padding.
    a.pad_x = _desc.kernelSize == 1 ? 0 : (int) offs[0];
    a.pad_y = _desc.kernelSize == 1 ? 0 : (int) offs[2];
    a.pad_mode = padModeId(_desc.padding.mode);
    a.act      = fusedAct >= 0 ? fusedAct : _desc.activation.id;
    a.alpha    = fusedAct >= 0 ? fusedAlpha : _desc.activation.alpha;
    a.precision = opt.precision;
    a.shortcut = shortcutIn, a.sc_stride = shortcut ? (int) shortcut->_desc.stride : 1;
    const int want = algo != SNNB_ALGO_AUTO ? algo : opt.convAlgo;
    if (want != SNNB_ALGO_SIMT && conv2d_umma_supported(a)) return launch_conv2d_umma(ctx, a);
    if (shortcut) {
        set_error("%s: a folded projection shortcut runs on the tensor-core kernel only; load the model with fuse=0 for another algorithm", name.c_str());
        return 2;
    }
    if (want == SNNB_ALGO_TCGEN05) {
        set_error("%s: tcgen05 path requested but unsupported for this shape", name.c_str());
        return 2;
    }
    return launch_conv2d_simt(ctx, a);
}

// ---- Depthwise -------------------------------------------------------------------------------------------
void SeparableConv2DLayer::getOutputDims(uint32_t& width, uint32_t& height, uint32_t& depth) const { // separableconvolution.cpp:77-86
    uint32_t po[4];
    _desc.padding.offsets((int) _desc.kernelSize, true, po);
    width = height = depth = 0;
    for (auto& dim : inputDims) {
        width  = (dim.width - _desc.kernelSize + po[0] + po[2]) / _desc.stride + 1;
        height = (dim.height - _desc.kernelSize + po[1] + po[3]) / _desc.stride + 1;
        depth  = dim.depth;
        break;
    }
}
void SeparableConv2DLayer::packWeights(PackedHost& p) {
    const auto& bn = _desc.batchNormalization;
    const bool use = _desc.useBatchNormalization;
    pack_depthwise_host((int) numInputPlanes, (int) _desc.kernelSize, _desc.weights.data(), _desc.biases.empty() ? nullptr : _desc.biases.data(),
                        use ? bnv(bn, "gamma") : nullptr, use ? bnv(bn, "beta") : nullptr, use ? bnv(bn, "movingMean") : nullptr,
                        use ? bnv(bn, "movingVariance") : nullptr, p);
}
int SeparableConv2DLayer::run(snnb_context* ctx, const ExecOptions&) {
    uint32_t offs[4];
    _desc.padding.offsets((int) _desc.kernelSize, true, offs);
    ConvArgs a;
    a.in = inputs[0], a.residual = nullptr, a.out = output, a.w = &weights;
    a.k = (int) _desc.kernelSize, a.stride = (int) _desc.stride;
    a.pad_x = (int) offs[0], a.pad_y = (int) offs[2]; // separableconvolutionVulkan.cpp:112-113
    a.pad_mode = SNNB_PAD_CONSTANT, a.act = _desc.activation.id, a.alpha = _desc.activation.alpha;
    return launch_depthwise(ctx, a);
}

// ---- Pools -----------------------------------------------------------------------------------------------
GenericModelLayer::Transform PoolingLayer::getOutputScaleDimAdjustment() const { // maxpool2d.cpp:26-35 / avgpool2d.cpp:21-30
    float scale = 1.0f / _desc.stride, translation;
    if (_desc.padding.validLike())
        translation = 1.0f - (static_cast<float>(_desc.kernelSize) / static_cast<float>(_desc.stride));
    else
        translation = 1.0f - 1.0f / static_cast<float>(_desc.stride);
    return Transform {scale, scale, translation, translation};
}
int PoolingLayer::run(snnb_context* ctx, const ExecOptions&) { return launch_pool(ctx, inputs[0], output, (int) _desc.kernelSize, (int) _desc.stride, isAvg); }

void AdaptiveAvgPool2dLayer::getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const {
    w = h = poolSize;
    d     = inputDims.empty() ? numOutputPlanes : inputDims[0].depth;
}
int AdaptiveAvgPool2dLayer::run(snnb_context* ctx, const ExecOptions&) {
    // only the evenly-dividing case (incl. global pooling, pool = 1) maps onto the clipped-window kernel
    const snnb_tensor* in = inputs[0];
    if (in->h % (int) poolSize || in->w % (int) poolSize || in->h / (int) poolSize != in->w / (int) poolSize) {
        set_error("%s: AdaptiveAvgPool2d needs H and W divisible by pool (%d x %d -> %u)", name.c_str(), in->h, in->w, poolSize);
        return 2;
    }
    const int k = in->h / (int) poolSize;
    return launch_pool(ctx, in, output, k, k, true);
}

// ---- elementwise -----------------------------------------------------------------------------------------
int AddLayer::run(snnb_context* ctx, const ExecOptions&) { return launch_add(ctx, inputs[0], inputs[1], output, activation.id, activation.alpha); }
void BatchNormalizationLayer::packWeights(PackedHost& p) {
    pack_channels_host((int) numOutputPlanes, bnv(batchNormalization, "gamma"), bnv(batchNormalization, "beta"), bnv(batchNormalization, "movingMean"),
                       bnv(batchNormalization, "movingVariance"), p);
}
int BatchNormalizationLayer::run(snnb_context* ctx, const ExecOptions&) { return launch_batchnorm(ctx, inputs[0], output, &weights, activation.id, activation.alpha); }
void InstanceNormLayer::packWeights(PackedHost& p) { pack_channels_host((int) numOutputPlanes, gamma.data(), beta.data(), nullptr, nullptr, p); }
int InstanceNormLayer::run(snnb_context* ctx, const ExecOptions&) {
    return launch_instancenorm(ctx, inputs[0], output, &weights, activation.id, activation.alpha, scratch);
}
int ActivationLayer::run(snnb_context* ctx, const ExecOptions&) { return launch_activation(ctx, inputs[0], output, activation.id, activation.alpha); }

// ---- Dense / Flatten -------------------------------------------------------------------------------------
void DenseLayer::getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const {
    w = h = 1;
    d     = units;
}
void DenseLayer::packWeights(PackedHost& p) {
    pack_conv2d_host((int) numInputPlanes, (int) units, 1, kernel.data(), biases.empty() ? nullptr : biases.data(), nullptr, nullptr, nullptr, nullptr, p);
    p.kind = 3;
    std::vector<float>().swap(kernel);
}
int DenseLayer::run(snnb_context* ctx, const ExecOptions& opt) {
    if (gapSource && gapSource->output && gap_dense_supported(gapSource->output, output, &weights))
        return launch_gap_dense(ctx, gapSource->output, output, &weights, activation.id == SNNB_ACT_SOFTMAX ? SNNB_ACT_NONE : activation.id, activation.alpha,
                                activation.id == SNNB_ACT_SOFTMAX);
    const snnb_tensor* x = inputs[0];
    if (x->h * x->w != 1) { // CPU Flatten order = HWC (cpulayer.h:94-115)
        if (launch_flatten(ctx, x, flat)) return 1;
        x = flat;
    }
    const bool softmax = activation.id == SNNB_ACT_SOFTMAX;
    ConvArgs a {x, nullptr, output, &weights, 1, 1, 0, 0, SNNB_PAD_NONE, softmax ? SNNB_ACT_NONE : activation.id, activation.alpha};
    a.precision = opt.precision;
    // SiLU on the CPU Dense path is a by-value no-op in the reference (cpulayer.h:245-252); we apply the real SiLU (SURVEY Q10).
    if (conv2d_umma_supported(a) ? launch_conv2d_umma(ctx, a) : launch_conv2d_simt(ctx, a)) return 1;
    if (softmax) return launch_softmax(ctx, output, output);
    return 0;
}
void FlattenLayer::getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const {
    w = h = 1;
    d     = inputDims.empty() ? numOutputPlanes : inputDims[0].width * inputDims[0].height * inputDims[0].depth;
}
int FlattenLayer::run(snnb_context* ctx, const ExecOptions&) {
    if (launch_flatten(ctx, inputs[0], output)) return 1;
    if (activation.id == SNNB_ACT_SOFTMAX) return launch_softmax(ctx, output, output);
    if (activation.id != SNNB_ACT_NONE) return launch_activation(ctx, output, output, activation.id, activation.alpha);
    return 0;
}

// ---- layout layers ---------------------------------------------------------------------------------------
void ConcatenateLayer::getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const { // concatenation.h:33-37 (depth adds up)
    w = h = d = 0;
    for (auto& dim : inputDims) {
        w = std::max(w, dim.width), h = std::max(h, dim.height);
        d += dim.depth;
    }
}
int ConcatenateLayer::run(snnb_context* ctx, const ExecOptions&) { return launch_concat(ctx, inputs[0], inputs[1], output); }

int UpSampling2DLayer::run(snnb_context* ctx, const ExecOptions&) { return launch_upsample(ctx, inputs[0], output, scale, interpolationType == "bilinear"); }

GenericModelLayer::Transform PadLayer::getOutputScaleDimAdjustment() const { // padlayer.cpp:60-68
    uint32_t offset[4];
    padding.offsets(0, false, offset);
    return Transform {1.0f, 1.0f, static_cast<float>(offset[2] + offset[3]), static_cast<float>(offset[0] + offset[1])};
}
int PadLayer::run(snnb_context* ctx, const ExecOptions&) {
    uint32_t offs[4];
    padding.offsets(0, false, offs);
    // vk_pad.comp: s0 = pos.xy - uPad with uPad = (offsets[0], offsets[2]) = (T, L) (padlayerVulkan.cpp:81-82)
    int mode = SNNB_PAD_CONSTANT;
    if (this->mode == "replicate") mode = SNNB_PAD_REPLICATE;
    if (this->mode == "reflect") mode = SNNB_PAD_REFLECT;
    return launch_pad(ctx, inputs[0], output, (int) offs[0], (int) offs[2], mode);
}

void SubpixelLayer::getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const { // subpixelmerge.h:36-43
    w = h = d = 0;
    for (auto& dim : inputDims) {
        w = dim.width * kernelSize, h = dim.height * kernelSize;
        d = 1;
    }
}
int SubpixelLayer::run(snnb_context* ctx, const ExecOptions&) { return launch_subpixel(ctx, inputs[0], output, (int) kernelSize); }

// ---- YOLO (host decode; yololayer.cpp) ---------------------------------------------------------------------
void YOLOLayer::getOutputDims(uint32_t& w, uint32_t& h, uint32_t& d) const {
    w = 6, h = 100, d = 1; // <= 100 rows of {class, score, x, y, w, h}
}

namespace {
struct Box {
    int cls;
    float score, x, y, w, h;
};
float iou(const Box& a, const Box& b) { // yololayer.cpp:56-70
    const float ix0 = std::max(a.x, b.x), iy0 = std::max(a.y, b.y);
    const float ix1 = std::min(a.x + a.w, b.x + b.w), iy1 = std::min(a.y + a.h, b.y + b.h);
    if (ix1 < ix0 || iy1 < iy0) return 0;
    const float inter = (ix1 - ix0) * (iy1 - iy0);
    return inter / (a.w * a.h + b.w * b.h - inter);
}
} // namespace

namespace {
// yololayer.cpp:31-38
const int kGridScale[2] = {32, 16};
const float kAnchors[]  = {10, 14, 23, 27, 37, 58, 81, 82, 135, 169, 344, 319};
const float kMasks[]    = {3, 4, 5, 1, 2, 3};
const int GC = 3, NFIX = 5, ONUM = 6;
const float kConfThresh = 0.35f, kIouThresh = 0.45f; // yololayer.cpp:182-183

// one box from the six raw values of a (cell, anchor): yololayer.cpp:115-164. Returns false below the confidence threshold.
bool decodeCell(const float* d, int yi, int gx, int gy, int gc, int gw, int gh, Box& out) {
    int cls        = 0;
    float maxLogit = -3.402823466e+38f;
    for (int i = NFIX; i < ONUM; ++i)
        if (d[i] > maxLogit) maxLogit = d[i], cls = i - NFIX;
    const int ai   = (int) kMasks[gc + yi * GC];
    const float bw = kAnchors[ai * 2], bh = kAnchors[ai * 2 + 1];
    const int netW = kGridScale[yi] * gw, netH = kGridScale[yi] * gh;
    const float prob = 1.f / ((1.f + std::exp(-d[4]) * (1.f + std::exp(-maxLogit)))); // yololayer.cpp:136, as parenthesised
    if (!(prob > kConfThresh)) return false;
    const float cx = (gx + 1.0f / (1.0f + std::exp(-d[0]))) / gw;
    const float cy = (gy + 1.0f / (1.0f + std::exp(-d[1]))) / gh;
    const float w_ = std::exp(d[2]) * bw / netW, h_ = std::exp(d[3]) * bh / netH;
    out = Box {cls, prob, cx - w_ / 2, cy - h_ / 2, w_, h_};
    return true;
}
// NMS, yololayer.cpp:72-110: stable sort by score, greedy suppression within a class
void nms(std::vector<Box>& list, SNNModelOutputBoxes& out) {
    std::stable_sort(list.begin(), list.end(), [](const Box& l, const Box& r) { return l.score > r.score; });
    std::vector<char> merged(list.size(), 0);
    for (size_t i = 0; i < list.size(); ++i) {
        if (merged[i]) continue;
        for (size_t j = i + 1; j < list.size(); ++j) {
            if (merged[j] || list[i].cls != list[j].cls) continue;
            if (iou(list[i], list[j]) > kIouThresh) merged[j] = 1;
        }
        out.rows.push_back({(float) list[i].cls, list[i].score, list[i].x, list[i].y, list[i].w, list[i].h});
    }
}
} // namespace

int YOLOLayer::decode(snnb_context* ctx, std::vector<SNNModelOutputBoxes>& perImage) {
    if (inputs.size() < 2) {
        set_error("%s: YOLO expects two heads", name.c_str());
        return 2;
    }
    const int N = inputs[0]->n;
    std::vector<std::vector<float>> heads(2);
    for (int i = 0; i < 2; ++i) {
        heads[i].resize(inputs[i]->pixels() * inputs[i]->c);
        if (snnb_tensor_download_nhwc(ctx, inputs[i], heads[i].data())) return 1;
        if (inputs[i]->c < GC * ONUM) {
            set_error("%s: YOLO head %d has %d channels, need >= %d", name.c_str(), i, inputs[i]->c, GC * ONUM);
            return 2;
        }
    }
    perImage.assign(N, SNNModelOutputBoxes());
    // decode + NMS are per image and quadratic in the candidate count: one host thread per image (the reference is
    // single-image; the arithmetic and the order of every image's list are unchanged)
    auto decodeImage = [&](int n) {
        std::vector<Box> list;
        for (int yi = 0; yi < 2; ++yi) {
            const snnb_tensor* t = inputs[yi];
            // the reference derives the grid from a fixed 416 input (yololayer.cpp:178-191); we use the head's own dims,
            // which coincide for 416x416.
            const int gw = t->w, gh = t->h, C = t->c;
            const float* data = heads[yi].data() + (size_t) n * gw * gh * C;
            for (int gy = 0; gy < gh; ++gy)
                for (int gx = 0; gx < gw; ++gx)
                    for (int gc = 0; gc < GC; ++gc) {
                        Box b;
                        if (decodeCell(data + ((size_t) gy * gw + gx) * C + gc * ONUM, yi, gx, gy, gc, gw, gh, b)) list.push_back(b);
                    }
        }
        nms(list, perImage[n]);
    };
    const int nthreads = std::max(1, std::min(N, (int) std::min(32u, std::max(1u, std::thread::hardware_concurrency()))));
    if (nthreads == 1) {
        for (int n = 0; n < N; ++n) decodeImage(n);
    } else {
        std::vector<std::thread> pool;
        for (int t = 0; t < nthreads; ++t)
            pool.emplace_back([&, t]() {
                for (int n = t; n < N; n += nthreads) decodeImage(n);
            });
        for (auto& th : pool) th.join();
    }
    return 0;
}

int YOLOLayer::enqueueCandidates(snnb_context* ctx, void* devBuf) {
    if (inputs.size() < 2 || inputs[0]->c < GC * ONUM || inputs[1]->c < GC * ONUM) {
        set_error("%s: YOLO expects two heads of >= %d channels", name.c_str(), GC * ONUM);
        return 2;
    }
    int* counts = static_cast<int*>(devBuf);
    float* cand = reinterpret_cast<float*>(static_cast<char*>(devBuf) + 32);
    // margin below the threshold: the device's expf may differ from the host's std::exp in the last bits; the host decides
    return launch_yolo_candidates(ctx, inputs[0], inputs[1], kConfThresh - 1e-3f, maxCand(), counts, cand);
}

int YOLOLayer::finishDecode(const void* hostBuf, const void* devBuf, std::vector<SNNModelOutputBoxes>& perImage) const {
    const int N     = inputs[0]->n;
    const int total = *static_cast<const int*>(hostBuf);
    if (total < 0 || total > maxCand()) return -1;
    const float* cand = reinterpret_cast<const float*>(static_cast<const char*>(hostBuf) + 32);
    if (total > YOLO_HEAD_ROWS) { // more candidates than the head copy carried: fetch the rest now (the device list is still intact)
        float* rest = const_cast<float*>(cand) + (size_t) YOLO_HEAD_ROWS * 8;
        if (cudaMemcpy(rest, static_cast<const char*>(devBuf) + 32 + (size_t) YOLO_HEAD_ROWS * 32, (size_t) (total - YOLO_HEAD_ROWS) * 32, cudaMemcpyDeviceToHost) != cudaSuccess)
            return -1;
    }
    auto word = [](const float* r, int i) {
        int v;
        memcpy(&v, r + i, sizeof v);
        return v;
    };
    std::vector<std::vector<const float*>> byImage(N);
    for (int i = 0; i < total; ++i) {
        const float* r = cand + (size_t) i * 8;
        const int n    = word(r, 0);
        if (n < 0 || n >= N) return -1;
        byImage[n].push_back(r);
    }
    perImage.assign(N, SNNModelOutputBoxes());
    const int cells0 = inputs[0]->h * inputs[0]->w * GC;
    auto finishImage = [&](int n) {
        auto& rows = byImage[n];
        // the device appended in arbitrary order: back to the order the reference's loops visit the cells
        std::sort(rows.begin(), rows.end(), [&](const float* a, const float* b) { return word(a, 1) < word(b, 1); });
        std::vector<Box> list;
        for (const float* r : rows) {
            int s        = word(r, 1);
            const int yi = s >= cells0 ? 1 : 0;
            if (yi) s -= cells0;
            const int gw = inputs[yi]->w, gh = inputs[yi]->h;
            const int gc = s % GC, cell = s / GC, gx = cell % gw, gy = cell / gw;
            Box b;
            if (decodeCell(r + 2, yi, gx, gy, gc, gw, gh, b)) list.push_back(b);
        }
        nms(list, perImage[n]);
    };
    // NMS is quadratic in an image's candidate count: images with many candidates get a host thread each (as decode() does)
    long long work = 0;
    for (int n = 0; n < N; ++n) work += (long long) byImage[n].size() * (long long) byImage[n].size();
    const int nthreads = work < 200000 ? 1 : std::max(1, std::min(N, (int) std::min(32u, std::max(1u, std::thread::hardware_concurrency()))));
    if (nthreads == 1) {
        for (int n = 0; n < N; ++n) finishImage(n);
    } else {
        std::vector<std::thread> pool;
        for (int t = 0; t < nthreads; ++t)
            pool.emplace_back([&, t]() {
                for (int n = t; n < N; n += nthreads) finishImage(n);
            });
        for (auto& th : pool) th.join();
    }
    return 0;
}

} // namespace dp
} // namespace snn
